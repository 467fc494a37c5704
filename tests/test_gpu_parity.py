"""GPU parity: the CUDA path (through the C ABI) against the golden vectors produced by the
unmodified reference and against the CPU oracle on fresh seeded inputs.

Tolerances (north_star): level schedule / CSR bit-exact; embeddings, losses and gradients within
1e-4 relative (max-norm per tensor) in fp32; scale-relative for the mathematically-zero gradients."""
import pytest
import torch

from oracle import dg_oracle as O
from util import (ZERO_GRAD_TAGS as ZERO_TAGS, batch_from_arrays, build_model, check_grads, load_golden, oracle_inputs,
                  oracle_train_grads, rel)

pytestmark = pytest.mark.gpu
CASES = ["mig_b4_r1", "aig_b4_r1", "xmg_b3_r2", "xag_b3_r1"]
TOL = 1e-4


def golden_batch(g):
    return batch_from_arrays(g["code"], g["edge_index"], g["forward_level"], g["prob"], g["tt_pair_index"], g["tt_sim"])


# --------------------------------------------------------------------------- schedule (bit-exact)
def test_kats_on_device():
    from deepgate.utils import dag_utils
    k = load_golden("kats")
    ei = k["edge_index"].cuda()
    assert dag_utils.top_sort(ei, 9).cpu().tolist() == [0, 0, 0, 1, 2, 3, 4, 4, 0]
    sub, _ = dag_utils.subgraph(torch.tensor([5, 3]), ei, dim=1)
    assert sub.cpu().tolist() == [[4, 1, 0, 1, 2], [5, 5, 3, 3, 3]]
    fl, fi, bl, bi = dag_utils.return_order_info(ei, 9)
    assert torch.equal(bl.cpu(), O.top_sort(k["edge_index"].flip(0), 9)) and torch.equal(fi.cpu(), torch.arange(9))


@pytest.mark.parametrize("name", CASES)
def test_level_csr_bit_exact(name):
    from deepgate.schedule import GraphCSR
    g = load_golden(name)
    n = g["code"].numel()
    csr = GraphCSR(g["edge_index"].cuda(), n, code=g["code"].cuda())
    level, L = csr.levelize()
    assert torch.equal(level.cpu().long(), g["forward_level"]) and L == int(g["forward_level"].max()) + 1
    rlevel, _ = csr.levelize(reverse=True)
    assert torch.equal(rlevel.cpu().long(), g["backward_level"])
    csr.set_levels(g["forward_level"].cuda())
    order, seg = csr.order.cpu().long(), csr.seg_ptr.cpu().long()
    in_ptr, in_src = csr.in_ptr.cpu().long(), csr.in_src.cpu().long()
    # node order == stable sort by (level, code); segments == G.forward_index[layer_mask & type_mask]
    key = g["forward_level"] * 8 + g["code"].long()
    assert torch.equal(order[:n], torch.sort(key, stable=True).indices)
    nodes, ptr = g["kat_nodes"].long(), g["kat_ptr"].tolist()
    keys = nodes[0] * 8 + nodes[1]
    for si, kk in enumerate(torch.unique_consecutive(keys).tolist()):
        sel = nodes[2][keys == kk]
        assert torch.equal(order[seg[kk]:seg[kk + 1]], sel)
        want = g["kat_edges"][:, ptr[si]:ptr[si + 1]]              # reference subgraph(l_node, edge_index, dim=1)
        got_src = torch.cat([in_src[in_ptr[v]:in_ptr[v + 1]] for v in sel.tolist()])
        got_dst = torch.cat([torch.full((int(in_ptr[v + 1] - in_ptr[v]),), v) for v in sel.tolist()])
        assert torch.equal(torch.stack([got_src, got_dst]), want)
    # out-CSR: ascending edge id per source, slots point back into the in-CSR
    ei = g["edge_index"]
    out_ptr, out_pack, out_slot = csr.out_ptr.cpu().long(), csr.out_pack.cpu().long(), csr.out_slot.cpu().long()
    stable = torch.sort(ei[0], stable=True).indices
    assert torch.equal(out_pack[:ei.size(1)] & ((1 << 28) - 1), ei[1][stable])
    assert torch.equal(out_pack[:ei.size(1)] >> 28, g["code"].long()[ei[1][stable]])
    assert torch.equal(in_src[out_slot[:ei.size(1)]], ei[0][stable])
    assert torch.equal(out_ptr, torch.cat([torch.zeros(1, dtype=torch.long), torch.cumsum(torch.bincount(ei[0], minlength=n), 0)]))


def test_levelize_large_and_cycle():
    from deepgate import synth
    from deepgate.schedule import GraphCSR
    c = synth.make_circuit("mig", 16, 30000, seed=4242, window=300)
    ei = torch.as_tensor(c["edge_index"]).t().contiguous()
    n = c["x"].shape[0]
    csr = GraphCSR(ei.cuda(), n, code=torch.as_tensor(c["x"][:, 1]).cuda())
    level, L = csr.levelize()
    ref = O.top_sort(ei, n)
    assert torch.equal(level.cpu().long(), ref) and L == int(ref.max()) + 1 and L > 150
    csr.set_levels()
    key = ref * 8 + torch.as_tensor(c["x"][:, 1])
    assert torch.equal(csr.order.cpu().long(), torch.sort(key, stable=True).indices)
    stable = torch.sort(ei[1], stable=True).indices                 # in-CSR == stable sort by destination
    assert torch.equal(csr.in_src.cpu().long(), ei[0][stable])
    cyc = torch.tensor([[0, 1, 2, 3], [1, 2, 0, 0]]).cuda()
    with pytest.raises(RuntimeError, match="cycle"):
        GraphCSR(cyc, 4).levelize()
    with pytest.raises(RuntimeError, match="outside"):
        GraphCSR(torch.tensor([[0, 9], [1, 2]]).cuda(), 4)
    empty = GraphCSR(torch.zeros(2, 0, dtype=torch.long).cuda(), 5, code=torch.zeros(5, dtype=torch.int32).cuda())
    lv, L0 = empty.levelize()
    assert lv.cpu().tolist() == [0] * 5 and L0 == 1


# --------------------------------------------------------------------------- forward / losses / grads vs golden
@pytest.mark.parametrize("name", CASES)
def test_forward_losses_grads_match_reference_golden(name):
    import deepgate
    g = load_golden(name)
    sd = O.synth_state_dict(g["kind"], g["weight_seed"])
    model = build_model(g["kind"], sd, g["num_rounds"])
    batch = golden_batch(g)
    hs, hf = model(batch)
    assert rel(hs, g["hs"]) < TOL and rel(hf, g["hf"]) < TOL
    assert float(hf.detach()[g["forward_level"].cuda() == 0].abs().max()) == 0.0        # PI rows exactly zero
    rec, pred_bin, _ = model.recon_loss(hs, g["train_pos_edge_index"].cuda(), g["neg_edge_index"].cuda())
    prob_loss = torch.nn.L1Loss()(model.pred_prob(hf), batch.prob)
    _, _, _, func = deepgate.ops.vae_func_loss(hf=hf, tt_pair_index=batch.tt_pair_index, tt_sim=batch.tt_sim)
    for got, key in ((rec, "recon_loss"), (prob_loss, "prob_loss"), (func, "func_loss")):
        assert abs(float(got) - float(g[key])) < TOL * max(1.0, abs(float(g[key]))), key
    assert float((pred_bin.cpu() != g["pred_bin"].int()).float().mean()) < 0.01
    if "grads" in g:
        w = g["loss_weights"]
        (w[0] * rec + w[1] * prob_loss + w[2] * func).backward()
        named = {k: p.grad for k, p in model.named_parameters()}
        assert all(v is not None for v in named.values()), "every parameter must receive a gradient"
        check_grads(named, g["grads"], TOL, name)


# --------------------------------------------------------------------------- fresh inputs vs the oracle
@pytest.mark.parametrize("kind,mix,batch,n_pi,n_gates,window,rounds", [
    ("mig", "mig4", 6, 16, 400, None, 1),
    ("xmg", "xmg", 4, 12, 300, 40, 3),
    ("aig", "aig", 5, (8, 24), (100, 500), None, 2),
    ("xag", "xag", 2, 8, 900, 6, 1),          # deep: > 150 levels
])
def test_train_step_matches_oracle(kind, mix, batch, n_pi, n_gates, window, rounds):
    import deepgate
    from deepgate import synth
    circuits = synth.make_circuits(mix, batch, n_pi, n_gates, cfg=21 + rounds, window=window, n_pairs=40)
    G = deepgate.circuits_to_batch(circuits, "cuda")
    sd = O.synth_state_dict(kind, 5 + rounds)
    model = build_model(kind, sd, rounds)
    gen = torch.Generator().manual_seed(3)
    E, n = G.edge_index.size(1), G.x.size(0)
    pos = G.edge_index.cpu()[:, torch.randperm(E, generator=gen)]
    neg = torch.randint(0, n, (2, E), generator=gen)
    weights = (1.0, 4.0, 4.0)
    hs, hf = model(G)
    rec, _, _ = model.recon_loss(hs, pos.cuda(), neg.cuda())
    prb = torch.nn.L1Loss()(model.pred_prob(hf), G.prob)
    _, _, _, fnc = deepgate.ops.vae_func_loss(hf=hf, tt_pair_index=G.tt_pair_index, tt_sim=G.tt_sim)
    (weights[0] * rec + weights[1] * prb + weights[2] * fnc).backward()
    total, parts, grads = oracle_train_grads(kind, sd, oracle_inputs(G, pos, neg), weights, rounds)
    assert rel(hs, parts["hs"]) < TOL and rel(hf, parts["hf"]) < TOL
    for got, key in ((rec, "recon"), (prb, "prob"), (fnc, "func")):
        assert abs(float(got) - float(parts[key])) < TOL * max(1.0, abs(float(parts[key]))), key
    check_grads({k: p.grad for k, p in model.named_parameters()}, grads, TOL, kind)


def test_struct_encoder_standalone_and_no_layernorm():
    import deepgate
    from deepgate import synth
    c = synth.make_circuits("mig", 2, 8, 120, cfg=31)
    G = deepgate.circuits_to_batch(c, "cuda")
    for layernorm, rounds in ((False, 1), (True, 2)):
        sd = O.synth_state_dict("mig", 40, layernorm=layernorm)
        enc = deepgate.digae_layer.DirectMultiGCNEncoder(dim_hidden=64, dim_feature=6, s_rounds=rounds,
                                                         t_rounds=rounds + 1, layernorm=layernorm).cuda()
        enc.load_state_dict({k[len("mig_struct_encoder."):]: v for k, v in sd.items() if k.startswith("mig_struct_encoder.")})
        code = G.gate.reshape(-1).long()
        feat = torch.nn.functional.one_hot((code == 1).long(), 6).float()
        s, t = enc(feat, feat, G.edge_index)                       # different round counts -> two separate launches
        (s.sin().sum() + (t * t).sum()).backward()
        P = {k: v.clone().requires_grad_(True) for k, v in sd.items() if k.startswith("mig_struct_encoder.")}
        so = O.multi_gcn_encoder(P, "mig_struct_encoder.source_conv", feat.cpu(), G.edge_index.cpu(), rounds, layernorm)
        to = O.multi_gcn_encoder(P, "mig_struct_encoder.target_conv", feat.cpu(), G.edge_index.cpu(), rounds + 1, layernorm)
        (so.sin().sum() + (to * to).sum()).backward()
        assert rel(s, so) < TOL and rel(t, to) < TOL
        for k, p in enc.named_parameters():
            assert rel(p.grad, P["mig_struct_encoder." + k].grad) < TOL, k


def test_vae_kernel_matches_reference_golden():
    import deepgate
    v = load_golden("vae")
    vae = deepgate.digvae_model.DirectedGVAE(torch.nn.Identity(), 64).cuda()
    vae.load_state_dict(v["params"])
    s, t = v["s"].cuda().requires_grad_(True), v["t"].cuda().requires_grad_(True)
    zs, zt = vae.sample(s, t, v["eps_s"].cuda(), v["eps_t"].cuda())
    kl = vae.kl_loss()
    assert rel(zs, v["z_s"]) < 1e-5 and rel(zt, v["z_t"]) < 1e-5
    assert abs(float(kl) - float(v["kl"])) < 1e-5 * abs(float(v["kl"]))
    (kl * 1000.0 + (zs * zs).mean() + zt.sin().mean()).backward()
    assert rel(s.grad, v["grad_s"]) < TOL and rel(t.grad, v["grad_t"]) < TOL
    for k, p in vae.named_parameters():
        assert rel(p.grad, v["grads"][k]) < TOL, k


def test_func_loss_edge_cases():
    import deepgate
    torch.manual_seed(0)
    hf = torch.randn(50, 64)
    hf[:5] = 0.0                                                   # zero rows (PIs): cos = 0, eps-clamped
    pair = torch.randint(0, 50, (2, 300))
    pair[:, :10] = torch.tensor([[0, 1, 2, 3, 4, 0, 7, 8, 9, 9], [9, 8, 7, 3, 11, 0, 7, 1, 2, 9]])
    tt = torch.rand(300)
    hf_o = hf.clone().requires_grad_(True)
    lo = O.func_loss(hf_o, pair, tt)
    lo.backward()
    hf_g = hf.cuda().requires_grad_(True)
    _, _, _, lg = deepgate.ops.vae_func_loss(hf=hf_g, tt_pair_index=pair.cuda(), tt_sim=tt.cuda())
    lg.backward()
    assert abs(float(lg) - float(lo)) < 1e-5
    nz = hf.abs().sum(1) > 0                                       # gradient into zero rows is 1e8-scaled junk the
    assert rel(hf_g.grad[nz.cuda()], hf_o.grad[nz]) < TOL          # sweep drops; compare the live rows


# --------------------------------------------------------------------------- size-independent properties at bench size
def test_properties_at_cfg2_size():
    import deepgate
    from deepgate import synth
    circuits = synth.make_circuits("aig", 64, (16, 64), (500, 1500), cfg=2)
    G = deepgate.circuits_to_batch(circuits, "cuda")
    model = build_model("aig", O.synth_state_dict("aig", 2), 1)
    hs1, hf1 = model(G)
    hs2, hf2 = model(G)
    assert torch.equal(hs1, hs2) and torch.equal(hf1, hf2)                     # deterministic, run to run
    assert torch.isfinite(hf1).all() and torch.isfinite(hs1).all()
    code = G.gate.reshape(-1)
    untouched = (G.forward_level == 0) | ~((code == 1) | (code == 2))
    assert float(hf1[untouched].abs().max()) == 0.0
    assert float(hf1[~untouched].abs().min(dim=1).values.max()) > 0.0
    # circuits are independent: a circuit's rows do not change when it is evaluated alone
    sub = deepgate.circuits_to_batch(circuits[:1], "cuda")
    hs_s, hf_s = model(sub)
    n0 = sub.x.size(0)
    assert rel(hf_s, hf1[:n0]) < 1e-5 and rel(hs_s, hs1[:n0]) < 1e-5
    # backward determinism of the pull-style sweep
    def grads():
        model.zero_grad()
        hs, hf = model(G)
        (hf.square().mean() + hs.mean()).backward()
        return torch.cat([p.grad.reshape(-1) for p in model.parameters() if p.grad is not None])
    g1, g2 = grads(), grads()
    assert torch.isfinite(g1).all() and rel(g1, g2) < 1e-6


def test_recon_loss_kernel_and_negative_sampler():
    """Fused decoder + BCE (dg_ae_model_mig.py:169-191) against plain torch; sampler: no self loops, no edges."""
    import deepgate
    from deepgate import ops, synth
    from deepgate.schedule import schedule_for_batch, check_deferred_errors
    G = deepgate.circuits_to_batch(synth.make_circuits("xmg", 3, 16, 300, cfg=31), "cuda")
    n, E = G.x.size(0), G.edge_index.size(1)
    g = torch.Generator().manual_seed(3)
    st = torch.randn(n, 128, generator=g).cuda().requires_grad_(True)
    pos = G.edge_index[:, torch.randperm(E, generator=g).cuda()]
    neg = torch.randint(0, n, (2, E + 17), generator=g).cuda()
    loss, pred = ops.recon_loss(st, pos, neg)
    (3.0 * loss).backward()
    st2 = st.detach().clone().requires_grad_(True)
    s, t = st2.chunk(2, dim=-1)
    pp = torch.sigmoid((s[pos[0]] * t[pos[1]]).sum(1))
    pn = torch.sigmoid((s[neg[0]] * t[neg[1]]).sum(1))
    ref = -torch.log(pp + 1e-15).mean() - torch.log(1 - pn + 1e-15).mean()
    (3.0 * ref).backward()
    assert abs(float(loss) - float(ref)) < 1e-5 * abs(float(ref))
    assert rel(st.grad, st2.grad) < 1e-5
    assert torch.equal(pred, torch.cat([pp > 0.5, pn > 0.5]).int())
    sch = schedule_for_batch(G)
    smp = ops.negative_sample(sch, 4 * E)
    assert smp.shape == (2, 4 * E) and int(smp.min()) >= 0 and int(smp.max()) < n
    assert not bool((smp[0] == smp[1]).any())
    key = G.edge_index[0] * n + G.edge_index[1]
    assert not bool(torch.isin(smp[0] * n + smp[1], key).any())
    assert len(torch.unique(smp[0] * n + smp[1])) > 3 * E          # not degenerate
    check_deferred_errors()


def test_async_schedule_equals_sync_schedule_and_flags_bad_input():
    """Host metadata attached at collate (data.attach_schedule_meta) removes every sync; results are identical."""
    import deepgate
    from deepgate import synth
    from deepgate.schedule import GraphCSR, schedule_for_batch, check_deferred_errors
    host = deepgate.circuits_to_batch(synth.make_circuits("mig4", 5, 16, 400, cfg=32, window=30))
    assert host.num_levels == int(host.forward_level.max()) + 1
    G = host.copy_to("cuda", non_blocking=False)
    a = schedule_for_batch(G, streams=1)                            # asynchronous form (metadata present)
    b = GraphCSR(G.edge_index.contiguous(), G.x.size(0), code=G.gate.reshape(-1)).set_levels(G.forward_level)
    assert a.L == b.L and a.code_count == b.code_count and a.streams == b.streams == 1
    for k in ("in_ptr", "in_src", "out_ptr", "out_pack", "out_slot", "order", "seg_ptr", "deg_order_in", "deg_order_out", "sweep_desc"):
        assert torch.equal(getattr(a, k), getattr(b, k)), k
    # the same batch cut into its two circuit sets (data.attach_streams): lists sorted by (stream, level, code).  c wraps the
    # schedule the HOST built at collate time (per-circuit CSRs merged by offset, data.attach_host_schedule); d is built on the
    # device from edge_index: every array must be bit-identical
    c = schedule_for_batch(G)
    assert getattr(G, "sched_order", None) is not None and c.in_ptr.data_ptr() == G.sched_in_ptr.data_ptr()
    d = GraphCSR(G.edge_index.contiguous(), G.x.size(0), code=G.gate.reshape(-1)).set_levels(
        G.forward_level, stream_of_node=G.sweep_stream, streams=2)
    assert c.streams == d.streams == 2 and c.code_count == d.code_count == a.code_count and c.L == d.L
    for k in ("in_ptr", "out_ptr", "order", "seg_ptr", "deg_order_in", "deg_order_out", "sweep_desc", "gdesc_in", "gdesc_out",
              "tile_cost_in", "tile_cost_out"):
        assert torch.equal(getattr(c, k), getattr(d, k)), k
    for k in ("in_src", "out_pack", "out_slot"):
        assert torch.equal(getattr(c, k)[:c.E], getattr(d, k)[:c.E]), k
    key = (G.sweep_stream.long() * a.L + G.forward_level.long()) * 8 + G.gate.reshape(-1).long().clamp(0, 6)
    assert torch.equal(c.order.long(), torch.sort(key, stable=True).indices)
    assert torch.equal(c.seg_ptr.long(), torch.cat([key.new_zeros(1), torch.bincount(key, minlength=2 * a.L * 8).cumsum(0)]))
    o = c.order.long()
    assert torch.equal(c.sweep_desc[:, 0].long(), o)
    assert torch.equal(c.sweep_desc[:, 2], (c.in_ptr[1:] - c.in_ptr[:-1])[o]) and torch.equal(c.sweep_desc[:, 4], (c.out_ptr[1:] - c.out_ptr[:-1])[o])
    check_deferred_errors()
    bad = G.edge_index.clone()
    bad[0, 0] = G.x.size(0) + 5
    GraphCSR(bad, G.x.size(0), code=G.gate.reshape(-1), validate=False)
    with pytest.raises(RuntimeError):
        check_deferred_errors()
    check_deferred_errors()                                         # flag was cleared
    with pytest.raises(RuntimeError):
        GraphCSR(bad, G.x.size(0), code=G.gate.reshape(-1), validate=True)


@pytest.mark.parametrize("cut", [2, 7, 3])
def test_sweep_result_does_not_depend_on_the_stream_cut(cut, monkeypatch):
    """One stream (the reference's plain level order), two circuit-set streams (grid mode) and one set per cluster (cluster mode:
    7 sets = one circuit each, 3 sets = clusters walking several circuits per level) give the same embeddings (the arithmetic of a
    node does not depend on which stream runs it) and the same gradients up to summation order."""
    import deepgate
    from deepgate import synth, ops
    from deepgate.schedule import schedule_for_batch
    from oracle import dg_oracle as O
    monkeypatch.setenv("MGV_SWEEP_STREAMS", str(cut))
    host = deepgate.circuits_to_batch(synth.make_circuits("xmg", 7, 16, 700, cfg=41, window=40))
    monkeypatch.delenv("MGV_SWEEP_STREAMS")
    assert host.sched_streams == cut
    G = host.copy_to("cuda", non_blocking=False)
    enc = deepgate.digae_layer.DirectMultiGCNEncoder(dim_hidden=64, dim_feature=6, s_rounds=1, t_rounds=1, layernorm=True)
    model = deepgate.dg_ae_model_xmg.Model(struct_encoder=enc, num_rounds=1, dim_hidden=64)
    model.load_state_dict(O.synth_state_dict("xmg", 3), strict=False)
    model = model.cuda()
    codes = [c for c, _ in model.GATE_MODULES]
    mods = [(getattr(model, "aggr_%s_func" % s), getattr(model, "update_%s_func" % s)) for _, s in model.GATE_MODULES]
    torch.manual_seed(5)
    hs0 = torch.randn(G.x.size(0), 64, device="cuda")
    gout = torch.randn(G.x.size(0), 64, device="cuda")
    res = []
    for streams in (1, cut):
        sch = schedule_for_batch(G, streams=streams)
        assert sch.streams == streams
        hs = hs0.clone().requires_grad_(True)
        model.zero_grad(set_to_none=True)
        hf = ops.level_sweep(hs, sch, 1, codes, mods)
        (hf * gout).sum().backward()
        res.append((hf.detach().clone(), hs.grad.clone(), {k: v.grad.clone() for k, v in model.named_parameters() if v.grad is not None}))
    assert float((res[0][0] - res[1][0]).abs().max()) <= 1e-6 * float(res[0][0].abs().max())
    print("stream cut: hf bit-identical", torch.equal(res[0][0], res[1][0]))
    assert float((res[0][1] - res[1][1]).abs().max()) <= 1e-5 * float(res[0][1].abs().max())
    for k, g in res[0][2].items():
        assert float((g - res[1][2][k]).abs().max()) <= 2e-5 * max(float(g.abs().max()), 1e-6), k


# --------------------------------------------------------------------------- bf16 configuration (stated tolerance)
BF16_TOL = 2e-2          # embeddings / losses, max-norm relative; gradients 5e-2 (one bf16 plane, fp32 accumulate)


def test_bf16_mode_within_stated_tolerance():
    """cfg4's bf16 configuration: tensor-core operands rounded to ONE bf16 plane (fp32 accumulation and fp32
    storage); the reference has no bf16 path, so the bar is the fp32 oracle within the stated tolerance."""
    import deepgate
    from deepgate import ops, synth
    circuits = synth.make_circuits("xmg", 4, 12, 300, cfg=24, window=40, n_pairs=40)
    G = deepgate.circuits_to_batch(circuits, "cuda")
    sd = O.synth_state_dict("xmg", 6)
    model = build_model("xmg", sd, 2)
    gen = torch.Generator().manual_seed(3)
    E, n = G.edge_index.size(1), G.x.size(0)
    pos = G.edge_index.cpu()[:, torch.randperm(E, generator=gen)]
    neg = torch.randint(0, n, (2, E), generator=gen)
    weights = (1.0, 4.0, 4.0)
    ops.set_precision("bf16")
    try:
        hs, hf = model(G)
        rec, _, _ = model.recon_loss(hs, pos.cuda(), neg.cuda())
        prb = torch.nn.L1Loss()(model.pred_prob(hf), G.prob)
        _, _, _, fnc = ops.vae_func_loss(hf=hf, tt_pair_index=G.tt_pair_index, tt_sim=G.tt_sim)
        (weights[0] * rec + weights[1] * prb + weights[2] * fnc).backward()
    finally:
        ops.set_precision("fp32")
    total, parts, grads = oracle_train_grads("xmg", sd, oracle_inputs(G, pos, neg), weights, 2)
    e_hs, e_hf = rel(hs, parts["hs"]), rel(hf, parts["hf"])
    assert e_hs < BF16_TOL and e_hf < BF16_TOL, (e_hs, e_hf)
    assert e_hs > 1e-5, "bf16 mode did not engage (result is fp32-accurate)"
    for got, key in ((rec, "recon"), (prb, "prob"), (fnc, "func")):
        assert abs(float(got) - float(parts[key])) < BF16_TOL * max(1.0, abs(float(parts[key]))), key
    worst = 0.0
    for k, p in model.named_parameters():
        ref = grads.get(k)
        if ref is None or any(t in k for t in ZERO_TAGS) or k.endswith("attn_lin.weight") or k.endswith("msg_k.weight"):
            continue
        worst = max(worst, rel(p.grad, ref))
    assert worst < 5e-2, worst


def struct_reference(sd, feat, ei, loss, round=None):
    """Float64 CPU reference of DirectMultiGCNEncoder (2 + 2 rounds, layernorm) for the struct-backward tests: outputs s, t
    and the gradients of ``loss(s, t)`` under the module's parameter names.  ``round``: the bf16-operand form of the oracle
    (multi_gcn_encoder_composed), otherwise the plain encoder."""
    P = {k[len("mig_struct_encoder."):]: v.clone().to(torch.float64).requires_grad_(True)
         for k, v in sd.items() if k.startswith("mig_struct_encoder.")}
    enc = O.multi_gcn_encoder if round is None else (lambda *a: O.multi_gcn_encoder_composed(*a, round=round))
    s = enc(P, "source_conv", feat.cpu(), ei.cpu(), 2, True)
    t = enc(P, "target_conv", feat.cpu(), ei.cpu(), 2, True)
    loss(s, t).backward()
    return s.detach(), t.detach(), {k: p.grad for k, p in P.items()}


def test_struct_backward_matches_fp64_oracle_on_a_large_heavy_tailed_graph(monkeypatch):
    """The tcgen05 backward (csrc/struct_bwd_tc.cu: one chunk and many chunks of tiles) against the float64 oracle on
    ~20 000 nodes with fan-outs up to the hundreds (tile hand-off buffers, per-tile power-of-two scales, chunk-wide rescale,
    tile order = degree order)."""
    import deepgate
    from deepgate import synth
    import numpy as np
    circuits = synth.make_circuits("mig", 3, 12, 6500, cfg=77)
    for ci, c in enumerate(circuits):             # hubs: re-route one fan-in of ~300 gates per circuit to 3 primary inputs
        ei = c["edge_index"]
        rng = np.random.default_rng(900 + ci)
        for hub, cnt in ((0, 200), (1, 90), (2, 40)):
            gates = rng.choice(np.arange(200, c["x"].shape[0]), size=cnt, replace=False)
            for gte in gates:
                rows = np.nonzero(ei[:, 1] == gte)[0]
                if rows.size and not (ei[rows, 0] == hub).any():
                    ei[rows[0], 0] = hub
    G = deepgate.circuits_to_batch(circuits, "cuda")
    sd = O.synth_state_dict("mig", 41, layernorm=True)
    code = G.gate.reshape(-1).long()
    feat = torch.nn.functional.one_hot((code == 1).long(), 6).float()
    gsrc = torch.Generator().manual_seed(5)
    ws = torch.randn(G.x.size(0), 64, generator=gsrc).cuda()
    wt = torch.randn(G.x.size(0), 64, generator=gsrc).cuda()
    outdeg = torch.bincount(G.edge_index[0], minlength=code.numel())
    assert int(outdeg.max()) >= 64, "the generator should produce heavy fan-out nodes"
    loss = lambda s, t: (s * ws.to(s)).sum() + (t * wt.to(t)).sum()

    def run(env):
        monkeypatch.delenv("MGV_STRUCT_CHUNK", raising=False)
        for k, v in env.items():
            monkeypatch.setenv(k, v)
        enc = deepgate.digae_layer.DirectMultiGCNEncoder(dim_hidden=64, dim_feature=6, s_rounds=2, t_rounds=2, layernorm=True).cuda()
        enc.load_state_dict({k[len("mig_struct_encoder."):]: v for k, v in sd.items() if k.startswith("mig_struct_encoder.")})
        s, t = enc(feat, feat, G.edge_index)
        loss(s, t).backward()
        torch.cuda.synchronize()
        return s.detach(), t.detach(), {k: p.grad.clone() for k, p in enc.named_parameters()}

    s0, t0, g0 = struct_reference(sd, feat, G.edge_index, loss)
    s1 = t1 = None
    for env in ({}, {"MGV_STRUCT_CHUNK": "16"}):
        s, t, g = run(env)
        if s1 is None:
            s1, t1 = s, t
            print("fwd rel(s, fp64) %.2e rel(t, fp64) %.2e" % (rel(s, s0), rel(t, t0)))
            assert rel(s, s0) < 1e-4 and rel(t, t0) < 1e-4, (rel(s, s0), rel(t, t0))
        assert torch.equal(s, s1) and torch.equal(t, t1)              # same forward kernel
        print(env, "worst grad rel vs fp64 %.2e" % max(rel(g[k], g0[k]) for k in g0))
        for k in g0:
            assert rel(g[k], g0[k]) < 1e-4, (env, k, rel(g[k], g0[k]))


def test_struct_backward_bf16_matches_the_bf16_operand_reference(monkeypatch):
    """bf16 mode: the tcgen05 backward (single bf16 plane: the forward's saved hi planes, bf16 gate-gradient planes, no tile
    scale) against a float64 reference that rounds the same operands to bf16 (oracle multi_gcn_encoder_composed: tile
    operands and weights in the forward, the gate pre-activation gradients in the backward) and against the fp32-accurate
    gradients.  The kernel accumulates in fp32 and reads h from the bf16 plane (2^-9): 2e-2 of the gradient's max-norm
    against the reference.  Against fp32: 5e-2 (BF16 gradient tolerance of the configuration)."""
    import deepgate
    from deepgate import ops, synth
    G = deepgate.circuits_to_batch(synth.make_circuits("mig", 4, 12, 3000, cfg=31), "cuda")
    sd = O.synth_state_dict("mig", 43, layernorm=True)
    code = G.gate.reshape(-1).long()
    feat = torch.nn.functional.one_hot((code == 1).long(), 6).float()
    gsrc = torch.Generator().manual_seed(6)
    ws = torch.randn(G.x.size(0), 64, generator=gsrc).cuda()
    wt = torch.randn(G.x.size(0), 64, generator=gsrc).cuda()
    loss = lambda s, t: (s * ws.to(s)).sum() + (t * wt.to(t)).sum()

    def run(env, precision):
        monkeypatch.delenv("MGV_STRUCT_CHUNK", raising=False)
        for k, v in env.items():
            monkeypatch.setenv(k, v)
        ops.set_precision(precision)
        try:
            enc = deepgate.digae_layer.DirectMultiGCNEncoder(dim_hidden=64, dim_feature=6, s_rounds=2, t_rounds=2, layernorm=True).cuda()
            enc.load_state_dict({k[len("mig_struct_encoder."):]: v for k, v in sd.items() if k.startswith("mig_struct_encoder.")})
            s, t = enc(feat, feat, G.edge_index)
            loss(s, t).backward()
            torch.cuda.synchronize()
        finally:
            ops.set_precision("fp32")
        return s.detach(), t.detach(), {k: p.grad.clone() for k, p in enc.named_parameters()}

    s32, t32, g32 = run({}, "fp32")
    _, _, g0 = struct_reference(sd, feat, G.edge_index, loss, round=torch.bfloat16)
    s1 = t1 = None
    for env in ({}, {"MGV_STRUCT_CHUNK": "16"}):
        s, t, g = run(env, "bf16")
        if s1 is None:
            s1, t1 = s, t
        assert torch.equal(s, s1) and torch.equal(t, t1)              # same forward kernel (the chunking is backward only)
        assert rel(s, s32) > 1e-5, "bf16 mode did not engage"
        print(env, "worst grad rel vs bf16 reference %.2e, vs fp32 %.2e" % (max(rel(g[k], g0[k]) for k in g0),
                                                                           max(rel(g[k], g32[k]) for k in g0)))
        for k in g0:
            assert rel(g[k], g0[k]) < 2e-2, (env, k, rel(g[k], g0[k]))
            assert rel(g[k], g32[k]) < 5e-2, (env, k, rel(g[k], g32[k]))


@pytest.mark.parametrize("n_nodes", [1, 2, 127, 128, 129, 256, 385])
def test_struct_backward_matches_fp64_oracle_at_tile_boundaries(n_nodes):
    """Node counts around the 128-row tile size (and degenerate graphs): tcgen05 forward and backward vs the float64 oracle."""
    import deepgate
    g = torch.Generator().manual_seed(n_nodes)
    # random DAG: every node i > 0 draws up to 3 distinct predecessors among 0 .. i-1
    src, dst = [], []
    for i in range(1, n_nodes):
        k = min(i, int(torch.randint(1, 4, (1,), generator=g)))
        for j in torch.randperm(i, generator=g)[:k].tolist():
            src.append(j); dst.append(i)
    ei = torch.tensor([src, dst], dtype=torch.int64).reshape(2, -1).cuda()
    feat = torch.nn.functional.one_hot(torch.randint(0, 2, (n_nodes,), generator=g), 6).float().cuda()
    sd = O.synth_state_dict("mig", 43, layernorm=True)
    ws = torch.randn(n_nodes, 64, generator=g).cuda()
    loss = lambda s, t: (s * ws.to(s)).sum() + (t * t).sum()

    enc = deepgate.digae_layer.DirectMultiGCNEncoder(dim_hidden=64, dim_feature=6, s_rounds=2, t_rounds=2, layernorm=True).cuda()
    enc.load_state_dict({k[len("mig_struct_encoder."):]: v for k, v in sd.items() if k.startswith("mig_struct_encoder.")})
    s1, t1 = enc(feat, feat, ei)
    loss(s1, t1).backward()
    torch.cuda.synchronize()
    s0, t0, g0 = struct_reference(sd, feat, ei, loss)
    assert torch.isfinite(s1).all() and torch.isfinite(t1).all()
    assert rel(s1, s0) < 1e-4 and rel(t1, t0) < 1e-4, (rel(s1, s0), rel(t1, t0))
    print("fwd rel s %.2e t %.2e, worst grad rel vs fp64 %.2e" % (rel(s1, s0), rel(t1, t0),
                                                                   max(rel(p.grad, g0[k]) for k, p in enc.named_parameters())))
    for k, p in enc.named_parameters():
        assert rel(p.grad, g0[k]) < 1e-4, (k, rel(p.grad, g0[k]))


@pytest.mark.parametrize("n_nodes", [3969, 4000, 4096, 135400, 137000])
def test_struct_forward_at_the_tile_search_boundaries(n_nodes):
    """Tile counts at which the warp-cooperative range search of the struct forward (csrc/mgv_tc.cuh warp_lower_bound) ends
    on a window of exactly 32 entries with no entry >= the target (32 tiles; 1057-1089 tiles): round 1 returned lo - 1 there
    and the last CTA skipped its trailing tiles (states stayed uninitialised).  Every row of the output is compared."""
    import deepgate
    from deepgate import synth
    c = synth.make_circuit("mig", 16, n_nodes - 16, seed=n_nodes, window=2000)
    G = deepgate.circuits_to_batch([c], "cuda")
    assert G.x.size(0) == n_nodes
    sd = O.synth_state_dict("mig", 44, layernorm=True)
    enc = deepgate.digae_layer.DirectMultiGCNEncoder(dim_hidden=64, dim_feature=6, s_rounds=1, t_rounds=1, layernorm=True).cuda()
    enc.load_state_dict({k[len("mig_struct_encoder."):]: v for k, v in sd.items() if k.startswith("mig_struct_encoder.")})
    code = G.gate.reshape(-1).long()
    feat = torch.nn.functional.one_hot((code == 1).long(), 6).float()
    with torch.no_grad():
        s, t = enc(feat, feat, G.edge_index)
    P = {k: v for k, v in sd.items() if k.startswith("mig_struct_encoder.")}
    so = O.multi_gcn_encoder(P, "mig_struct_encoder.source_conv", feat.cpu(), G.edge_index.cpu(), 1, True)
    to = O.multi_gcn_encoder(P, "mig_struct_encoder.target_conv", feat.cpu(), G.edge_index.cpu(), 1, True)
    assert torch.isfinite(s).all() and torch.isfinite(t).all()
    err_s = (s.cpu() - so).abs().max(dim=1).values
    assert float(err_s.max()) < TOL * float(so.abs().max()), int(err_s.argmax())
    assert rel(t, to) < TOL


@pytest.mark.parametrize("E", [0, 1, 2, 3, 17, 256, 257, 4097, 98256])
def test_edge_split_is_a_random_permutation_of_the_edges(E):
    """``split_edges`` (preprocessing.py:8-83 with zero val / test ratios): ``train_pos_edge_index`` holds every edge exactly once,
    source and target moved together, in an order that changes from call to call (``mgv_permute_edges``, Feistel + cycle walking)."""
    from deepgate import ops
    g = torch.Generator().manual_seed(E)
    ei = torch.randint(0, 1 << 20, (2, E), generator=g, dtype=torch.int64).cuda()
    a, b = ops.permute_edges(ei), ops.permute_edges(ei)
    assert a.shape == ei.shape and a.dtype == torch.int64
    key = lambda t: torch.sort(t[0] * (1 << 21) + t[1]).values
    assert torch.equal(key(a), key(ei)) and torch.equal(key(b), key(ei))
    if E >= 256:
        assert (a[0] != ei[0]).float().mean() > 0.9 and (a[0] != b[0]).float().mean() > 0.9
        # the order is not a shift or another low-complexity map: neighbours in the output come from far apart
        pos = {int(k): i for i, k in enumerate((ei[0] * (1 << 21) + ei[1]).tolist())}
        src = torch.tensor([pos[int(k)] for k in (a[0] * (1 << 21) + a[1]).tolist()][:4096])
        assert (src[1:] - src[:-1]).abs().float().mean() > E / 8
