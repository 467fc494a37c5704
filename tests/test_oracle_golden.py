"""Pins oracle/dg_oracle.py (the CPU restatement) against outputs of the unmodified
reference (tests/golden/*.pt, produced by oracle/make_golden.py under the shim)."""
import os

import pytest
import torch

from oracle import dg_oracle as O
from util import absmax, rel

CASES = ["mig_b4_r1", "aig_b4_r1", "xmg_b3_r2", "xag_b3_r1"]


def load(golden_dir, name):
    return torch.load(os.path.join(golden_dir, name + ".pt"), weights_only=False)


def test_structural_kats(golden_dir):
    k = load(golden_dir, "kats")
    assert k["top_sort"].tolist() == [0, 0, 0, 1, 2, 3, 4, 4, 0]            # SURVEY.md section 3.3
    assert k["subgraph_5_3"].tolist() == [[4, 1, 0, 1, 2], [5, 5, 3, 3, 3]]  # SURVEY.md section 8c
    assert torch.equal(O.top_sort(k["edge_index"], 9), k["top_sort"])
    for literal in (True, False):
        assert torch.equal(O.subgraph(torch.tensor([5, 3]), k["edge_index"], 1, literal), k["subgraph_5_3"])


@pytest.mark.parametrize("name", CASES)
def test_schedule_matches_reference(golden_dir, name):
    g = load(golden_dir, name)
    n = g["code"].numel()
    assert torch.equal(O.top_sort(g["edge_index"], n), g["forward_level"])
    fl, fi, bl, bi = O.return_order_info(g["edge_index"], n)
    assert torch.equal(bl, g["backward_level"]) and torch.equal(fi, torch.arange(n))
    ptr = g["kat_ptr"].tolist()
    nodes = g["kat_nodes"].long()
    keys = nodes[0] * 8 + nodes[1]
    seg = 0
    for key in torch.unique_consecutive(keys).tolist():
        sel = nodes[2][keys == key]
        want = g["kat_edges"][:, ptr[seg]:ptr[seg + 1]]
        for literal in (True, False):
            assert torch.equal(O.subgraph(sel, g["edge_index"], 1, literal), want)
        seg += 1
    assert seg == len(ptr) - 1


@pytest.mark.parametrize("name", CASES)
def test_forward_and_losses_match_reference(golden_dir, name):
    g = load(golden_dir, name)
    P = O.synth_state_dict(g["kind"], g["weight_seed"])
    G = {k: g[k] for k in ("edge_index", "forward_level", "prob", "tt_pair_index", "tt_sim",
                           "train_pos_edge_index", "neg_edge_index")}
    G["code"] = g["code"].long()
    with_grads = "grads" in g
    for k, p in P.items():
        p.requires_grad_(with_grads and "running" not in k)
    total, parts = O.train_step_losses(P, g["kind"], G, g["loss_weights"], g["num_rounds"],
                                       literal_subgraph=(name == "xag_b3_r1"))
    assert rel(parts["hs"].detach(), g["hs"]) < 2e-6
    assert rel(parts["hf"].detach(), g["hf"]) < 2e-6
    lvl0 = g["forward_level"] == 0
    assert float(parts["hf"].detach()[lvl0].abs().max()) == 0.0          # PI rows stay exactly zero
    for key in ("recon", "prob", "func"):
        assert abs(float(parts[key].detach()) - float(g[key + "_loss"])) < 2e-6 * max(1.0, abs(float(g[key + "_loss"])))
    if with_grads:
        total.backward()
        scale = {}
        for k, ref in g["grads"].items():
            got = P[k].grad
            if ref is None:
                assert got is None or float(got.abs().max()) == 0.0
                continue
            assert got is not None, k
            mathematically_zero = (".msg_q." in k or k.endswith("msg_k.bias") or k.endswith("attn_lin.bias"))
            if mathematically_zero:
                # scale-relative bound (SURVEY.md section 7 hard part 3): pure rounding noise on both sides
                kw = k.split(".")[0] + ".msg_k.weight"
                assert float(got.abs().max()) <= 1e-4 * absmax(g["grads"][kw]) + 1e-12, k
                continue
            assert rel(got, ref) < 5e-5, (k, rel(got, ref))


def test_composed_struct_encoder_equals_the_encoder():
    """The kernel-shaped restatement (one tile product per step, AggConv composed into the GRU input weights) is the same
    function as multi_gcn_encoder: outputs and every parameter gradient agree in float64."""
    g = torch.Generator().manual_seed(12)
    n = 90
    src, dst = [], []
    for i in range(1, n):                       # random DAG: up to 3 distinct predecessors among 0 .. i-1
        for j in torch.randperm(i, generator=g)[:min(i, int(torch.randint(1, 4, (1,), generator=g)))].tolist():
            src.append(j); dst.append(i)
    ei = torch.tensor([src, dst])
    x6 = torch.nn.functional.one_hot(torch.randint(0, 2, (n,), generator=g), 6)
    w = torch.randn(n, 64, generator=g, dtype=torch.float64)
    name = "mig_struct_encoder.source_conv"
    out = []
    for fn in (O.multi_gcn_encoder, O.multi_gcn_encoder_composed):
        P = {k: v.clone().requires_grad_(True) for k, v in O.synth_state_dict("mig", 45, dtype=torch.float64).items()
             if k.startswith(name + ".")}
        s = fn(P, name, x6, ei, 2, True)
        (s * w).sum().backward()
        out.append((s.detach(), {k: p.grad for k, p in P.items()}))
    (s0, g0), (s1, g1) = out
    assert rel(s1, s0) < 1e-12
    assert g0.keys() == g1.keys() and len(g0) == 14
    for k in g0:
        assert rel(g1[k], g0[k]) < 1e-12, (k, rel(g1[k], g0[k]))


def test_vae_matches_reference(golden_dir):
    v = load(golden_dir, "vae")
    s, t = v["s"].clone().requires_grad_(True), v["t"].clone().requires_grad_(True)
    V = {k: p.clone().requires_grad_(True) for k, p in v["params"].items()}
    zs, zt, (s_mu, s_ls, t_mu, t_ls) = O.vae_sample(V, s, t, v["eps_s"], v["eps_t"])
    kl = O.kl_loss(s_mu, s_ls, t_mu, t_ls, s.size(0))
    assert rel(zs.detach(), v["z_s"]) < 1e-6 and rel(zt.detach(), v["z_t"]) < 1e-6
    assert abs(float(kl) - float(v["kl"])) < 1e-6 * abs(float(v["kl"]))
    (kl * 1000.0 + (zs * zs).mean() + zt.sin().mean()).backward()
    assert rel(s.grad, v["grad_s"]) < 1e-5 and rel(t.grad, v["grad_t"]) < 1e-5
    for k, ref in v["grads"].items():
        assert rel(V[k].grad, ref) < 1e-5, k
