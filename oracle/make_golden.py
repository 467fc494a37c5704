"""Generate tests/golden/*.pt by executing the UNMODIFIED reference source
(the DG_VAE directory of the reference checkout, package ``deepgate``) under the
dependency shim in oracle/shim.

TEST INFRASTRUCTURE.  Needs the reference checkout; the tests only read the files:

    python oracle/make_golden.py <reference checkout>/DG_VAE    # writes tests/golden/<case>.pt

Each file holds the inputs (synthetic circuits, seeds in SURVEY.md section 8d form),
the weights (regenerable from ``oracle.dg_oracle.synth_state_dict(kind, seed)``, so
only the seed is stored), and what the reference produced: forward_level (top_sort),
the per-level / per-type incoming-edge lists (subgraph), hs, hf, the three losses
and the gradient of ``1*recon + 4*prob + 4*func`` w.r.t. every parameter.  A gradient
of more than GRAD_WHOLE entries is stored as a seeded sample of GRAD_SAMPLE of them
(``sampled_grad``), which keeps every file under 1 MB.
"""
import importlib.util
import os
import sys
import zlib

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if len(sys.argv) != 2:
    sys.exit("usage: python oracle/make_golden.py <reference checkout>/DG_VAE")
REFERENCE = os.path.abspath(sys.argv[1])
sys.path[:0] = [os.path.join(ROOT, "oracle", "shim"), REFERENCE, ROOT]

import deepgate                                              # noqa: E402  (the reference package)
import deepgate.dg_ae_model_aig, deepgate.dg_ae_model_mig    # noqa: E402,E401
import deepgate.dg_ae_model_xmg, deepgate.dg_ae_model_xag    # noqa: E402,E401
import deepgate.digae_layer, deepgate.digvae_model           # noqa: E402,E401
from deepgate import parser_func, parser_func_others         # noqa: E402
from deepgate.utils.dag_utils import subgraph, top_sort      # noqa: E402
from deepgate.utils.utils import zero_normalization          # noqa: E402
from torch_geometric.data import collate                     # noqa: E402  (shim)

from oracle.dg_oracle import GATE_MODULES, synth_state_dict  # noqa: E402

assert deepgate.__file__.startswith(REFERENCE + os.sep), deepgate.__file__
_spec = importlib.util.spec_from_file_location(
    "mgv_synth", os.path.join(ROOT, "multi-gate-vae_b200", "deepgate", "synth.py"))
synth = importlib.util.module_from_spec(_spec)
_spec.loader.exec_module(synth)

MODELS = {"aig": deepgate.dg_ae_model_aig.Model, "mig": deepgate.dg_ae_model_mig.Model,
          "xmg": deepgate.dg_ae_model_xmg.Model, "xag": deepgate.dg_ae_model_xag.Model}

# name: (model kind, gate mix, batch, n_pi, n_gates, window, num_rounds, cfg id, weight seed, with grads)
CASES = {
    "mig_b4_r1": ("mig", "mig4", 4, 16, 200, None, 1, 1, 11, True),
    "aig_b4_r1": ("aig", "aig", 4, 12, 160, None, 1, 2, 12, True),
    "xmg_b3_r2": ("xmg", "xmg", 3, 10, 150, 24, 2, 3, 13, True),
    "xag_b3_r1": ("xag", "xag", 3, 8, 120, 12, 1, 4, 14, False),
}
LOSS_W = (1.0, 4.0, 4.0)
GRAD_WHOLE, GRAD_SAMPLE = 1024, 512


def sampled_grad(name, t):
    """``t`` itself up to GRAD_WHOLE entries; above, GRAD_SAMPLE entries drawn with a seed taken from the parameter
    name, plus the largest |entry|, as {shape, index (flat, ascending), values, absmax} (tests/util.py reads both)."""
    if t is None or t.numel() <= GRAD_WHOLE:
        return t
    flat = t.reshape(-1)
    g = torch.Generator().manual_seed(zlib.crc32(name.encode()))
    idx = torch.unique(torch.cat([torch.randperm(flat.numel(), generator=g)[:GRAD_SAMPLE], flat.abs().argmax().reshape(1)]))
    return {"shape": tuple(t.shape), "index": idx.to(torch.int32), "values": flat[idx].clone(),
            "absmax": flat.abs().max().clone()}


def build_batch(kind, circuits):
    graphs = []
    for c in circuits:
        if kind == "aig":      # AIG on-disk layout: edge_index [2,E], tt_pair_index [2,P] (parser.py:100-119)
            g = parser_func.parse_pyg_mlpgate(c["x"], c["edge_index"].T.copy(), c["prob"], c["tt_sim"],
                                              c["tt_pair_index"].T.copy())
            g.gate = torch.tensor(c["x"][:, 1:2])
        else:                  # others: [E,2] / [P,2], transposed by the parser (parser_func_others.py:46-62)
            g = parser_func_others.parse_pyg_mlpgate(c["x"], c["edge_index"], c["prob"], c["tt_sim"],
                                                     c["tt_pair_index"])
        graphs.append(g)
    return collate(graphs)


def run_case(name):
    kind, mix, batch, n_pi, n_gates, window, rounds, cfg, wseed, with_grads = CASES[name]
    circuits = synth.make_circuits(mix, batch, n_pi, n_gates, cfg=cfg, window=window, n_pairs=48)
    G = build_batch(kind, circuits)
    enc = deepgate.digae_layer.DirectMultiGCNEncoder(dim_hidden=64, dim_feature=6, enable_reverse=True,
                                                     s_rounds=4, t_rounds=4, layernorm=True)
    model = MODELS[kind](struct_encoder=enc, num_rounds=rounds, dim_hidden=64)
    sd = synth_state_dict(kind, wseed)
    missing, unexpected = model.load_state_dict(sd, strict=False)
    assert not unexpected and all(k.endswith("num_batches_tracked") for k in missing), (missing, unexpected)
    model.eval()                                       # BatchNorm running stats, dropout off

    code = G.gate.squeeze(1).long()
    n = code.numel()
    # structural KATs straight from the reference's own functions
    level = top_sort(G.edge_index, n)
    assert torch.equal(level, G.forward_level.long())
    kat_nodes, kat_edges, kat_ptr = [], [], [0]
    for lv in range(1, int(level.max()) + 1):
        for gcode in sorted(GATE_MODULES[kind]):
            nodes = G.forward_index[(G.forward_level == lv) & (code == gcode)]
            if nodes.numel() == 0:
                continue
            sub, _ = subgraph(nodes, G.edge_index, dim=1)
            kat_nodes.append(torch.stack([torch.full_like(nodes, lv), torch.full_like(nodes, gcode), nodes]))
            kat_edges.append(sub)
            kat_ptr.append(kat_ptr[-1] + sub.size(1))

    g = torch.Generator().manual_seed(100 + cfg)
    E = G.edge_index.size(1)
    perm = torch.randperm(E, generator=g)
    pos_ei = G.edge_index[:, perm]
    neg_ei = torch.randint(0, n, (2, E), generator=g)

    hs, hf = model(G)
    rec, pred_bin, gt_bin = model.recon_loss(hs, pos_ei, neg_ei)
    prob = model.pred_prob(hf)
    prob_loss = torch.nn.L1Loss()(prob, G["prob"])
    a, b = hf[G["tt_pair_index"][0]], hf[G["tt_pair_index"][1]]
    dis = 1 - torch.cosine_similarity(a, b, eps=1e-8)
    func = torch.nn.L1Loss()(zero_normalization(dis), zero_normalization(G["tt_sim"]))
    total = LOSS_W[0] * rec + LOSS_W[1] * prob_loss + LOSS_W[2] * func
    out = {
        "case": name, "kind": kind, "mix": mix, "num_rounds": rounds, "weight_seed": wseed,
        "loss_weights": LOSS_W, "s_rounds": 4, "t_rounds": 4, "layernorm": True,
        "code": code.to(torch.int32), "edge_index": G.edge_index.clone(), "forward_level": level,
        "backward_level": G.backward_level.long(), "prob": G.prob.clone(),
        "tt_pair_index": G.tt_pair_index.clone(), "tt_sim": G.tt_sim.clone(),
        "train_pos_edge_index": pos_ei, "neg_edge_index": neg_ei,
        "kat_nodes": torch.cat(kat_nodes, dim=1).to(torch.int32), "kat_edges": torch.cat(kat_edges, dim=1),
        "kat_ptr": torch.tensor(kat_ptr),
        "hs": hs.detach().clone(), "hf": hf.detach().clone(),
        "recon_loss": rec.detach().clone(), "prob_loss": prob_loss.detach().clone(),
        "func_loss": func.detach().clone(), "total_loss": total.detach().clone(),
        "pred_bin": pred_bin.to(torch.int8),
    }
    if with_grads:
        total.backward()
        out["grads"] = {k: sampled_grad(k, p.grad.detach().clone() if p.grad is not None else None)
                        for k, p in model.named_parameters()}
    return out


def run_vae():
    """Reparameterisation (digvae_model.py:134-142) and KL (trainer.py:145-148), reference code."""
    torch.manual_seed(5)
    enc = torch.nn.Identity()
    vae = deepgate.digvae_model.DirectedGVAE(enc, 64, decoder=None)
    rng = np.random.default_rng(77)
    V = {}
    for k, p in sorted(vae.named_parameters()):
        V[k] = torch.tensor((rng.random(tuple(p.shape)) * 2 - 1) * 0.125, dtype=torch.float32)
        p.data.copy_(V[k])
    n = 160
    s = torch.tensor(rng.standard_normal((n, 64)), dtype=torch.float32, requires_grad=True)
    t = torch.tensor(rng.standard_normal((n, 64)), dtype=torch.float32, requires_grad=True)
    torch.manual_seed(9)
    eps_s, eps_t = torch.randn(n, 64), torch.randn(n, 64)
    torch.manual_seed(9)
    zs, zt = vae.sample(s, t)
    # trainer.py:145-148 verbatim (u.size(0) == v.size(0) == number of nodes)
    s_kl = -0.5 / n * (1 + 2 * vae.s_logstd - vae.s_mu ** 2 - torch.exp(vae.s_logstd) ** 2).sum(1).mean()
    t_kl = -0.5 / n * (1 + 2 * vae.t_logstd - vae.t_mu ** 2 - torch.exp(vae.t_logstd) ** 2).sum(1).mean()
    kl = s_kl + t_kl
    obj = kl * 1000.0 + (zs * zs).mean() + (zt.sin()).mean()
    obj.backward()
    return {"params": V, "s": s.detach(), "t": t.detach(), "eps_s": eps_s, "eps_t": eps_t,
            "z_s": zs.detach(), "z_t": zt.detach(), "kl": kl.detach(),
            "s_mu": vae.s_mu.detach(), "s_logstd": vae.s_logstd.detach(),
            "grad_s": s.grad.clone(), "grad_t": t.grad.clone(),
            "grads": {k: p.grad.clone() for k, p in vae.named_parameters()}}


def run_kats():
    """SURVEY.md section 3.3 / section 8c structural known-answer tests, evaluated by the reference."""
    ei = torch.tensor([[0, 1, 2, 3, 0, 4, 1, 5, 5], [3, 3, 3, 4, 4, 5, 5, 6, 7]])
    lv = top_sort(ei, 9)
    sub, _ = subgraph(torch.tensor([5, 3]), ei, dim=1)
    return {"edge_index": ei, "top_sort": lv, "subgraph_5_3": sub}


if __name__ == "__main__":
    dst = os.path.join(ROOT, "tests", "golden")
    os.makedirs(dst, exist_ok=True)
    torch.save(run_kats(), os.path.join(dst, "kats.pt"))
    torch.save(run_vae(), os.path.join(dst, "vae.pt"))
    for name in CASES:
        res = run_case(name)
        torch.save(res, os.path.join(dst, name + ".pt"))
        print(name, "N=%d E=%d L=%d" % (res["code"].numel(), res["edge_index"].size(1),
                                         int(res["forward_level"].max()) + 1),
              "recon %.6f prob %.6f func %.6f" % (res["recon_loss"], res["prob_loss"], res["func_loss"]))
