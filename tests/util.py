"""Shared helpers for the parity tests."""
import os

import torch

from oracle import dg_oracle as O

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
KIND_MODULE = {"aig": "dg_ae_model_aig", "mig": "dg_ae_model_mig", "xmg": "dg_ae_model_xmg", "xag": "dg_ae_model_xag"}
ZERO_GRAD_TAGS = (".msg_q.", "msg_k.bias", "attn_lin.bias")


def load_golden(name):
    return torch.load(os.path.join(GOLDEN, name + ".pt"), weights_only=False)


def is_sampled(ref):
    """A golden tensor stored as a seeded sample of its entries (oracle/make_golden.py: ``shape``, flat ``index``,
    ``values`` and the whole tensor's ``absmax``)."""
    return isinstance(ref, dict)


def absmax(ref):
    """max |ref| over the whole tensor, also for a sampled golden tensor."""
    return float(ref["absmax"]) if is_sampled(ref) else float(ref.detach().abs().max())


def maxdiff(got, ref):
    """max |got - ref| over the entries the golden tensor holds (all of them, or its sample)."""
    got = got.detach().double().cpu()
    if is_sampled(ref):
        assert tuple(got.shape) == tuple(ref["shape"]), (tuple(got.shape), ref["shape"])
        got, ref = got.reshape(-1)[ref["index"].long()], ref["values"]
    return float((got - ref.detach().double().cpu()).abs().max())


def rel(a, b):
    """max |a - b| / max |b| (max-norm relative error); ``b`` may be a sampled golden tensor."""
    if is_sampled(b):
        return maxdiff(a, b) / max(absmax(b), 1e-30)
    a, b = a.detach().double().cpu(), b.detach().double().cpu()
    return float((a - b).abs().max() / b.abs().max().clamp_min(1e-30))


def build_model(kind, state_dict, num_rounds=1, device="cuda", s_rounds=4, t_rounds=4, layernorm=True, variational=False):
    import deepgate
    enc = deepgate.digae_layer.DirectMultiGCNEncoder(dim_hidden=64, dim_feature=6, enable_reverse=True,
                                                     s_rounds=s_rounds, t_rounds=t_rounds, layernorm=layernorm)
    kw = {"variational": True} if variational else {}
    model = getattr(deepgate, KIND_MODULE[kind]).Model(struct_encoder=enc, num_rounds=num_rounds, dim_hidden=64, **kw)
    missing, unexpected = model.load_state_dict(state_dict, strict=False)
    assert not unexpected and all(k.endswith("num_batches_tracked") for k in missing), (missing, unexpected)
    return model.to(device).eval()


def batch_from_arrays(code, edge_index, forward_level, prob, tt_pair_index, tt_sim, device="cuda"):
    """A batch object with the fields Model.forward / Trainer.run_batch read."""
    from deepgate.data import OrderedData
    code = code.long()
    g = OrderedData(x=torch.nn.functional.one_hot(code, 6).float(), edge_index=edge_index.long(),
                    gate=code.float().unsqueeze(1), forward_level=forward_level.long(),
                    forward_index=torch.arange(code.numel()), prob=prob.float().reshape(-1, 1),
                    tt_pair_index=tt_pair_index.long(), tt_sim=tt_sim.float())
    return g.to(device)


def oracle_inputs(batch, pos_ei, neg_ei):
    G = {"code": batch.gate.reshape(-1).long().cpu(), "edge_index": batch.edge_index.cpu(),
         "forward_level": batch.forward_level.cpu(), "prob": batch.prob.cpu(),
         "tt_pair_index": batch.tt_pair_index.cpu(), "tt_sim": batch.tt_sim.cpu(),
         "train_pos_edge_index": pos_ei.cpu(), "neg_edge_index": neg_ei.cpu()}
    return G


def check_grads(named_grads, ref_grads, tol, what=""):
    """Element-relative (max-norm) for ordinary tensors; scale-relative for the tensors whose
    reference gradient is mathematically zero (SURVEY.md section 7 hard part 3)."""
    worst = 0.0
    for k, ref in ref_grads.items():
        got = named_grads.get(k)
        if ref is None:
            assert got is None or float(got.abs().max()) == 0.0, k
            continue
        assert got is not None, "no gradient for %s" % k
        if any(t in k for t in ZERO_GRAD_TAGS):
            scale = absmax(ref_grads[k.split(".")[0] + ".msg_k.weight"])
            assert float(got.abs().max()) <= 1e-4 * scale + 1e-12, (what, k)
            continue
        if k.endswith("attn_lin.weight") or k.endswith("msg_k.weight"):
            # attention parameters: exactly zero for fan-in-1 gates (alpha == 1), and the query half of
            # attn_lin.weight is mathematically zero -> absolute floor tied to the value path's scale (only reached by
            # the fan-in-1 codes; for the others the bound is tol * max |ref|, the plain max-norm relative bar)
            vscale = absmax(ref_grads[k.split(".")[0] + ".msg_v.weight"])
            floor = tol * max(absmax(ref), 1e-3 * vscale)
            if k.endswith("attn_lin.weight"):
                assert float(got[:, :64].abs().max()) <= floor + 1e-12, (what, k)
                got, ref = got[:, 64:], ref[:, 64:]
            err = maxdiff(got, ref)
            assert err <= floor, (what, k, err, floor)
            continue
        r = rel(got, ref)
        worst = max(worst, r)
        assert r < tol, (what, k, r)
    return worst


def oracle_train_grads(kind, state_dict, G, weights, num_rounds, dtype=torch.float32, **kw):
    P = {k: v.clone().to(dtype) if v.is_floating_point() else v.clone() for k, v in state_dict.items()}
    for k, p in P.items():
        p.requires_grad_("running" not in k)
    Gd = dict(G)
    for k in ("prob", "tt_sim"):
        Gd[k] = G[k].to(dtype)
    total, parts = O.train_step_losses(P, kind, Gd, weights, num_rounds, literal_subgraph=False, **kw)
    total.backward()
    grads = {k: p.grad for k, p in P.items() if p.requires_grad}
    return total.detach(), {k: v.detach() for k, v in parts.items()}, grads
