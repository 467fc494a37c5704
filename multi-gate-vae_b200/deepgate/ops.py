"""Autograd bindings of the CUDA kernels (libmgv_b200.so) for the hot path.

  level_sweep(...)        dg_ae_model_*.py level loop  (TFMlpAggr + GRU per level / gate code)
  struct_encoder(...)     MultiGCNEncoder x {source, target}  (digae_layer.py:257-297)
  vae_func_loss(...)      reparam + KL + func loss  (digvae_model.py:134-142, trainer.py:145-163)

Every function fails loudly when its inputs are not on a CUDA device or the library is
missing; nothing here falls back to PyTorch ops for the arithmetic.
"""
import ctypes
import os

import torch

from . import _native as nat

_AGGR_KEYS = ("attn_lin.weight", "attn_lin.bias", "msg_q.weight", "msg_q.bias", "msg_k.weight", "msg_k.bias",
              "msg_v.weight", "msg_v.bias")
_GRU_KEYS = ("weight_ih_l0", "weight_hh_l0", "bias_ih_l0", "bias_hh_l0")
PARAMS_PER_CODE = len(_AGGR_KEYS) + len(_GRU_KEYS)      # 12


# Arithmetic of the tensor-core products: "fp32" (default; fp16 hi/lo planes, fp32-accurate) or "bf16" (one bf16 plane,
# fp32 accumulation; embeddings / gradients within 2e-2 -- the stated tolerance of the bf16 configuration).  Read at
# forward time; the backward of a graph uses the precision of its forward.
PRECISION = "fp32"


def set_precision(name):
    global PRECISION
    if name not in ("fp32", "bf16"):
        raise ValueError("precision must be 'fp32' or 'bf16'")
    PRECISION = name


def _prec():
    return nat.PRECISION_BF16 if PRECISION == "bf16" else nat.PRECISION_FP32


# Optional per-kernel timing (bench.py): PROFILE = {} enables CUDA-event brackets around each
# library call on the launching stream; entries are name -> [(start_event, end_event), ...].
PROFILE = None


class _timed(object):
    def __init__(self, name, device):
        self.name, self.device = name, device

    def __enter__(self):
        if PROFILE is not None:
            self.ev = (torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))
            self.ev[0].record(torch.cuda.current_stream(self.device))
        return self

    def __exit__(self, *exc):
        if PROFILE is not None:
            self.ev[1].record(torch.cuda.current_stream(self.device))
            PROFILE.setdefault(self.name, []).append(self.ev)
        return False


def profile_summary():
    """name -> (calls, total ms); call after torch.cuda.synchronize()."""
    return {k: (len(v), sum(a.elapsed_time(b) for a, b in v)) for k, v in (PROFILE or {}).items()}


def _f32(t, name):
    # fast path (called ~100 times per training step): a contiguous fp32 CUDA tensor is used as is -- callers take its pointer
    # or use it inside an autograd.Function, where grad mode is off; a detach() per parameter costs the host 0.3 ms a step
    if t.is_cuda and t.dtype == torch.float32 and t.is_contiguous():
        return t
    return nat.require_cuda(t.detach().contiguous(), name, torch.float32)


# =========================================================================== level sweep
def _ptr_table(tensors):
    return (ctypes.c_void_p * len(tensors))(*[t.data_ptr() for t in tensors])


def _code_table(codes):
    return (ctypes.c_int32 * len(codes))(*codes)


def _sweep_tables(params, codes):
    """Pointer table of the parameters mgv_sweep_pack / mgv_sweep_unpack_grads read, per listed gate code."""
    D = nat.D
    sel = []
    for i in range(len(codes)):
        aw, ab, qw, qb, kw, kb, vw, vb, wih, whh, bih, bhh = params[i * PARAMS_PER_CODE:(i + 1) * PARAMS_PER_CODE]
        if tuple(vw.shape) != (D, 2 * D) or tuple(wih.shape) != (3 * D, D):
            raise RuntimeError("mgv_b200: level sweep kernels are built for dim_hidden=%d" % D)
        sel += [_f32(t, "sweep parameter") for t in (aw, kw, vw, vb, wih, whh, bih, bhh)]
    return sel


def _sweep_pack(params, codes, device, prec):
    """Natural weight blocks [8][66112] + the tensor-core weight images (include/mgv_b200.h), one launch."""
    lib = nat.lib()
    pack = torch.zeros(lib.mgv_sweep_pack_bytes() // 4, dtype=torch.float32, device=device)
    sel = _sweep_tables(params, codes)
    with nat.on_device(device), _timed("sweep_pack", device):
        nat.check(lib.mgv_sweep_pack(_ptr_table(sel), _code_table(codes), len(codes), nat.ptr(pack), prec,
                                     nat.stream_of(device)), "mgv_sweep_pack")
    return pack


class LevelSweepFunction(torch.autograd.Function):
    @staticmethod
    def forward(ctx, hs, sched, rounds, codes, *params):
        lib = nat.lib()
        dev = hs.device
        hs_c = _f32(hs, "hs")
        N = sched.N
        if hs_c.shape != (N, nat.D):
            raise RuntimeError("mgv_b200: hs must be [N, %d]" % nat.D)
        mask = 0
        for c in codes:
            mask |= 1 << c
        prec = _prec()
        pack = _sweep_pack(params, codes, dev, prec)
        hf_all = torch.zeros(rounds, max(N, 1), nat.D, dtype=torch.float32, device=dev)
        sync = torch.empty(64, dtype=torch.int32, device=dev)          # zeroed by the call
        with nat.on_device(dev):
            with _timed("level_sweep_fwd", dev):
              nat.check(lib.mgv_level_sweep_fwd(sched.c_struct(), rounds, mask, nat.ptr(pack), nat.ptr(hs_c),
                                              nat.ptr(hf_all), nat.ptr(sync), prec, nat.stream_of(dev)),
                      "mgv_level_sweep_fwd")
        ctx.sched, ctx.rounds, ctx.codes, ctx.mask, ctx.prec = sched, rounds, tuple(codes), mask, prec
        ctx.save_for_backward(hs_c, hf_all, pack, *params)
        ctx.launches = 1
        return hf_all[rounds - 1][:N]

    @staticmethod
    def backward(ctx, g_hf):
        lib = nat.lib()
        hs_c, hf_all, pack = ctx.saved_tensors[:3]
        params = ctx.saved_tensors[3:]
        sched, rounds, codes = ctx.sched, ctx.rounds, ctx.codes
        dev = hs_c.device
        N, D = sched.N, nat.D
        ghs = torch.zeros(max(N, 1), D, dtype=torch.float32, device=dev)
        if N > 0:
            ghf = g_hf.to(torch.float32).contiguous().clone()             # in/out for the library: a private copy
        else:
            ghf = torch.zeros(1, D, dtype=torch.float32, device=dev)
        grads = torch.empty(nat.NCODE, nat.SWEEP_GRAD_FLOATS, dtype=torch.float32, device=dev)
        sync = torch.empty(64, dtype=torch.int32, device=dev)          # zeroed by the call
        with nat.on_device(dev):
            nb = lib.mgv_sweep_bwd_workspace_bytes(N, sched.E)
            ws = nat.workspace(nb, dev)
            with _timed("level_sweep_bwd", dev):
              nat.check(lib.mgv_level_sweep_bwd(sched.c_struct(), rounds, ctx.mask, nat.ptr(pack), nat.ptr(hs_c),
                                              nat.ptr(hf_all), nat.ptr(ghs), nat.ptr(ghf), nat.ptr(grads),
                                              nat.ptr(ws), nb, nat.ptr(sync), ctx.prec, nat.stream_of(dev)),
                      "mgv_level_sweep_bwd")
        sel = _sweep_tables(params, codes)
        extra = torch.empty(max(len(codes), 1), 128 + D * 2 * D, dtype=torch.float32, device=dev)
        # query / key-bias / attn-bias cancel in the softmax: exact zeros, one DISJOINT slice per parameter (gradients must not alias)
        ZQ = 1 + D * 2 * D + 2 * D
        zero = torch.zeros(max(len(codes), 1), ZQ, dtype=torch.float32, device=dev)
        with nat.on_device(dev), _timed("sweep_unpack_grads", dev):
            nat.check(lib.mgv_sweep_unpack_grads(_ptr_table(sel), _code_table(list(codes)), len(codes), nat.ptr(grads),
                                                 nat.ptr(extra), nat.stream_of(dev)), "mgv_sweep_unpack_grads")
        out = []
        for i, c in enumerate(codes):
            g = grads[c]
            z = zero[i]
            out += [extra[i, :128].view(1, 2 * D), z[:1], z[1:1 + D * 2 * D].view(D, 2 * D), z[1 + D * 2 * D:1 + D * 2 * D + D],
                    extra[i, 128:].view(D, 2 * D), z[1 + D * 2 * D + D:],
                    g[128:8320].view(D, 2 * D), g[8320:8384],
                    g[8384:20672].view(3 * D, D), g[20672:32960].view(3 * D, D), g[32960:33152], g[33152:33344]]
        return (ghs[:N], None, None, None) + tuple(out)


def level_sweep(hs, sched, rounds, codes, modules):
    """hf [N, 64] after ``rounds`` sweeps.  ``modules`` = [(TFMlpAggr, nn.GRU)] aligned with ``codes``."""
    params = []
    for aggr, gru in modules:
        sd = dict(aggr.named_parameters())
        params += [sd[k] for k in _AGGR_KEYS]
        gd = dict(gru.named_parameters())
        params += [gd[k] for k in _GRU_KEYS]
    return LevelSweepFunction.apply(hs, sched, int(rounds), tuple(int(c) for c in codes), *params)


# =========================================================================== small Linear layers (one row per node)
def _linear_tc(inp, weight, bias, P, Q, transposed):
    """out[N][P] = inp[N][Q] . M[P][Q]^T (+ bias) on the tensor cores (csrc/linear_tc.cu)."""
    dev = inp.device
    N = inp.shape[0]
    out = torch.empty(N, P, dtype=torch.float32, device=dev)
    lib = nat.lib()
    with nat.on_device(dev), _timed("linear_tc", dev):
        nat.check(lib.mgv_linear_tc(nat.ptr(inp), N, nat.ptr(weight), nat.ptr(bias), P, Q, int(transposed), nat.ptr(out),
                                    nat.stream_of(dev)), "mgv_linear_tc")
    return out


def _tc_shape(weight):
    return weight.shape[0] in (64, 128) and weight.shape[1] in (64, 128) and not os.environ.get("MGV_LINEAR_TORCH")


class LinearFunction(torch.autograd.Function):
    """y = x W^T + b.  Forward and d x: tcgen05 tiles over the nodes (csrc/linear_tc.cu) for 64 / 128-wide layers, library
    GEMMs otherwise; d W / d b sum over the NODES into at most 128 x 128 outputs -- one tile on one SM for a library GEMM --
    and run in csrc/linear.cu."""

    @staticmethod
    def forward(ctx, x, weight, bias):
        nat.require_cuda(x, "x")
        x_c = _f32(x, "x")
        ctx.save_for_backward(x_c, weight)
        ctx.has_bias = bias is not None
        if _tc_shape(weight) and x_c.shape[0] > 0:
            O, I = weight.shape
            return _linear_tc(x_c, _f32(weight, "weight"), None if bias is None else _f32(bias, "bias"), O, I, False)
        return torch.addmm(bias, x_c, weight.t()) if bias is not None else x_c @ weight.t()

    @staticmethod
    def backward(ctx, gy):
        x_c, weight = ctx.saved_tensors
        dev = x_c.device
        gy_c = _f32(gy, "gy")
        O, I = weight.shape
        N = x_c.shape[0]
        if not ctx.needs_input_grad[0]:
            gx = None
        elif _tc_shape(weight) and N > 0:
            gx = _linear_tc(gy_c, _f32(weight, "weight"), None, I, O, True)
        else:
            gx = gy_c @ weight
        dW = torch.empty_like(weight, dtype=torch.float32)
        db = torch.empty(O, dtype=torch.float32, device=dev) if ctx.has_bias else None
        lib = nat.lib()
        with nat.on_device(dev):
            nb = lib.mgv_linear_wgrad_workspace_bytes(N, I, O)
            ws = nat.workspace(nb, dev)
            with _timed("linear_wgrad", dev):
                nat.check(lib.mgv_linear_wgrad(nat.ptr(x_c), nat.ptr(gy_c), N, I, O, nat.ptr(dW), nat.ptr(db) if db is not None else None,
                                               nat.ptr(ws), nb, nat.stream_of(dev)), "mgv_linear_wgrad")
        return gx, dW, db


def linear(x, weight, bias=None):
    if x.dim() != 2 or weight.shape[0] > 128 or weight.shape[1] > 128 or not x.is_cuda:
        return torch.nn.functional.linear(x, weight, bias)      # shapes outside the kernel's range: plain library path
    return LinearFunction.apply(x, weight, bias)


class Linear(torch.nn.Linear):
    """nn.Linear (same parameters / checkpoint keys) whose weight gradient runs in csrc/linear.cu."""

    def forward(self, x):
        return linear(x, self.weight, self.bias)


# =========================================================================== struct encoder
_S_WCX, _S_WHH, _S_BC, _S_BIH, _S_BHH, _S_LNW, _S_LNB = 0, 14592, 27648, 27840, 28032, 28224, 28288
_LDC, _LDM = 76, 68


def _struct_pack(enc_params, layernorm, device):
    """[num_enc][2][28416] weight blocks (include/mgv_b200.h), one launch.  enc_params[e] = (aggr.w, aggr.b, upd.wih, upd.whh,
    upd.bih, upd.bhh, aggr_r.w, aggr_r.b, upd_r.wih, upd_r.whh, upd_r.bih, upd_r.bhh[, ln.w, ln.b]).
    The AggConv linear is pre-composed into the GRU input weights: Wc = wih[:, :64] @ w, bc = wih[:, :64] @ b."""
    D = nat.D
    flat = []
    feat = None
    for ps in enc_params:
        for d in range(2):
            w, wih = ps[6 * d], ps[6 * d + 2]
            f = wih.shape[1] - D
            if tuple(w.shape) != (D, D) or f < 0 or f > nat.MAX_FEAT or (feat is not None and f != feat):
                raise RuntimeError("mgv_b200: struct encoder kernels need dim_hidden=%d, dim_feature<=%d" % (D, nat.MAX_FEAT))
            feat = f
        flat += [_f32(t, "struct encoder parameter") for t in ps]
    pack = torch.empty(len(enc_params), 2, nat.STRUCT_PACK_FLOATS, dtype=torch.float32, device=device)
    with torch.cuda.device(device), _timed("struct_pack", device):
        nat.check(nat.lib().mgv_struct_pack(_ptr_table(flat), len(enc_params), int(bool(layernorm)), feat, nat.ptr(pack),
                                            nat.stream_of(device)), "mgv_struct_pack")
    return pack


class StructEncoderFunction(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, csr, rounds, layernorm, num_enc, *params):
        lib = nat.lib()
        dev = x.device
        x_c = _f32(x.to(torch.float32), "x")
        N = csr.N
        feat = int(x_c.shape[1])
        per = len(params) // num_enc
        enc_params = [params[e * per:(e + 1) * per] for e in range(num_enc)]
        prec = _prec()
        pack = _struct_pack(enc_params, layernorm, dev)
        states = torch.empty(num_enc, 2, max(N, 1), nat.D, dtype=torch.float32, device=dev)     # ping-pong slots
        # training: the forward also saves every step's tensor-core operand tile; the backward recomputes from those
        # instead of gathering the neighbour sums a second time (bf16 mode: the single bf16 plane of each tile)
        need_tiles = N > 0 and any(ctx.needs_input_grad[5:])
        tiles = (torch.empty(lib.mgv_struct_tiles_bytes(N, num_enc, rounds), dtype=torch.uint8, device=dev)
                 if need_tiles else None)
        with nat.on_device(dev):
            nb = lib.mgv_struct_fwd_workspace_bytes(N, num_enc)
            ws = nat.workspace(nb, dev)
            with _timed("struct_encoder_fwd", dev):
              nat.check(lib.mgv_struct_encoder_fwd(csr.c_struct(), num_enc, rounds, int(layernorm), feat,
                                                 nat.ptr(x_c), nat.ptr(pack), nat.ptr(states), nat.ptr(tiles), nat.ptr(ws), nb,
                                                 prec, nat.stream_of(dev)),
                      "mgv_struct_encoder_fwd")
        ctx.tiles = tiles
        ctx.csr, ctx.rounds, ctx.layernorm, ctx.num_enc, ctx.feat, ctx.per = csr, rounds, layernorm, num_enc, feat, per
        ctx.prec = prec
        ctx.save_for_backward(x_c, pack)
        ctx.saved_params = params
        # one output per encoder (views of slot 0, which the last step writes): indexing a stacked [num_enc, N, 64] output costs
        # the backward two zero-fills, two slice copies and an add of N x 64 tensors (autograd's select backward), 50 us at cfg2
        return tuple(states[e, 0, :N] for e in range(num_enc))

    @staticmethod
    def backward(ctx, *gouts):
        lib = nat.lib()
        x_c, pack = ctx.saved_tensors
        csr, rounds, num_enc, feat, per = ctx.csr, ctx.rounds, ctx.num_enc, ctx.feat, ctx.per
        dev = x_c.device
        N, D = csr.N, nat.D
        if N > 0:
            g = torch.empty(num_enc, N, D, dtype=torch.float32, device=dev)
            for e in range(num_enc):
                if gouts[e] is None:
                    g[e].zero_()
                else:
                    g[e].copy_(gouts[e])
        else:
            g = torch.zeros(num_enc, 1, D, dtype=torch.float32, device=dev)
        grads = torch.empty(num_enc, 2, nat.STRUCT_GRAD_FLOATS, dtype=torch.float32, device=dev)
        with nat.on_device(dev):
            nb = lib.mgv_struct_bwd_workspace_bytes(N, num_enc)
            ws = nat.workspace(nb, dev)
            with _timed("struct_encoder_bwd", dev):
              nat.check(lib.mgv_struct_encoder_bwd(csr.c_struct(), num_enc, rounds, int(ctx.layernorm), feat,
                                                 nat.ptr(x_c), nat.ptr(pack), nat.ptr(ctx.tiles), nat.ptr(g),
                                                 nat.ptr(grads), nat.ptr(ws), nb, ctx.prec, nat.stream_of(dev)),
                      "mgv_struct_encoder_bwd")
        params = ctx.saved_params
        ldw = D + feat
        per_dir = D * D + D + 3 * D * ldw + 3 * D * D + 6 * D
        per_enc = 2 * per_dir + (2 * D if ctx.layernorm else 0)
        flat = [_f32(t, "struct encoder parameter") for t in params]
        buf = torch.empty(num_enc, per_enc, dtype=torch.float32, device=dev)
        with nat.on_device(dev), _timed("struct_unpack_grads", dev):
            nat.check(lib.mgv_struct_unpack_grads(_ptr_table(flat), num_enc, int(bool(ctx.layernorm)), feat, nat.ptr(grads),
                                                  nat.ptr(buf), nat.stream_of(dev)), "mgv_struct_unpack_grads")
        # one split per encoder (a C++ loop) instead of a Python slice per parameter
        shapes = [(D, D), (D,), (3 * D, ldw), (3 * D, D), (3 * D,), (3 * D,)] * 2 + ([(D,), (D,)] if ctx.layernorm else [])
        counts = [shp[0] * (shp[1] if len(shp) > 1 else 1) for shp in shapes]
        out = []
        for e in range(num_enc):
            out += [v if len(shp) == 1 else v.view(shp) for v, shp in zip(buf[e].split(counts), shapes)]
        return (None, None, None, None, None) + tuple(out)


def struct_encoder(x, csr, rounds, layernorm, encoders):
    """Final node states of ``encoders`` (MultiGCNEncoder modules, same rounds): a tuple of num_enc tensors [N, 64]."""
    params = []
    for enc in encoders:
        params += [enc.aggr.msg.weight, enc.aggr.msg.bias, enc.update.weight_ih_l0, enc.update.weight_hh_l0,
                   enc.update.bias_ih_l0, enc.update.bias_hh_l0,
                   enc.aggr_r.msg.weight, enc.aggr_r.msg.bias, enc.update_r.weight_ih_l0, enc.update_r.weight_hh_l0,
                   enc.update_r.bias_ih_l0, enc.update_r.bias_hh_l0]
        if layernorm:
            params += [enc.ln.weight, enc.ln.bias]
    return StructEncoderFunction.apply(x, csr, int(rounds), bool(layernorm), len(encoders), *params)


# =========================================================================== reconstruction loss + negative sampler
_NEG_COUNTER = [0]


def negative_sample(csr, count):
    """``count`` random ordered node pairs that are neither self loops nor edges of ``csr`` (device kernel, no host
    sync) -- the role of torch_geometric.utils.negative_sampling at dg_ae_model_mig.py:177-180.  Seeded from
    torch's global seed and a call counter."""
    lib = nat.lib()
    dev = csr.device
    if csr.N < 2:
        raise RuntimeError("mgv_b200: negative sampling needs at least 2 nodes")
    neg = torch.empty(2, int(count), dtype=torch.int64, device=dev)
    _NEG_COUNTER[0] += 1
    seed = (torch.initial_seed() * 0x9E3779B97F4A7C15 + _NEG_COUNTER[0]) & 0xFFFFFFFFFFFFFFFF
    with nat.on_device(dev):
        nat.check(lib.mgv_negative_sample(nat.ptr(csr.out_ptr), nat.ptr(csr.out_pack), csr.N, int(count), seed,
                                          nat.ptr(neg), nat.stream_of(dev)), "mgv_negative_sample")
    return neg


def permute_edges(edge_index):
    """``edge_index[:, perm]`` for a pseudo-random permutation of the edges, one launch (csrc/recon.cu, ``mgv_permute_edges``):
    the per-batch edge split of the training loop (preprocessing.py:8-83 with val_ratio = test_ratio = 0).  Seeded from torch's
    global seed and a call counter."""
    ei = nat.require_cuda(edge_index.contiguous(), "edge_index", torch.int64)
    if ei.dim() != 2 or ei.shape[0] != 2:
        raise RuntimeError("mgv_b200: edge_index must be [2, E]")
    out = torch.empty_like(ei)
    _NEG_COUNTER[0] += 1
    seed = (torch.initial_seed() * 0xD1B54A32D192ED03 + _NEG_COUNTER[0]) & 0xFFFFFFFFFFFFFFFF
    with nat.on_device(ei.device):
        nat.check(nat.lib().mgv_permute_edges(nat.ptr(ei), int(ei.shape[1]), seed, nat.ptr(out), nat.stream_of(ei.device)),
                  "mgv_permute_edges")
    return out


class ReconLossFunction(torch.autograd.Function):
    @staticmethod
    def forward(ctx, st, pos, neg):
        lib = nat.lib()
        dev = st.device
        st_c = _f32(st, "st")
        N = int(st_c.shape[0])
        if st_c.dim() != 2 or st_c.shape[1] != 2 * nat.D:
            raise RuntimeError("mgv_b200: recon loss expects hs_decompose(hs) of shape [N, %d]" % (2 * nat.D))
        pos_c = nat.require_cuda(pos.contiguous(), "pos_edge_index", torch.int64)
        neg_c = nat.require_cuda(neg.contiguous(), "neg_edge_index", torch.int64)
        Ep, En = int(pos_c.shape[1]), int(neg_c.shape[1])
        out = torch.empty(3, dtype=torch.float32, device=dev)
        sig = torch.empty(max(Ep + En, 1), dtype=torch.float32, device=dev)
        pred = torch.empty(max(Ep + En, 1), dtype=torch.int32, device=dev)
        ws = nat.workspace(16, dev)
        from .schedule import error_word
        with nat.on_device(dev):
            with _timed("recon_loss_fwd", dev):
              nat.check(lib.mgv_recon_loss_fwd(nat.ptr(st_c), N, nat.ptr(pos_c), Ep, nat.ptr(neg_c), En, nat.ptr(out),
                                             nat.ptr(sig), nat.ptr(pred), nat.ptr(ws), 16, nat.ptr(error_word(dev)),
                                             nat.stream_of(dev)), "mgv_recon_loss_fwd")
        ctx.save_for_backward(st_c, pos_c, neg_c, sig)
        ctx.mark_non_differentiable(pred)
        return out[0], pred[:Ep + En]

    @staticmethod
    def backward(ctx, g_loss, _g_pred):
        lib = nat.lib()
        st_c, pos_c, neg_c, sig = ctx.saved_tensors
        dev = st_c.device
        gst = torch.zeros_like(st_c)
        gl = g_loss.detach().to(torch.float32).reshape(1).contiguous()
        with nat.on_device(dev):
            with _timed("recon_loss_bwd", dev):
              nat.check(lib.mgv_recon_loss_bwd(nat.ptr(st_c), int(st_c.shape[0]), nat.ptr(pos_c), int(pos_c.shape[1]),
                                             nat.ptr(neg_c), int(neg_c.shape[1]), nat.ptr(sig), nat.ptr(gl), nat.ptr(gst),
                                             nat.stream_of(dev)), "mgv_recon_loss_bwd")
        return gst, None, None


def recon_loss(st, pos_edge_index, neg_edge_index):
    """(loss, pred_bin int32 [Ep + En]) of the directed inner-product decoder over ``st = [s | t]``."""
    return ReconLossFunction.apply(st, pos_edge_index, neg_edge_index)


# =========================================================================== reparam + KL + func loss
class VaeFuncLossFunction(torch.autograd.Function):
    @staticmethod
    def forward(ctx, mu, logstd, eps, hf, pair, tt_sim):
        """mu/logstd/eps [2,N,64] or None; hf [Nf,64], pair [2,P] int64, tt_sim [P] or None.
        Returns (z [2,N,64], kl, func_loss)."""
        lib = nat.lib()
        has_vae, has_func = mu is not None, pair is not None
        dev = mu.device if has_vae else hf.device
        N = int(mu.shape[1]) if has_vae else 0
        P = int(pair.shape[1]) if has_func else 0
        mu_c = _f32(mu, "mu") if has_vae else None
        ls_c = _f32(logstd, "logstd") if has_vae else None
        eps_c = _f32(eps, "eps") if has_vae else None
        hf_c = _f32(hf, "hf") if has_func else None
        pair_c = nat.require_cuda(pair.contiguous(), "tt_pair_index", torch.int64) if has_func else None
        tt_c = _f32(tt_sim.to(torch.float32), "tt_sim") if has_func else None
        z = torch.empty(2, N, nat.D, dtype=torch.float32, device=dev)
        out = torch.zeros(8, dtype=torch.float32, device=dev)
        with nat.on_device(dev):
            nb = lib.mgv_vae_func_workspace_bytes(P)
            ws = nat.workspace(nb, dev, zero=True)
            with _timed("vae_func_loss_fwd", dev):
              nat.check(lib.mgv_vae_func_loss_fwd(nat.ptr(mu_c), nat.ptr(ls_c), nat.ptr(eps_c), nat.ptr(z), N,
                                                nat.ptr(hf_c), nat.ptr(pair_c), nat.ptr(tt_c), P, nat.ptr(out),
                                                nat.ptr(ws), nb, nat.stream_of(dev)), "mgv_vae_func_loss_fwd")
        ctx.N, ctx.P, ctx.has_vae, ctx.has_func = N, P, has_vae, has_func
        ctx.hf_shape = tuple(hf.shape) if has_func else None
        ctx.save_for_backward(mu_c, ls_c, eps_c, hf_c, pair_c, tt_c, out, ws)
        return z, out[0].clone(), out[1].clone()

    @staticmethod
    def backward(ctx, gz, gkl, gfunc):
        lib = nat.lib()
        mu_c, ls_c, eps_c, hf_c, pair_c, tt_c, out, ws = ctx.saved_tensors
        dev = out.device
        N, P = ctx.N, ctx.P
        g2 = torch.zeros(2, dtype=torch.float32, device=dev)
        if gkl is not None:
            g2[0] = gkl
        if gfunc is not None:
            g2[1] = gfunc
        gmu = gls = ghf = None
        gz_c = None
        if ctx.has_vae:
            gz_c = _f32(gz, "gz") if gz is not None else torch.zeros(2, N, nat.D, dtype=torch.float32, device=dev)
            gmu, gls = torch.empty_like(mu_c), torch.empty_like(mu_c)
        if ctx.has_func:
            ghf = torch.zeros(ctx.hf_shape, dtype=torch.float32, device=dev)
        with nat.on_device(dev):
            with _timed("vae_func_loss_bwd", dev):
              nat.check(lib.mgv_vae_func_loss_bwd(nat.ptr(g2), nat.ptr(gz_c), nat.ptr(mu_c), nat.ptr(ls_c),
                                                nat.ptr(eps_c), nat.ptr(gmu), nat.ptr(gls), N, nat.ptr(hf_c),
                                                nat.ptr(pair_c), nat.ptr(tt_c), P, nat.ptr(out), nat.ptr(ws),
                                                nat.ptr(ghf), nat.stream_of(dev)), "mgv_vae_func_loss_bwd")
        return gmu, gls, None, ghf, None, None


def vae_func_loss(mu=None, logstd=None, eps=None, hf=None, tt_pair_index=None, tt_sim=None):
    """Fused reparameterisation + KL + truth-table-similarity loss (one launch).  Either half may be
    omitted.  Returns (z_s, z_t, kl, func_loss); absent halves come back as None."""
    if mu is None and tt_pair_index is None:
        raise RuntimeError("mgv_b200: vae_func_loss needs the VAE inputs, the func-loss inputs, or both")
    z, kl, func = VaeFuncLossFunction.apply(mu, logstd, eps, hf, tt_pair_index, tt_sim)
    if mu is None:
        return None, None, None, func
    return z[0], z[1], kl, (func if tt_pair_index is not None else None)


# =========================================================================== fused readout head (probability MLP + clamp + L1 loss)
_READOUT_CALLS = [0]


class ReadoutFunction(torch.autograd.Function):
    """pred = clamp(MLP(x), 0, 1) and, with a target, loss = mean |pred - target| -- one launch forward, one backward
    (csrc/readout.cu; reference arch/mlp.py:14-56, dg_ae_model_mig.py:150-152, trainer.py:154-156).
    ``bufs`` = (bn1.running_mean, bn1.running_var, bn2.running_mean, bn2.running_var), updated in place in training mode;
    ``params`` = (fc0.w, fc0.b, bn1.w, bn1.b, fc4.w, fc4.b, bn2.w, bn2.b, fc8.w, fc8.b)."""

    @staticmethod
    def forward(ctx, x, target, training, p_drop, seed, momentum, eps, want_mask, bufs, *params):
        nat.require_cuda(x, "hf")
        dev = x.device
        x_c = _f32(x, "hf")
        N = x_c.shape[0]
        t_c = None if target is None else _f32(target.reshape(-1), "prob")
        if t_c is not None and t_c.numel() != N:
            raise RuntimeError("mgv_b200: the readout target must have one entry per node")
        ps = [_f32(p, "readout parameter") for p in params]
        table = [ps[0], ps[1], ps[2], ps[3], bufs[0], bufs[1], ps[4], ps[5], ps[6], ps[7], bufs[2], bufs[3], ps[8], ps[9]]
        f32 = dict(dtype=torch.float32, device=dev)
        pred = torch.empty(N, 1, **f32)
        loss = torch.empty((), **f32)
        saved = torch.empty(max(N, 1), 64, **f32)
        stats = torch.empty(128, **f32)
        mask = torch.empty(max(N, 1), 2, dtype=torch.int32, device=dev) if want_mask else None
        sync = torch.empty(1, dtype=torch.int32, device=dev)
        lib = nat.lib()
        with nat.on_device(dev), _timed("readout_fwd", dev):
            nb = lib.mgv_readout_workspace_bytes(N)
            ws = nat.workspace(nb, dev)
            nat.check(lib.mgv_readout_fwd(nat.ptr(x_c), N, _ptr_table(table), int(bool(training)), float(p_drop), int(seed),
                                          float(momentum), float(eps), nat.ptr(t_c), nat.ptr(pred), nat.ptr(loss), nat.ptr(saved),
                                          nat.ptr(stats), nat.ptr(mask), nat.ptr(ws), nb, nat.ptr(sync), nat.stream_of(dev)),
                      "mgv_readout_fwd")
        ctx.save_for_backward(x_c, t_c, saved, stats, *table)
        ctx.cfg = (int(bool(training)), float(p_drop), int(seed))
        ctx.mark_non_differentiable(*[t for t in (mask,) if t is not None])
        if t_c is None:
            loss = loss.zero_()
        return (pred, loss, mask) if want_mask else (pred, loss)

    @staticmethod
    def backward(ctx, g_pred, g_loss, *unused):
        x_c, t_c, saved, stats = ctx.saved_tensors[:4]
        table = list(ctx.saved_tensors[4:])
        training, p_drop, seed = ctx.cfg
        dev = x_c.device
        N = x_c.shape[0]
        gp = None if g_pred is None else _f32(g_pred.reshape(-1), "g_pred")
        gl = None if (g_loss is None or t_c is None) else _f32(g_loss.reshape(1), "g_loss")
        gx = torch.empty(max(N, 1), 64, dtype=torch.float32, device=dev)
        grads = torch.empty(3297, dtype=torch.float32, device=dev)
        sync = torch.empty(1, dtype=torch.int32, device=dev)
        lib = nat.lib()
        with nat.on_device(dev), _timed("readout_bwd", dev):
            nb = lib.mgv_readout_workspace_bytes(N)
            ws = nat.workspace(nb, dev)
            nat.check(lib.mgv_readout_bwd(nat.ptr(x_c), N, _ptr_table(table), training, p_drop, seed, nat.ptr(t_c), nat.ptr(saved),
                                          nat.ptr(stats), nat.ptr(gp), nat.ptr(gl), nat.ptr(gx), nat.ptr(grads), nat.ptr(ws), nb,
                                          nat.ptr(sync), nat.stream_of(dev)), "mgv_readout_bwd")
        g = grads
        out = (g[0:2048].view(32, 64), g[2048:2080], g[2080:2112], g[2112:2144], g[2144:3168].view(32, 32), g[3168:3200],
               g[3200:3232], g[3232:3264], g[3264:3296].view(1, 32), g[3296:3297])
        return (gx[:N], None, None, None, None, None, None, None, None) + out          # disjoint views of one fresh buffer


def readout_head(x, target, mlp, want_mask=False):
    """``mlp``: arch.mlp.MLP in its readout configuration (Linear-BatchNorm-ReLU-Dropout x 2 + Linear, 64 -> 32 -> 32 -> 1)."""
    fc = mlp.fc
    bn1, bn2 = fc[1], fc[5]
    training = mlp.training
    seed = 0
    if training:
        _READOUT_CALLS[0] += 1
        seed = (torch.initial_seed() * 0x9E3779B1 + _READOUT_CALLS[0]) & 0x7FFFFFFFFFFFFFFF
        with torch.no_grad():
            bn1.num_batches_tracked += 1
            bn2.num_batches_tracked += 1
    momentum = bn1.momentum if bn1.momentum is not None else 0.1
    return ReadoutFunction.apply(x, target, training, fc[3].p if training else 0.0, seed, momentum, bn1.eps, want_mask,
                                 (bn1.running_mean, bn1.running_var, bn2.running_mean, bn2.running_var),
                                 fc[0].weight, fc[0].bias, bn1.weight, bn1.bias, fc[4].weight, fc[4].bias, bn2.weight, bn2.bias,
                                 fc[8].weight, fc[8].bias)
