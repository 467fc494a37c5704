"""ctypes binding of libmgv_b200.so (the C ABI declared in include/mgv_b200.h).

The library is the only compute backend of this package: there is no CPU, PyG or
Triton fallback.  If the shared library has not been built, or a tensor lives on
the wrong device, the calls below raise instead of degrading.
"""
import ctypes
import os

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
# MGV_B200_LIB: development knob -- load another build of the same library (e.g. the phase-trace build of scripts/)
LIB_PATH = os.environ.get("MGV_B200_LIB") or os.path.join(_HERE, "_lib", "libmgv_b200.so")

D = 64
NCODE = 8
CODE_SHIFT = 28
MAX_FEAT = 8
TILE_ROWS = 128
PRECISION_FP32, PRECISION_BF16 = 0, 1
SWEEP_PACK_FLOATS = 66112
SWEEP_GRAD_FLOATS = 33344
STRUCT_PACK_FLOATS = 28416
STRUCT_GRAD_FLOATS = 28416

_vp = ctypes.c_void_p
_i32 = ctypes.c_int32
_i64 = ctypes.c_int64
_u32 = ctypes.c_uint32
_sz = ctypes.c_size_t


class mgv_schedule(ctypes.Structure):
    _fields_ = [("N", _i32), ("L", _i32), ("E", _i64),
                ("order", _vp), ("seg_ptr", _vp), ("in_ptr", _vp), ("in_src", _vp),
                ("out_ptr", _vp), ("out_pack", _vp), ("out_slot", _vp),
                ("code_count", _i64 * NCODE),
                ("deg_order_in", _vp), ("deg_order_out", _vp), ("tile_cost_in", _vp), ("tile_cost_out", _vp),
                ("gdesc_in", _vp), ("gdesc_out", _vp), ("streams", _i32), ("reserved0", _i32),
                ("sweep_desc", _vp)]


_SP = ctypes.POINTER(mgv_schedule)
_PROTOTYPES = {
    "mgv_last_error_string": (ctypes.c_char_p, []),
    "mgv_version": (ctypes.c_int, []),
    "mgv_sm_count": (ctypes.c_int, []),
    "mgv_kernel_launches": (ctypes.c_longlong, []),
    "mgv_csr_workspace_bytes": (_sz, [_i64, _i64]),
    "mgv_build_csr": (ctypes.c_int, [_vp, _i64, _i32, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _sz, _vp, _vp]),
    "mgv_levelize_workspace_bytes": (_sz, [_i64]),
    "mgv_levelize": (ctypes.c_int, [_vp, _vp, _vp, _i32, _vp, ctypes.POINTER(_i32), _vp, _sz, _vp]),
    "mgv_level_lists_workspace_bytes": (_sz, [_i64, _i32]),
    "mgv_build_level_lists": (ctypes.c_int, [_vp, _vp, _vp, _i32, _i32, _i32, _vp, _vp, ctypes.POINTER(_i64), _vp, _sz, _vp, _vp]),
    "mgv_build_sweep_desc": (ctypes.c_int, [_vp, _vp, _vp, _vp, _i32, _vp, _vp]),
    "mgv_degree_order_workspace_bytes": (_sz, [_i64]),
    "mgv_build_degree_order": (ctypes.c_int, [_vp, _vp, _i32, _vp, _vp, _vp, _vp, _sz, _vp]),
    "mgv_build_degree_tiles": (ctypes.c_int, [_vp, _vp, _vp, _i32, _vp, _vp, _vp, _sz, _vp]),
    "mgv_level_sweep_fwd": (ctypes.c_int, [_SP, _i32, _u32, _vp, _vp, _vp, _vp, _i32, _vp]),
    "mgv_sweep_bwd_grid": (ctypes.c_int, []),
    "mgv_sweep_bwd_workspace_bytes": (_sz, [_i64, _i64]),
    "mgv_level_sweep_bwd": (ctypes.c_int, [_SP, _i32, _u32, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _sz, _vp, _i32, _vp]),
    "mgv_struct_fwd_workspace_bytes": (_sz, [_i64, _i32]),
    "mgv_struct_tiles_bytes": (_sz, [_i64, _i32, _i32]),
    "mgv_struct_encoder_fwd": (ctypes.c_int, [_SP, _i32, _i32, _i32, _i32, _vp, _vp, _vp, _vp, _vp, _sz, _i32, _vp]),
    "mgv_struct_bwd_workspace_bytes": (_sz, [_i64, _i32]),
    "mgv_struct_encoder_bwd": (ctypes.c_int, [_SP, _i32, _i32, _i32, _i32, _vp, _vp, _vp, _vp, _vp, _vp, _sz, _i32, _vp]),
    "mgv_vae_func_workspace_bytes": (_sz, [_i64]),
    "mgv_vae_func_loss_fwd": (ctypes.c_int, [_vp, _vp, _vp, _vp, _i64, _vp, _vp, _vp, _i64, _vp, _vp, _sz, _vp]),
    "mgv_vae_func_loss_bwd": (ctypes.c_int, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _i64, _vp, _vp, _vp, _i64,
                                             _vp, _vp, _vp, _vp]),
    "mgv_struct_pack": (ctypes.c_int, [_vp, _i32, _i32, _i32, _vp, _vp]),
    "mgv_struct_unpack_grads": (ctypes.c_int, [_vp, _i32, _i32, _i32, _vp, _vp, _vp]),
    "mgv_sweep_pack_bytes": (_sz, []),
    "mgv_sweep_pack": (ctypes.c_int, [_vp, _vp, _i32, _vp, _i32, _vp]),
    "mgv_sweep_unpack_grads": (ctypes.c_int, [_vp, _vp, _i32, _vp, _vp, _vp]),
    "mgv_negative_sample": (ctypes.c_int, [_vp, _vp, _i32, _i64, ctypes.c_uint64, _vp, _vp]),
    "mgv_permute_edges": (ctypes.c_int, [_vp, _i64, ctypes.c_uint64, _vp, _vp]),
    "mgv_recon_loss_fwd": (ctypes.c_int, [_vp, _i32, _vp, _i64, _vp, _i64, _vp, _vp, _vp, _vp, _sz, _vp, _vp]),
    "mgv_recon_loss_bwd": (ctypes.c_int, [_vp, _i32, _vp, _i64, _vp, _i64, _vp, _vp, _vp, _vp]),
    "mgv_readout_workspace_bytes": (_sz, [_i64]),
    "mgv_readout_fwd": (ctypes.c_int, [_vp, _i64, _vp, _i32, ctypes.c_float, ctypes.c_uint64, ctypes.c_float, ctypes.c_float,
                                       _vp, _vp, _vp, _vp, _vp, _vp, _vp, _sz, _vp, _vp]),
    "mgv_readout_bwd": (ctypes.c_int, [_vp, _i64, _vp, _i32, ctypes.c_float, ctypes.c_uint64, _vp, _vp, _vp, _vp, _vp,
                                       _vp, _vp, _vp, _sz, _vp, _vp]),
    "mgv_linear_wgrad_workspace_bytes": (_sz, [_i64, _i32, _i32]),
    "mgv_linear_wgrad": (ctypes.c_int, [_vp, _vp, _i64, _i32, _i32, _vp, _vp, _vp, _sz, _vp]),
    "mgv_linear_tc": (ctypes.c_int, [_vp, _i64, _vp, _vp, _i32, _i32, _i32, _vp, _vp]),
    "mgv_tc_selftest": (ctypes.c_int, [_i32, _vp, _vp, _vp, _i32, _i32, _vp]),
    "mgv_logic_sim_bytes": (_sz, [_i64, _i32]),
    "mgv_logic_sim_validate": (ctypes.c_int, [_SP, _vp, _vp, ctypes.POINTER(_i32), _vp, _i64, _vp, _sz, _vp]),
    "mgv_logic_sim_pass": (ctypes.c_int, [_SP, _vp, _vp, ctypes.POINTER(_i32), _i32, ctypes.c_uint64, _i64, _i32,
                                          _vp, _vp, _vp, _i64, _vp, _vp]),
}
EXPORTED_SYMBOLS = tuple(_PROTOTYPES)

_lib = None


def lib():
    """The loaded library; raises (never falls back) when it has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                "mgv_b200: %s is missing -- build it with multi-gate-vae_b200/csrc/build.sh "
                "(or __graft_entry__.build()); this package has no CPU/PyTorch fallback" % LIB_PATH)
        handle = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in _PROTOTYPES.items():
            fn = getattr(handle, name)
            fn.restype, fn.argtypes = res, args
        _lib = handle
    return _lib


def check(rc, what):
    if rc != 0:
        msg = lib().mgv_last_error_string()
        raise RuntimeError("mgv_b200 %s failed (%d): %s" % (what, rc, msg.decode() if msg else "?"))


def require_cuda(t, name, dtype=None):
    if not torch.is_tensor(t) or not t.is_cuda:
        raise RuntimeError("mgv_b200: %s must be a CUDA tensor (this package has no CPU path)" % name)
    if dtype is not None and t.dtype != dtype:
        raise RuntimeError("mgv_b200: %s must be %s, got %s" % (name, dtype, t.dtype))
    if not t.is_contiguous():
        raise RuntimeError("mgv_b200: %s must be contiguous" % name)
    return t


def ptr(t):
    return _vp(t.data_ptr()) if t is not None else _vp(0)


_raw_stream = getattr(torch._C, "_cuda_getCurrentRawStream", None)


def stream_of(device):
    """cudaStream_t of torch's current stream on ``device`` (the raw handle: no Stream object per call)."""
    if _raw_stream is not None:
        idx = device.index if isinstance(device, torch.device) else None
        if idx is not None:
            return _vp(_raw_stream(idx))
    return _vp(torch.cuda.current_stream(device).cuda_stream)


class _NoCtx(object):
    def __enter__(self):
        return self

    def __exit__(self, *exc):
        return False


_NOCTX = _NoCtx()


def on_device(device):
    """``torch.cuda.device(device)`` -- skipped when ``device`` already is the current device (the common case: one
    process per GPU), which saves two context switches per library call."""
    try:
        if device.index is not None and torch.cuda.current_device() == device.index:
            return _NOCTX
    except Exception:
        pass
    return torch.cuda.device(device)


def workspace(nbytes, device, zero=False):
    n = max(int(nbytes), 256)
    return (torch.zeros if zero else torch.empty)(n, dtype=torch.uint8, device=device)
