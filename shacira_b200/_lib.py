"""ctypes binding of the C-ABI library (include/shacira_b200.h) + thin torch-tensor wrappers.

PyTorch is plumbing here: it owns device memory and the current stream; every compute call
goes through `libshacira_b200.so`. There is NO fallback: if the library is missing or a call
fails, a RuntimeError is raised.
"""
import ctypes
import os
import threading

import torch

_PKG = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("SHACIRA_LIB") or os.path.join(_PKG, "libshacira_b200.so")  # env: kernel-tuning builds

OK = 0
ERR_INVALID_ARGUMENT = -1
ERR_UNSUPPORTED = -2
ERR_CUDA = -3
ERR_Q2_WINDOW = -4
ERR_NO_DEVICE = -5
MAX_LEVELS = 32

_c_int32_p = ctypes.POINTER(ctypes.c_int32)
_vp = ctypes.c_void_p
_i32 = ctypes.c_int32
_i64 = ctypes.c_int64

class AdamSeg(ctypes.Structure):
    """shacira_adam_seg_t (include/shacira_b200.h)."""
    _fields_ = [("param", _vp), ("grad", _vp), ("exp_avg", _vp), ("exp_avg_sq", _vp), ("grad_scale", _vp),
                ("grad_div", _vp), ("n", _i32), ("grad_rows", _i32), ("grad_row_stride", _i32), ("div_group", _i32),
                ("lr", ctypes.c_float), ("weight_decay", ctypes.c_float), ("grad_mul", ctypes.c_float),
                ("zero_grad", ctypes.c_float)]


MAX_ADAM_SEGS = 32


class FitSnapshot(ctypes.Structure):
    """shacira_fit_snapshot_t (include/shacira_b200.h)."""
    _fields_ = [("sse", _vp), ("count", _i64), ("best_loss", _vp), ("best_step", _vp), ("table", _vp),
                ("seg_param", _vp * MAX_ADAM_SEGS), ("div", _vp), ("A", _vp)]


LAMBDA_FIX = 0
LAMBDA_COSINE = 1


class FitSchedule(ctypes.Structure):
    """shacira_fit_schedule_t (include/shacira_b200.h)."""
    _fields_ = [("num_epochs", _i32), ("lambda_kind", _i32), ("lambda_start", ctypes.c_double),
                ("lambda_end", ctypes.c_double), ("temperature_end", ctypes.c_double), ("decay_period", ctypes.c_double),
                ("sse", _vp), ("count", _i64), ("log", _vp), ("log_capacity", _i64)]

# name -> (restype, argtypes); mirrors include/shacira_b200.h one to one.
SIGNATURES = {
    "shacira_abi_version": (ctypes.c_int, []),
    "shacira_last_error": (ctypes.c_char_p, []),
    "shacira_launch_count": (_i64, []),
    "shacira_device_info": (ctypes.c_int, [_c_int32_p, ctypes.POINTER(_i64), ctypes.POINTER(_i64)]),
    "shacira_l2_pin": (ctypes.c_int, [_vp, _i64, _vp]),
    "shacira_hashgrid_forward": (ctypes.c_int, [_i32, _vp, _i64, _vp, _c_int32_p, _c_int32_p, _i32, _i32, _i32, _vp, _vp]),
    "shacira_hashgrid_backward": (ctypes.c_int, [_i32, _vp, _i64, _vp, _c_int32_p, _c_int32_p, _i32, _i32, _i32, _i64, _i32, _vp, _vp]),
    "shacira_hashgrid_corners": (ctypes.c_int, [_i32, _vp, _i64, _c_int32_p, _i32, _i32, _vp, _vp, _vp]),
    "shacira_latent_forward": (ctypes.c_int, [_i32, _vp, _i64, _vp, _c_int32_p, _c_int32_p, _i32, _i32, _i32, _i32, _i32, _vp, _vp, _i32, _vp, _vp, _vp]),
    "shacira_latent_backward": (ctypes.c_int, [_i32, _vp, _i64, _vp, _vp, _c_int32_p, _c_int32_p, _i32, _i32, _i32, _i32, _vp, _i32, _i64, _i32, _vp, _vp, _vp, _vp]),
    "shacira_latent_backward_levels": (ctypes.c_int, [_i32, _vp, _i64, _vp, _vp, _c_int32_p, _c_int32_p, _i32, _i32, _i32, _i32, _vp, _i32, _i64, _i32, ctypes.c_uint32, _vp, _vp, _vp, _vp]),
    "shacira_plan_create": (ctypes.c_int, [_i32, _vp, _i64, _i32, _vp, ctypes.POINTER(_vp)]),
    "shacira_plan_rebuild": (ctypes.c_int, [_vp, _i32, _vp, _i64, _i32, _vp]),
    "shacira_plan_destroy": (ctypes.c_int, [_vp]),
    "shacira_plan_info": (ctypes.c_int, [_vp, ctypes.POINTER(_i64), _c_int32_p, _c_int32_p, _c_int32_p]),
    "shacira_plan_debug": (ctypes.c_int, [_vp, ctypes.POINTER(_vp), ctypes.POINTER(_vp), ctypes.POINTER(_vp)]),
    "shacira_plan_set_sorted_io": (ctypes.c_int, [_vp, _i32]),
    "shacira_latent_forward_planned": (ctypes.c_int, [_vp, _vp, _c_int32_p, _c_int32_p, _i32, _i32, _i32, _i32, _i32, _vp, _vp, _i32, _vp, _vp]),
    "shacira_latent_backward_planned": (ctypes.c_int, [_vp, _vp, _vp, _c_int32_p, _c_int32_p, _i32, _i32, _i32, _i32, _i32, _vp, _i32, _i64, _i32, _vp, _vp, _vp, _vp]),
    "shacira_latent_backward_planned_bounded": (ctypes.c_int, [_vp, _vp, _vp, _c_int32_p, _c_int32_p, _i32, _i32, _i32, _i32, _i32, _vp, _i32, _i64, _i32, _vp, _vp, _vp, _vp, _vp]),
    "shacira_latent_forward_planned_z": (ctypes.c_int, [_vp, _vp, _c_int32_p, _c_int32_p, _i32, _i32, _i32, _i32, _i32, _vp, _vp, _i32, _vp, _vp, _vp]),
    "shacira_latent_backward_planned_z": (ctypes.c_int, [_vp, _vp, _vp, _c_int32_p, _c_int32_p, _i32, _i32, _i32, _i32, _vp, _i32, _i64, _i32, _vp, _vp, _vp, _vp]),
    "shacira_entropy_bits": (ctypes.c_int, [_vp, _vp, _i64, _i32, _vp, _i32, _c_int32_p, _i32, _vp, _vp, _vp, _vp, _i64, _vp]),
    "shacira_entropy_bits_rng": (ctypes.c_int, [_vp, ctypes.c_uint64, _vp, _i64, _i32, _vp, _i32, _c_int32_p, _i32, _vp, _vp, _vp, _vp, _i64, _vp]),
    "shacira_entropy_scratch_bytes": (_i64, [_i32, _i32]),
    "shacira_quantize_symbols": (ctypes.c_int, [_vp, _i64, _i32, _vp, _vp, _vp]),
    "shacira_symbol_histogram": (ctypes.c_int, [_vp, _i64, _i32, _c_int32_p, _i32, _vp, _vp]),
    "shacira_mlp_mse_step": (ctypes.c_int, [_vp, _vp, _i64, _i32, _i32, _i32, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "shacira_mlp_mse_step_bounded": (ctypes.c_int, [_vp, _vp, _i64, _i32, _i32, _i32, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "shacira_fit_tile_step": (ctypes.c_int, [_vp, _vp, _c_int32_p, _c_int32_p, _i32, _i32, _i32, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i64, _vp, _vp, _vp, _vp, _vp]),
    "shacira_fit_render": (ctypes.c_int, [_vp, _vp, _c_int32_p, _c_int32_p, _i32, _i32, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "shacira_peer_flags_offset": (_i64, [_i64]),
    "shacira_peer_alloc": (ctypes.c_int, [_i64, ctypes.POINTER(_vp)]),
    "shacira_peer_free": (ctypes.c_int, [_vp]),
    "shacira_peer_export": (ctypes.c_int, [_vp, _vp]),
    "shacira_peer_open": (ctypes.c_int, [_vp, ctypes.POINTER(_vp)]),
    "shacira_peer_close": (ctypes.c_int, [_vp]),
    "shacira_peer_enable_access": (ctypes.c_int, [_i32, _i32]),
    "shacira_peer_allreduce": (ctypes.c_int, [ctypes.POINTER(_vp), _i64, _i32, _i32, _i64, _vp]),
    "shacira_peer_status": (ctypes.c_int, [_vp, _i64, ctypes.POINTER(_i32)]),
    "shacira_peer_allreduce_multimem": (ctypes.c_int, [_vp, ctypes.POINTER(_vp), _i64, _i32, _i32, _i64, _vp]),
    "shacira_peer_allreduce_adam": (ctypes.c_int, [ctypes.POINTER(_vp), _i64, _i32, _i32, _i64, ctypes.POINTER(_vp), _i64, _vp, _vp, _vp, ctypes.c_float, ctypes.c_float, ctypes.c_float, ctypes.c_float, ctypes.c_float, _vp]),
    "shacira_fit_optimizer_step": (ctypes.c_int, [_vp, _i32, _vp, _vp, _vp, _vp, _vp, ctypes.c_float, _vp, _vp, _i64, ctypes.c_float, ctypes.c_float, ctypes.c_float, ctypes.c_float, ctypes.c_float, _vp, _vp, _vp, _vp, _vp, _i32, _i32, _vp, _i32, ctypes.c_uint64, _vp, _vp, _vp, _vp, _i32, _vp, ctypes.c_uint64, _vp, _vp, _vp, _vp, _i64, _vp, _vp]),
    "shacira_fit_optimizer_step_best": (ctypes.c_int, [_vp, _i32, _vp, _vp, _vp, _vp, _vp, ctypes.c_float, _vp, _vp, _i64, ctypes.c_float, ctypes.c_float, ctypes.c_float, ctypes.c_float, ctypes.c_float, _vp, _vp, _vp, _vp, _vp, _i32, _i32, _vp, _i32, ctypes.c_uint64, _vp, _vp, _vp, _vp, _i32, _vp, ctypes.c_uint64, _vp, _vp, _vp, _vp, _i64, _vp, _vp, _vp]),
    "shacira_fit_optimizer_step_sched": (ctypes.c_int, [_vp, _i32, _vp, _vp, _vp, _vp, _vp, ctypes.c_float, _vp, _vp, _i64, ctypes.c_float, ctypes.c_float, ctypes.c_float, ctypes.c_float, ctypes.c_float, _vp, _vp, _vp, _vp, _vp, _i32, _i32, _vp, _i32, ctypes.c_uint64, _vp, _vp, _vp, _vp, _i32, _vp, ctypes.c_uint64, _vp, _vp, _vp, _vp, _i64, _vp, _vp, _vp, _vp]),
    "shacira_adam_step": (ctypes.c_int, [_vp, _vp, _vp, _vp, _i64, ctypes.c_float, ctypes.c_float, ctypes.c_float, ctypes.c_float, ctypes.c_float, _vp, _i32, _vp]),
    "shacira_adam_step_sum": (ctypes.c_int, [_vp, _vp, _vp, _vp, ctypes.c_float, _vp, _vp, _i64, ctypes.c_float, ctypes.c_float, ctypes.c_float, ctypes.c_float, ctypes.c_float, _vp, _i32, _i32, _vp]),
    "shacira_adam_step_sum_mul": (ctypes.c_int, [_vp, _vp, _vp, _vp, _vp, ctypes.c_float, _vp, _vp, _i64, ctypes.c_float, ctypes.c_float, ctypes.c_float, ctypes.c_float, ctypes.c_float, _vp, _i32, _i32, _vp]),
    "shacira_sga_quantize": (ctypes.c_int, [_vp, _vp, _i64, _vp, _i32, ctypes.c_uint64, _vp, _vp, _vp, _vp]),
    "shacira_multi_adam_step": (ctypes.c_int, [_vp, _i32, ctypes.c_float, ctypes.c_float, ctypes.c_float, _vp, _vp, _vp, _vp, _vp, _i32, _i32, _vp, _vp]),
    "shacira_integrate_forward": (ctypes.c_int, [_vp, _vp, _vp, _i32, _i32, _vp, _vp, _vp, _vp]),
    "shacira_integrate_backward": (ctypes.c_int, [_vp, _vp, _vp, _vp, _i32, _i32, _vp, _vp, _vp, _vp, _vp]),
    "shacira_voxel_samples": (ctypes.c_int, [_vp, _vp, _vp, _vp, _vp, _i64, _i32, _vp, _vp, _vp, _vp, _vp, _vp]),
    "shacira_raytrace_dense_count": (ctypes.c_int, [_vp, _i32, _vp, _vp, _i32, _vp, _vp]),
    "shacira_raytrace_dense_fill": (ctypes.c_int, [_vp, _i32, _vp, _vp, _i32, _vp, _vp, _vp, _vp, _vp]),
    "shacira_prune_samples": (ctypes.c_int, [_i32, _vp, _vp, _vp]),
    "shacira_prune_update": (ctypes.c_int, [_i64, _vp, ctypes.c_float, ctypes.c_float, _vp, _vp, _vp]),
    "shacira_nerf_heads_forward": (ctypes.c_int, [_vp, _i64, _i32, _i32, _vp, _i32, _i32, _vp, ctypes.POINTER(_vp), _i32, _vp, _vp, _vp]),
    "shacira_nerf_heads_workspace_bytes": (_i64, [_i32]),
    "shacira_nerf_heads_backward": (ctypes.c_int, [_vp, _i64, _i32, _i32, _vp, _i32, _i32, _vp, ctypes.POINTER(_vp), _vp, _vp, _vp, ctypes.POINTER(_vp), _vp, _i64, _vp]),
    "shacira_ac_encode": (_i64, [_vp, _i64, _vp, _i32, _vp, _i64]),
    "shacira_ac_decode": (ctypes.c_int, [_vp, _i64, _vp, _i32, _vp, _i64]),
    "shacira_latent_step_host": (ctypes.c_int, [_i32, _vp, _i64, _vp, _i64, _c_int32_p, _c_int32_p, _i32, _i32, _i32, _i32, _i32, _vp, _vp, _i32, _vp, _vp, _vp]),
    "shacira_host_session_create": (ctypes.c_int, [_i32, _i64, _i64, _c_int32_p, _c_int32_p, _i32, _i32, _i32, _i32, _i32, ctypes.POINTER(_vp)]),
    "shacira_host_session_destroy": (ctypes.c_int, [_vp]),
    "shacira_host_session_set_coords": (ctypes.c_int, [_vp, _vp]),
    "shacira_host_session_set_table": (ctypes.c_int, [_vp, _vp, _vp, _vp, _i32]),
    "shacira_host_session_step_async": (ctypes.c_int, [_vp, _vp, _vp, _vp, _vp, _vp, _c_int32_p]),
    "shacira_host_session_wait": (ctypes.c_int, [_vp, _i32]),
}

_lib = None
_lock = threading.Lock()


class ShaciraError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__("shacira_b200 [%d]: %s" % (code, msg))
        self.code = code


def load():
    """Load the C-ABI library. Raises (never falls back) when it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    with _lock:
        if _lib is not None:
            return _lib
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                "shacira_b200: %s is missing -- build it with `python -m shacira_b200.build` "
                "(or __graft_entry__.build()). There is no CPU / PyTorch fallback." % LIB_PATH)
        lib = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(lib, name)  # AttributeError if the ABI drifted
            fn.restype = res
            fn.argtypes = args
        _lib = lib
    return _lib


def _check(rc):
    if rc != 0:
        raise ShaciraError(rc, load().shacira_last_error().decode("utf-8", "replace"))


_arr_cache = {}


def _i32_array(values):
    key = tuple(int(v) for v in values)
    arr = _arr_cache.get(key)
    if arr is None:
        arr = (ctypes.c_int32 * len(key))(*key)
        if len(_arr_cache) > 4096:
            _arr_cache.clear()
        _arr_cache[key] = arr
    return arr, len(key)


def _stream():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def _f32c(t, name):
    if not t.is_cuda:
        raise ShaciraError(ERR_INVALID_ARGUMENT, "%s must be a CUDA tensor (no CPU fallback)" % name)
    if t.dtype != torch.float32:
        raise ShaciraError(ERR_UNSUPPORTED, "%s must be float32 (fp32 is the supported path), got %s" % (name, t.dtype))
    return t if t.is_contiguous() else t.contiguous()


def _ptr(t):
    return ctypes.c_void_p(t.data_ptr()) if t is not None else ctypes.c_void_p(0)


def launch_count():
    return int(load().shacira_launch_count())


def device_info():
    sm, l2, pers = ctypes.c_int32(0), ctypes.c_int64(0), ctypes.c_int64(0)
    _check(load().shacira_device_info(ctypes.byref(sm), ctypes.byref(l2), ctypes.byref(pers)))
    return {"sm_count": sm.value, "l2_bytes": l2.value, "l2_persist_max": pers.value}


def l2_pin(tensor):
    """Pin `tensor` in L2 for kernels launched on the current stream (None clears the window)."""
    if tensor is None:
        _check(load().shacira_l2_pin(None, 0, _stream()))
    else:
        _check(load().shacira_l2_pin(_ptr(tensor), tensor.numel() * tensor.element_size(), _stream()))


def _dim_of(coords):
    if coords.dim() != 2 or coords.shape[1] not in (2, 3):
        raise ShaciraError(ERR_INVALID_ARGUMENT, "coords must be [N, 2] or [N, 3], got %s" % (tuple(coords.shape),))
    return coords.shape[1]


def _check_table_rows(rows, first_idx, resolutions, bitwidth, dim, what):
    """The forward ABI carries no table size: make sure here that every level ends inside the table."""
    need = max(int(f) + min(1 << int(bitwidth), int(r) ** dim) for f, r in zip(first_idx, resolutions))
    if rows < need:
        raise ShaciraError(ERR_INVALID_ARGUMENT, "%s has %d rows, the levels need %d" % (what, rows, need))


def hashgrid_forward(coords, codebook, first_idx, resolutions, bitwidth):
    """feats[N, L*F]; first_idx / resolutions are host int sequences."""
    lib = load()
    coords = _f32c(coords, "coords")
    codebook = _f32c(codebook, "codebook")
    dim = _dim_of(coords)
    fi, L = _i32_array(first_idx)
    rs, L2 = _i32_array(resolutions)
    if L != L2:
        raise ShaciraError(ERR_INVALID_ARGUMENT, "first_idx and resolutions differ in length")
    _check_table_rows(codebook.shape[0], first_idx, resolutions, bitwidth, dim, "codebook")
    n, F = coords.shape[0], codebook.shape[1]
    feats = torch.empty((n, L * F), dtype=torch.float32, device=coords.device)
    with torch.cuda.device(coords.device):
        _check(lib.shacira_hashgrid_forward(dim, _ptr(coords), n, _ptr(codebook), fi, rs, L, bitwidth, F,
                                            _ptr(feats), _stream()))
    return feats


def hashgrid_backward(coords, grad_output, first_idx, resolutions, bitwidth, feature_dim, table_rows, out=None):
    lib = load()
    coords = _f32c(coords, "coords")
    grad_output = _f32c(grad_output, "grad_output")
    dim = _dim_of(coords)
    fi, L = _i32_array(first_idx)
    rs, _ = _i32_array(resolutions)
    n = coords.shape[0]
    if tuple(grad_output.shape) != (n, L * feature_dim):
        raise ShaciraError(ERR_INVALID_ARGUMENT, "grad_output must be [N, L*F] = %s, got %s" % ((n, L * feature_dim), tuple(grad_output.shape)))
    zero_first = 1
    if out is None:
        out = torch.empty((table_rows, feature_dim), dtype=torch.float32, device=coords.device)
    else:
        zero_first = 0
    with torch.cuda.device(coords.device):
        _check(lib.shacira_hashgrid_backward(dim, _ptr(coords), n, _ptr(grad_output), fi, rs, L, bitwidth,
                                             feature_dim, table_rows, zero_first, _ptr(out), _stream()))
    return out


def hashgrid_corners(coords, resolutions, bitwidth):
    lib = load()
    coords = _f32c(coords, "coords")
    dim = _dim_of(coords)
    rs, L = _i32_array(resolutions)
    n = coords.shape[0]
    idx = torch.empty((n, L, 1 << dim), dtype=torch.int32, device=coords.device)
    w = torch.empty((n, L, 1 << dim), dtype=torch.float32, device=coords.device)
    with torch.cuda.device(coords.device):
        _check(lib.shacira_hashgrid_corners(dim, _ptr(coords), n, rs, L, bitwidth, _ptr(idx), _ptr(w), _stream()))
    return idx, w


def latent_forward(coords, latents, first_idx, resolutions, bitwidth, A, shift, feature_dim, round_flag, save_z):
    """A: [1|L, C, F]; shift: [1|L, F] or None. Returns (feats[N, L*F], z[N, L*C] or None)."""
    lib = load()
    coords = _f32c(coords, "coords")
    latents = _f32c(latents, "latents")
    A = _f32c(A, "A")
    shift = _f32c(shift, "shift") if shift is not None else None
    dim = _dim_of(coords)
    fi, L = _i32_array(first_idx)
    rs, _ = _i32_array(resolutions)
    n, C = coords.shape[0], latents.shape[1]
    per_level = 1 if A.shape[0] == L and L > 1 else 0
    if A.shape[0] not in (1, L) or tuple(A.shape[1:]) != (C, feature_dim):
        raise ShaciraError(ERR_INVALID_ARGUMENT, "A must be [1|L, C, F], got %s" % (tuple(A.shape),))
    _check_table_rows(latents.shape[0], first_idx, resolutions, bitwidth, dim, "latents")
    feats = torch.empty((n, L * feature_dim), dtype=torch.float32, device=coords.device)
    z = torch.empty((n, L * C), dtype=torch.float32, device=coords.device) if save_z else None
    with torch.cuda.device(coords.device):
        _check(lib.shacira_latent_forward(dim, _ptr(coords), n, _ptr(latents), fi, rs, L, bitwidth, C, feature_dim,
                                          1 if round_flag else 0, _ptr(A), _ptr(shift), per_level, _ptr(feats),
                                          _ptr(z), _stream()))
    return feats, z


def latent_backward(coords, grad_output, z, first_idx, resolutions, bitwidth, A, latent_dim, feature_dim,
                    table_rows, want_decoder_grads, level_chunks=None):
    """Returns (grad_latents[T, C], grad_A[L, C, F] or None, grad_shift[L, F] or None). `level_chunks`: list of level
    bit masks; the backward then runs as one launch per chunk (shacira_latent_backward_levels) into the same buffers."""
    lib = load()
    coords = _f32c(coords, "coords")
    grad_output = _f32c(grad_output, "grad_output")
    A = _f32c(A, "A")
    dim = _dim_of(coords)
    fi, L = _i32_array(first_idx)
    rs, _ = _i32_array(resolutions)
    n = coords.shape[0]
    per_level = 1 if A.shape[0] == L and L > 1 else 0
    dev = coords.device
    if tuple(grad_output.shape) != (n, L * feature_dim):
        raise ShaciraError(ERR_INVALID_ARGUMENT, "grad_output must be [N, L*F] = %s, got %s" % ((n, L * feature_dim), tuple(grad_output.shape)))
    if z is not None and tuple(z.shape) != (n, L * latent_dim):
        raise ShaciraError(ERR_INVALID_ARGUMENT, "z must be [N, L*C], got %s" % (tuple(z.shape),))
    gl = torch.empty((table_rows, latent_dim), dtype=torch.float32, device=dev)
    gA = gS = None
    if want_decoder_grads:
        gA = torch.zeros((L, latent_dim, feature_dim), dtype=torch.float32, device=dev)
        gS = torch.zeros((L, feature_dim), dtype=torch.float32, device=dev)
    with torch.cuda.device(dev):
        for k, mask in enumerate(level_chunks or [0xFFFFFFFF]):
            _check(lib.shacira_latent_backward_levels(dim, _ptr(coords), n, _ptr(grad_output), _ptr(z), fi, rs, L,
                                                      bitwidth, latent_dim, feature_dim, _ptr(A), per_level, table_rows,
                                                      1 if k == 0 else 0, int(mask) & 0xFFFFFFFF, _ptr(gl), _ptr(gA),
                                                      _ptr(gS), _stream()))
    return gl, gA, gS


class Plan:
    """Spatial tile plan of one coordinate set (shacira_plan_create). Holds a reference to the
    coordinates it was built from so that their storage cannot be recycled while the plan lives."""

    def __init__(self, coords, tile_points=0):
        lib = load()
        coords = _f32c(coords, "coords")
        self.dim = _dim_of(coords)
        self.n = coords.shape[0]
        self.device = coords.device
        self.coords = coords
        self.users = 0  # autograd graphs that still need this plan for their backward (see grid_ops.plan_for)
        handle = ctypes.c_void_p(0)
        with torch.cuda.device(coords.device):
            _check(lib.shacira_plan_create(self.dim, _ptr(coords), self.n, int(tile_points), _stream(),
                                           ctypes.byref(handle)))
        self.handle = handle

    def rebuild(self, coords, tile_points=0):
        """Re-bin this plan for another coordinate set, reusing the device allocation (no cudaMalloc)."""
        coords = _f32c(coords, "coords")
        if coords.device != self.device:
            raise ShaciraError(ERR_INVALID_ARGUMENT, "plan and coords live on different devices")
        dim = _dim_of(coords)
        with torch.cuda.device(self.device):
            _check(load().shacira_plan_rebuild(self.handle, dim, _ptr(coords), coords.shape[0], int(tile_points), _stream()))
        self.dim, self.n, self.coords = dim, coords.shape[0], coords
        return self

    def set_sorted_io(self, flag=True):
        """Exchange feats / grad_output rows in the plan's sorted order (see shacira_plan_set_sorted_io)."""
        _check(load().shacira_plan_set_sorted_io(self.handle, 1 if flag else 0))
        self.sorted_io = bool(flag)
        return self

    def perm_tensor(self):
        """perm [n] int64 on the plan's device: original index of the point at each sorted position."""
        import numpy as np
        return torch.from_numpy(self.arrays()[0].astype(np.int64)).to(self.device)

    def info(self):
        n, d, g, t = ctypes.c_int64(0), ctypes.c_int32(0), ctypes.c_int32(0), ctypes.c_int32(0)
        _check(load().shacira_plan_info(self.handle, ctypes.byref(n), ctypes.byref(d), ctypes.byref(g), ctypes.byref(t)))
        return {"n": n.value, "dim": d.value, "tiles_per_axis": g.value, "ntiles": t.value}

    def arrays(self):
        """(perm[n] int32, coords_sorted[n, dim] float32, tile_off[ntiles+1] int32) copied to the host (tests)."""
        import numpy as np
        perm, cs, off = ctypes.c_void_p(0), ctypes.c_void_p(0), ctypes.c_void_p(0)
        _check(load().shacira_plan_debug(self.handle, ctypes.byref(perm), ctypes.byref(cs), ctypes.byref(off)))
        nt = self.info()["ntiles"]
        torch.cuda.synchronize(self.device)

        class _Dev:  # alias raw device memory through the CUDA array interface
            def __init__(self, ptr, count, typestr):
                self.__cuda_array_interface__ = {"shape": (count,), "typestr": typestr, "data": (ptr, False),
                                                 "version": 2}

        def grab(ptr, count, dtype):
            typestr = "<i4" if dtype == torch.int32 else "<f4"
            with torch.cuda.device(self.device):
                return torch.as_tensor(_Dev(ptr.value, count, typestr), device=self.device).clone().cpu().numpy()

        return (grab(perm, self.n, torch.int32), grab(cs, self.n * self.dim, torch.float32).reshape(self.n, self.dim),
                grab(off, nt + 1, torch.int32))

    def close(self):
        if getattr(self, "handle", None) is not None and self.handle.value:
            try:
                load().shacira_plan_destroy(self.handle)
            finally:
                self.handle = ctypes.c_void_p(0)
                self.coords = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def latent_forward_planned(plan, latents, first_idx, resolutions, bitwidth, A, shift, feature_dim, round_flag):
    lib = load()
    latents = _f32c(latents, "latents")
    A = _f32c(A, "A")
    shift = _f32c(shift, "shift") if shift is not None else None
    fi, L = _i32_array(first_idx)
    rs, _ = _i32_array(resolutions)
    C = latents.shape[1]
    per_level = 1 if A.shape[0] == L and L > 1 else 0
    if A.shape[0] not in (1, L) or tuple(A.shape[1:]) != (C, feature_dim):
        raise ShaciraError(ERR_INVALID_ARGUMENT, "A must be [1|L, C, F], got %s" % (tuple(A.shape),))
    feats = torch.empty((plan.n, L * feature_dim), dtype=torch.float32, device=plan.device)
    with torch.cuda.device(plan.device):
        _check(lib.shacira_latent_forward_planned(plan.handle, _ptr(latents), fi, rs, L, bitwidth, C, feature_dim,
                                                  1 if round_flag else 0, _ptr(A), _ptr(shift), per_level,
                                                  _ptr(feats), _stream()))
    return feats


def latent_backward_planned(plan, grad_output, latents, first_idx, resolutions, bitwidth, A, latent_dim, feature_dim,
                            table_rows, round_flag, want_decoder_grads, level_max=None):
    """`level_max` [L * F] (optional): upper bounds of |grad_output| per column; skips the kernel's own max pass."""
    lib = load()
    grad_output = _f32c(grad_output, "grad_output")
    A = _f32c(A, "A")
    latents = _f32c(latents, "latents") if latents is not None else None
    fi, L = _i32_array(first_idx)
    rs, _ = _i32_array(resolutions)
    per_level = 1 if A.shape[0] == L and L > 1 else 0
    dev = plan.device
    gl = torch.empty((table_rows, latent_dim), dtype=torch.float32, device=dev)
    gA = gS = None
    if want_decoder_grads:
        gA = torch.zeros((L, latent_dim, feature_dim), dtype=torch.float32, device=dev)
        gS = torch.zeros((L, feature_dim), dtype=torch.float32, device=dev)
    with torch.cuda.device(dev):
        _check(lib.shacira_latent_backward_planned_bounded(
            plan.handle, _ptr(grad_output), _ptr(latents), fi, rs, L, bitwidth, latent_dim, feature_dim,
            1 if round_flag else 0, _ptr(A), per_level, table_rows, 1, _ptr(gl), _ptr(gA), _ptr(gS),
            _ptr(_f32c(level_max, "level_max") if level_max is not None else None), _stream()))
    return gl, gA, gS


def latent_forward_planned_z(plan, latents, first_idx, resolutions, bitwidth, A, shift, feature_dim, round_flag,
                             save_z, feats=None, z=None):
    """3D plans: feats [n, L*F] (original order unless the plan is in sorted-I/O mode) and, with save_z, the
    interpolated latents z [n, L*C] in the plan's sorted order (scratch for latent_backward_planned_z)."""
    lib = load()
    latents = _f32c(latents, "latents")
    A = _f32c(A, "A")
    shift = _f32c(shift, "shift") if shift is not None else None
    fi, L = _i32_array(first_idx)
    rs, _ = _i32_array(resolutions)
    C = latents.shape[1]
    per_level = 1 if A.shape[0] == L and L > 1 else 0
    if A.shape[0] not in (1, L) or tuple(A.shape[1:]) != (C, feature_dim):
        raise ShaciraError(ERR_INVALID_ARGUMENT, "A must be [1|L, C, F], got %s" % (tuple(A.shape),))
    if feats is None:
        feats = torch.empty((plan.n, L * feature_dim), dtype=torch.float32, device=plan.device)
    if save_z and z is None:
        z = torch.empty((plan.n, L * C), dtype=torch.float32, device=plan.device)
    with torch.cuda.device(plan.device):
        _check(lib.shacira_latent_forward_planned_z(plan.handle, _ptr(latents), fi, rs, L, bitwidth, C, feature_dim,
                                                    1 if round_flag else 0, _ptr(A), _ptr(shift), per_level,
                                                    _ptr(feats), _ptr(z if save_z else None), _stream()))
    return feats, (z if save_z else None)


def latent_backward_planned_z(plan, grad_output, z, first_idx, resolutions, bitwidth, A, latent_dim, feature_dim,
                              table_rows, want_decoder_grads, out=None):
    """3D plans: (grad_latents[T, C], grad_A[L, C, F] | None, grad_shift[L, F] | None); `z` from the planned forward.
    `out`: accumulate into an existing (zeroed by the caller) grad_latents buffer instead of allocating one."""
    lib = load()
    grad_output = _f32c(grad_output, "grad_output")
    A = _f32c(A, "A")
    fi, L = _i32_array(first_idx)
    rs, _ = _i32_array(resolutions)
    per_level = 1 if A.shape[0] == L and L > 1 else 0
    dev = plan.device
    if tuple(grad_output.shape) != (plan.n, L * feature_dim):
        raise ShaciraError(ERR_INVALID_ARGUMENT, "grad_output must be [n, L*F], got %s" % (tuple(grad_output.shape),))
    gl = out if out is not None else torch.empty((table_rows, latent_dim), dtype=torch.float32, device=dev)
    gA = gS = None
    if want_decoder_grads:
        gA = torch.zeros((L, latent_dim, feature_dim), dtype=torch.float32, device=dev)
        gS = torch.zeros((L, feature_dim), dtype=torch.float32, device=dev)
    with torch.cuda.device(dev):
        _check(lib.shacira_latent_backward_planned_z(plan.handle, _ptr(grad_output), _ptr(z), fi, rs, L, bitwidth,
                                                     latent_dim, feature_dim, _ptr(A), per_level, table_rows,
                                                     0 if out is not None else 1, _ptr(gl), _ptr(gA), _ptr(gS),
                                                     _stream()))
    return gl, gA, gS


_ent_scratch = {}


def _entropy_scratch(device, C, L):
    """Zero-initialised scratch per (device, stream): reused by every entropy call on that stream."""
    key = (device.index, torch.cuda.current_stream(device).cuda_stream, C, L)
    buf = _ent_scratch.get(key)
    if buf is None:
        nbytes = int(load().shacira_entropy_scratch_bytes(C, L))
        side = torch.cuda.is_current_stream_capturing()
        if side:  # first use inside a graph capture: let the call allocate from the pool instead
            return None
        buf = torch.zeros(nbytes, dtype=torch.uint8, device=device)
        _ent_scratch[key] = buf
    return buf


def entropy_bits(latents, noise, params, num_layers, first_idx=None, want_grads=True, want_latent_grads=True):
    """params [4, 3, C]. Returns (bits[1+L] float64, grad_latents[T, C] | None, grad_params[4,3,C] | None).
    noise None = validation mode (x = rint(w)): the latents' gradient is zero there (want_latent_grads=False skips
    writing it)."""
    lib = load()
    latents = _f32c(latents, "latents")
    noise = _f32c(noise, "noise") if noise is not None else None
    params = _f32c(params, "params")
    T, C = latents.shape
    if first_idx is not None:
        fi, L = _i32_array(first_idx)
    else:
        fi, L = None, 0
    dev = latents.device
    bits = torch.empty((1 + L,), dtype=torch.float64, device=dev)
    gl = torch.empty_like(latents) if (want_grads and want_latent_grads) else None
    gp = torch.empty((4, 3, C), dtype=torch.float32, device=dev) if want_grads else None
    with torch.cuda.device(dev):
        scratch = _entropy_scratch(dev, C, L)
        _check(lib.shacira_entropy_bits(_ptr(latents), _ptr(noise), T, C, _ptr(params), num_layers, fi, L,
                                        _ptr(bits), _ptr(gl), _ptr(gp), _ptr(scratch),
                                        scratch.numel() if scratch is not None else 0, _stream()))
    return bits, gl, gp


def entropy_bits_rng(latents, seed, rng_step, params, num_layers, first_idx=None, scratch=None):
    """Training-mode bit-rate estimate with the noise drawn inside the kernel (shacira_entropy_bits_rng).
    `rng_step`: device int64/uint64 scalar tensor, advanced by the call. Returns (bits[1+L] f64, grad_latents, grad_params)."""
    lib = load()
    latents, params = _f32c(latents, "latents"), _f32c(params, "params")
    T, C = latents.shape
    fi, L = _i32_array(first_idx) if first_idx is not None else (None, 0)
    dev = latents.device
    bits = torch.empty((1 + L,), dtype=torch.float64, device=dev)
    gl = torch.empty_like(latents)
    gp = torch.empty((4, 3, C), dtype=torch.float32, device=dev)
    if scratch is None:
        scratch = torch.zeros(int(lib.shacira_entropy_scratch_bytes(C, L)), dtype=torch.uint8, device=dev)
    with torch.cuda.device(dev):
        _check(lib.shacira_entropy_bits_rng(_ptr(latents), int(seed) & 0xFFFFFFFFFFFFFFFF, _ptr(rng_step), T, C,
                                            _ptr(params), num_layers, fi, L, _ptr(bits), _ptr(gl), _ptr(gp),
                                            _ptr(scratch), scratch.numel(), _stream()))
    return bits, gl, gp


def sga_quantize(latents, temperature, diff_sampling, uniforms=None, seed=0, rng_step=None, want_dw=True):
    """SGA sample of the latents (shacira_sga_quantize): returns (w_hat, d w_hat / d w | None). `temperature`: python
    float or device float32 scalar tensor; `uniforms` [T, C, 2] (optional): the U(0,1) draws, else drawn in the kernel."""
    lib = load()
    latents = _f32c(latents, "latents")
    dev = latents.device
    if not isinstance(temperature, torch.Tensor):
        temperature = torch.tensor(float(temperature), dtype=torch.float32, device=dev)
    temperature = _f32c(temperature, "temperature")
    if uniforms is not None:
        uniforms = _f32c(uniforms, "uniforms")
        if uniforms.numel() != 2 * latents.numel():
            raise ShaciraError(ERR_INVALID_ARGUMENT, "uniforms must be [T, C, 2]")
    w_hat = torch.empty_like(latents)
    dw = torch.empty_like(latents) if want_dw else None
    with torch.cuda.device(dev):
        _check(lib.shacira_sga_quantize(_ptr(latents), _ptr(uniforms), latents.numel(), _ptr(temperature),
                                        1 if diff_sampling else 0, int(seed) & 0xFFFFFFFFFFFFFFFF, _ptr(rng_step),
                                        _ptr(w_hat), _ptr(dw), _stream()))
    return w_hat, dw


def mlp_mse_step(features, target, W1, b1, W2, b2, W3, b3, want_pred=False, absmax_out=None):
    """Fused decoder MLP + MSE: returns (loss scalar tensor, grad_features, pred | None, grads dict).
    `absmax_out` [in_dim] float32 (optional, in_dim = 16): receives max |grad_features| per column."""
    lib = load()
    features, target = _f32c(features, "features"), _f32c(target, "target")
    ws = [_f32c(t, "weights") for t in (W1, b1, W2, b2, W3, b3)]
    n, IN = features.shape
    H, OUT = ws[0].shape[0], ws[4].shape[0]
    dev = features.device
    gx = torch.empty_like(features)
    pred = torch.empty((n, OUT), dtype=torch.float32, device=dev) if want_pred else None
    n_par = H * IN + H + H * H + H + OUT * H + OUT
    out = torch.empty(2 + n_par, dtype=torch.float32, device=dev)  # 8-byte loss + packed gradients
    with torch.cuda.device(dev):
        _check(lib.shacira_mlp_mse_step_bounded(_ptr(features), _ptr(target), n, IN, H, OUT, *[_ptr(w) for w in ws],
                                                _ptr(gx), _ptr(pred), _ptr(out), _ptr(absmax_out), _stream()))
    sse = out[:2].view(torch.float64)[0]
    loss = (sse / (n * OUT)).to(torch.float32)
    return loss, gx, pred, out[2:]  # packed gradients: W1 | b1 | W2 | b2 | W3 | b3


def split_mlp_grads(packed, IN, H, OUT):
    parts = torch.split(packed, [H * IN, H, H * H, H, OUT * H, OUT])
    return [parts[0].view(H, IN), parts[1], parts[2].view(H, H), parts[3], parts[4].view(OUT, H), parts[5]]


def quantize_symbols(latents, want_symbols=True):
    """Returns (symbols[T, C] int16 | None, minmax[C, 2] int32)."""
    lib = load()
    latents = _f32c(latents, "latents")
    T, C = latents.shape
    dev = latents.device
    sym = torch.empty((T, C), dtype=torch.int16, device=dev) if want_symbols else None
    mm = torch.empty((C, 2), dtype=torch.int32, device=dev)
    with torch.cuda.device(dev):
        _check(lib.shacira_quantize_symbols(_ptr(latents), T, C, _ptr(sym), _ptr(mm), _stream()))
    return sym, mm


def symbol_histogram(latents, lo, num_bins):
    """counts[C, num_bins] int64 of rint(latents[:, c]) - lo[c]."""
    lib = load()
    latents = _f32c(latents, "latents")
    T, C = latents.shape
    lo_arr, nlo = _i32_array(lo)
    if nlo != C:
        raise ShaciraError(ERR_INVALID_ARGUMENT, "lo must have one entry per channel")
    counts = torch.zeros((C, num_bins), dtype=torch.int64, device=latents.device)
    with torch.cuda.device(latents.device):
        _check(lib.shacira_symbol_histogram(_ptr(latents), T, C, lo_arr, num_bins, _ptr(counts), _stream()))
    return counts


def latent_step_host(coords, latents, first_idx, resolutions, bitwidth, A, shift, grad_output, round_flag=True,
                     feats_out=None, grad_latents_out=None):
    """Host-buffer fwd+bwd (end-to-end entry): every tensor lives in (ideally pinned) host memory."""
    lib = load()
    for name, t in (("coords", coords), ("latents", latents), ("A", A), ("grad_output", grad_output)):
        if t.is_cuda or t.dtype != torch.float32 or not t.is_contiguous():
            raise ShaciraError(ERR_INVALID_ARGUMENT, "%s must be a contiguous float32 HOST tensor" % name)
    dim = _dim_of(coords)
    fi, L = _i32_array(first_idx)
    rs, _ = _i32_array(resolutions)
    n, (T, C) = coords.shape[0], latents.shape
    F = A.shape[2]
    per_level = 1 if A.shape[0] == L and L > 1 else 0
    if feats_out is None:
        feats_out = torch.empty((n, L * F), dtype=torch.float32).pin_memory()
    if grad_latents_out is None:
        grad_latents_out = torch.empty((T, C), dtype=torch.float32).pin_memory()
    _check(lib.shacira_latent_step_host(dim, _ptr(coords), n, _ptr(latents), T, fi, rs, L, bitwidth, C, F,
                                        1 if round_flag else 0, _ptr(A), _ptr(shift), per_level, _ptr(grad_output),
                                        _ptr(feats_out), _ptr(grad_latents_out)))
    return feats_out, grad_latents_out


class HostSession:
    """Host-buffer session (shacira_host_session_*): fused latent fwd + bwd steps over one coordinate set with every
    array in (pinned) host memory, pipelined two steps deep. `step()` returns the slot whose host buffers it will fill;
    `wait(slot)` blocks until they are complete."""

    def __init__(self, coords, table_rows, first_idx, resolutions, bitwidth, latent_dim, feature_dim, per_level=False,
                 device=None):
        lib = load()
        self._check_host(coords, "coords")
        self.dim = _dim_of(coords)
        self.n, self.T, self.C, self.F = coords.shape[0], int(table_rows), int(latent_dim), int(feature_dim)
        fi, self.L = _i32_array(first_idx)
        rs, _ = _i32_array(resolutions)
        self.device = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        handle = ctypes.c_void_p(0)
        with torch.cuda.device(self.device):
            _check(lib.shacira_host_session_create(self.dim, self.n, self.T, fi, rs, self.L, int(bitwidth), self.C, self.F,
                                                   1 if per_level else 0, ctypes.byref(handle)))
            self.handle = handle
            _check(lib.shacira_host_session_set_coords(self.handle, _ptr(coords)))
        self._keep = [coords]

    @staticmethod
    def _check_host(t, name):
        if t is not None and (t.is_cuda or t.dtype != torch.float32 or not t.is_contiguous()):
            raise ShaciraError(ERR_INVALID_ARGUMENT, "%s must be a contiguous float32 HOST tensor" % name)

    def set_table(self, latents, A, shift=None, round_flag=True):
        for name, t in (("latents", latents), ("A", A), ("shift", shift)):
            self._check_host(t, name)
        with torch.cuda.device(self.device):
            _check(load().shacira_host_session_set_table(self.handle, _ptr(latents), _ptr(A), _ptr(shift),
                                                         1 if round_flag else 0))
        self._keep_table = (latents, A, shift)

    def step(self, grad_output, feats_out, grad_latents_out, grad_A_out=None, grad_shift_out=None):
        for name, t in (("grad_output", grad_output), ("feats_out", feats_out), ("grad_latents_out", grad_latents_out),
                        ("grad_A_out", grad_A_out), ("grad_shift_out", grad_shift_out)):
            self._check_host(t, name)
        slot = ctypes.c_int32(-1)
        with torch.cuda.device(self.device):
            _check(load().shacira_host_session_step_async(self.handle, _ptr(grad_output), _ptr(feats_out),
                                                          _ptr(grad_latents_out), _ptr(grad_A_out), _ptr(grad_shift_out),
                                                          ctypes.byref(slot)))
        return slot.value

    def wait(self, slot):
        with torch.cuda.device(self.device):
            _check(load().shacira_host_session_wait(self.handle, int(slot)))

    def close(self):
        if getattr(self, "handle", None) is not None and self.handle.value:
            with torch.cuda.device(self.device):
                load().shacira_host_session_destroy(self.handle)
            self.handle = ctypes.c_void_p(0)

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def ac_encode(symbols, cdf):
    """symbols: int16 numpy/torch CPU array of dense ranks; cdf: uint32 array [K+1]. Returns bytes."""
    import numpy as np
    lib = load()
    sym = np.ascontiguousarray(symbols, dtype=np.int16)
    cdf = np.ascontiguousarray(cdf, dtype=np.uint32)
    cap = int(sym.size * 2 + 64)
    out = np.empty(cap, dtype=np.uint8)
    r = lib.shacira_ac_encode(sym.ctypes.data, sym.size, cdf.ctypes.data, cdf.size - 1, out.ctypes.data, cap)
    if r < 0:
        raise ShaciraError(int(r), lib.shacira_last_error().decode("utf-8", "replace"))
    return out[:r].tobytes()


def ac_decode(stream, cdf, n):
    import numpy as np
    lib = load()
    buf = np.frombuffer(stream, dtype=np.uint8)
    cdf = np.ascontiguousarray(cdf, dtype=np.uint32)
    out = np.empty(n, dtype=np.int16)
    _check(lib.shacira_ac_decode(buf.ctypes.data, buf.size, cdf.ctypes.data, cdf.size - 1, out.ctypes.data, n))
    return out


class TableAdam:
    """Adam for ONE large float32 tensor (the latent table) with torch.optim.Adam semantics, one kernel per step
    (SURVEY section 8 row f-4). State lives on the device; `step()` is CUDA-graph capturable."""

    def __init__(self, param, lr, betas=(0.9, 0.999), eps=1e-8, weight_decay=0.0):
        self.param = param
        self.lr, self.betas, self.eps, self.weight_decay = float(lr), betas, float(eps), float(weight_decay)
        self.exp_avg = torch.zeros_like(param)
        self.exp_avg_sq = torch.zeros_like(param)
        self.step_count = torch.zeros((), dtype=torch.float32, device=param.device)

    def step(self, zero_grad=False):
        p = self.param
        if p.grad is None:
            return
        g = p.grad if p.grad.is_contiguous() else p.grad.contiguous()
        with torch.cuda.device(p.device):
            _check(load().shacira_adam_step(_ptr(p.data), _ptr(g), _ptr(self.exp_avg), _ptr(self.exp_avg_sq), p.numel(),
                                            self.lr, self.betas[0], self.betas[1], self.eps, self.weight_decay,
                                            _ptr(self.step_count), 1 if zero_grad else 0, _stream()))
