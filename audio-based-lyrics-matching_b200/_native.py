"""ctypes binding of include/wealy_b200.h.  No torch types cross this boundary: only raw device
pointers (tensor.data_ptr()), sizes and the current CUDA stream handle."""
import ctypes
import os

_LIB_PATH = os.environ.get("WEALY_LIB") or os.path.join(os.path.dirname(os.path.abspath(__file__)), "lib",
                                                       "libwealy_b200.so")

if not os.path.isfile(_LIB_PATH):
    raise ImportError(
        f"{_LIB_PATH} is missing: the CUDA extension has not been built. Run "
        "`python -c 'import __graft_entry__ as g; g.build()'` (there is no CPU fallback).")

lib = ctypes.CDLL(_LIB_PATH)

OK, ERR_BAD_ARG, ERR_UNSUPPORTED, ERR_CUDA, ERR_WORKSPACE, ERR_ID_RANGE = range(6)
F32, F16, BF16, F64 = 0, 1, 2, 3
MODE_COSSIM, MODE_COS, MODE_DOTSIM, MODE_DOT, MODE_SQEUC, MODE_EUC = range(6)
LOSS_NTXENT, LOSS_CLEWS = 0, 1
REDUX = {"min": 0, "max": 1, "mean": 2, "meanmin": 3, "minmean": 4}
OUT_COUNT = 16

c_i64, c_int, c_f32, c_vp, c_sz = ctypes.c_int64, ctypes.c_int, ctypes.c_float, ctypes.c_void_p, ctypes.c_size_t
c_f64 = ctypes.c_double


class LossCfg(ctypes.Structure):
    _fields_ = [("kind", c_int), ("passes", c_int), ("temperature", c_f32), ("gamma", c_f32), ("b", c_f32),
                ("eps", c_f32), ("epsilon", c_f32), ("uw", c_f32), ("numerically_friendly", c_int),
                ("label_noise", c_int), ("grad_dtype", c_int)]


# every symbol include/wealy_b200.h declares: (restype, argtypes)
SIGNATURES = {
    "wealy_last_error": (ctypes.c_char_p, []),
    "wealy_version": (c_int, []),
    "wealy_pool_release": (c_int, []),
    "wealy_pool_stats": (c_int, [ctypes.POINTER(c_i64), ctypes.POINTER(c_i64), ctypes.POINTER(c_i64), ctypes.POINTER(c_i64)]),
    "wealy_sim_matrix_workspace_bytes": (c_sz, [c_i64, c_i64, c_i64, c_int]),
    "wealy_sim_matrix": (c_int, [c_vp, c_i64, c_i64, c_vp, c_i64, c_i64, c_i64, c_int, c_int, c_f32, c_f32, c_int,
                                 c_vp, c_i64, c_int, c_vp, c_sz, c_vp]),
    "wealy_sim_matrix_f64_workspace_bytes": (c_sz, [c_i64, c_i64]),
    "wealy_sim_matrix_f64": (c_int, [c_vp, c_i64, c_i64, c_vp, c_i64, c_i64, c_i64, c_int, c_f64, c_f64, c_vp, c_i64, c_vp, c_sz,
                                     c_vp]),
    "wealy_sim_matrix_backward_workspace_bytes": (c_sz, [c_i64, c_i64, c_i64, c_int]),
    "wealy_sim_matrix_backward": (c_int, [c_vp, c_i64, c_i64, c_vp, c_i64, c_i64, c_i64, c_int, c_int, c_f32, c_int, c_vp, c_i64,
                                          c_vp, c_i64, c_vp, c_i64, c_vp, c_i64, c_vp, c_sz, c_vp]),
    "wealy_dot_matrix_backward_workspace_bytes": (c_sz, [c_i64, c_i64, c_i64, c_int]),
    "wealy_dot_matrix_backward": (c_int, [c_vp, c_i64, c_vp, c_i64, c_vp, c_i64, c_vp, c_i64, c_i64, c_i64, c_i64, c_int, c_int,
                                          c_vp, c_i64, c_vp, c_i64, c_vp, c_sz, c_vp]),
    "wealy_eval_plan_create": (c_int, [c_vp, c_vp, c_i64, c_vp, c_vp, c_i64, c_vp, ctypes.POINTER(c_vp)]),
    "wealy_eval_plan_info": (c_int, [c_vp, ctypes.POINTER(c_i64), ctypes.POINTER(c_i64), ctypes.POINTER(c_i64)]),
    "wealy_eval_run": (c_int, [c_vp, c_vp, c_i64, c_vp, c_i64, c_i64, c_int, c_f32, c_int, c_int, c_vp, c_vp, c_vp,
                               c_vp, c_vp, c_vp]),
    "wealy_eval_plan_create_host": (c_int, [c_vp, c_vp, c_i64, c_vp, c_vp, c_i64, c_vp, c_i64, c_i64, c_int, c_f32, c_int, c_vp,
                                            ctypes.POINTER(c_vp)]),
    "wealy_eval_run_host": (c_int, [c_vp, c_vp, c_i64, c_i64, c_int, c_f32, c_int, c_vp, c_vp, c_vp, c_vp]),
    "wealy_eval_run_chunked": (c_int, [c_vp, c_vp, c_i64, c_vp, c_i64, c_i64, c_int, c_f32, c_int, c_int, c_int, c_int, c_vp,
                                       c_vp, c_vp, c_vp, c_vp, c_vp]),
    "wealy_eval_run_ragged": (c_int, [c_vp, c_vp, c_i64, c_vp, c_i64, c_i64, c_int, c_f32, c_int, c_int, c_int, c_int, c_vp,
                                      c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp]),
    "wealy_eval_sweep_shard": (c_int, [c_vp, c_vp, c_i64, c_i64, c_int, c_f32, c_int, c_int, c_int, c_vp]),
    "wealy_eval_shard_prepare": (c_int, [c_vp, c_vp, c_i64, c_i64, c_int, c_f32, c_int, c_int, c_int, c_vp]),
    "wealy_eval_plan_thresholds": (c_int, [c_vp, ctypes.POINTER(c_vp), ctypes.POINTER(c_i64)]),
    "wealy_eval_shard_sweep": (c_int, [c_vp, c_i64, c_int, c_int, c_int, c_vp]),
    "wealy_eval_sweep_shard_tracks": (c_int, [c_vp, c_vp, c_i64, c_i64, c_int, c_f32, c_int, c_int, c_int, c_vp, c_int,
                                              c_int, c_vp]),
    "wealy_eval_shard_prepare_tracks": (c_int, [c_vp, c_vp, c_i64, c_i64, c_int, c_f32, c_int, c_int, c_int, c_vp, c_int,
                                                c_int, c_vp]),
    "wealy_eval_shard_sweep_tracks": (c_int, [c_vp, c_i64, c_int, c_int, c_int, c_vp, c_int, c_int, c_vp]),
    "wealy_eval_sweep_shard_topk": (c_int, [c_vp, c_vp, c_i64, c_i64, c_int, c_f32, c_int, c_int, c_int, c_int, c_vp, c_vp,
                                            c_vp, c_vp]),
    "wealy_eval_topk_merge": (c_int, [c_vp, c_vp, c_vp, c_int, c_i64, c_int, c_vp, c_vp, c_vp, c_vp]),
    "wealy_eval_plan_counts": (c_int, [c_vp, ctypes.POINTER(c_vp), ctypes.POINTER(c_i64)]),
    "wealy_eval_finish": (c_int, [c_vp, c_vp, c_vp, c_vp, c_vp]),
    "wealy_eval_plan_ranks": (c_int, [c_vp, c_vp, c_vp, c_vp, c_vp]),
    "wealy_eval_plan_last_sweep_ms": (c_int, [c_vp, ctypes.POINTER(c_f32)]),
    "wealy_eval_plan_last_topk_path": (c_int, [c_vp, ctypes.POINTER(c_int)]),
    "wealy_eval_plan_stage_ms": (c_int, [c_vp, ctypes.POINTER(c_f32)]),
    "wealy_eval_plan_destroy": (None, [c_vp]),
    "wealy_masked_reduce": (c_int, [c_vp, c_vp, c_i64, c_i64, c_int, c_int, c_f32, c_f32, c_vp, c_vp]),
    "wealy_masked_reduce_backward": (c_int, [c_vp, c_vp, c_i64, c_i64, c_int, c_int, c_f32, c_f32, c_int, c_vp, c_vp, c_vp]),
    "wealy_distance_redux": (c_int, [c_vp, c_vp, c_i64, c_int, c_int, c_int, c_int, c_int, c_int, c_f32, c_f32, c_vp, c_vp]),
    "wealy_distance_redux_backward": (c_int, [c_vp, c_vp, c_i64, c_int, c_int, c_int, c_int, c_int, c_int, c_f32, c_f32, c_vp,
                                              c_vp, c_vp]),
    "wealy_mean_pool": (c_int, [c_vp, c_vp, c_i64, c_i64, c_i64, c_int, c_vp, c_int, c_vp]),
    "wealy_segment_mean": (c_int, [c_vp, c_vp, c_i64, c_i64, c_int, c_vp, c_vp]),
    "wealy_triplet_mine": (c_int, [c_vp, c_vp, c_i64, c_vp, c_vp, c_vp]),
    "wealy_triplet_forward": (c_int, [c_vp, c_i64, c_i64, c_i64, c_int, c_vp, c_vp, c_f32, c_f32, c_f32, c_int, c_vp,
                                      c_vp, c_vp]),
    "wealy_triplet_backward": (c_int, [c_vp, c_i64, c_i64, c_i64, c_int, c_vp, c_vp, c_f32, c_f32, c_int, c_vp, c_vp,
                                       c_int, c_int, c_vp, c_vp, c_vp]),
    "wealy_loss_workspace_bytes": (c_sz, [c_i64, c_i64, c_int]),
    "wealy_loss_forward": (c_int, [ctypes.POINTER(LossCfg), c_vp, c_i64, c_i64, c_i64, c_int, c_vp, c_vp, c_vp, c_vp, c_vp,
                                   c_sz, c_vp]),
    "wealy_loss_backward": (c_int, [ctypes.POINTER(LossCfg), c_vp, c_i64, c_i64, c_i64, c_int, c_vp, c_vp, c_i64,
                                    c_vp, c_sz, c_vp]),
    "wealy_loss_dp_workspace_bytes": (c_sz, [c_i64, c_i64, c_int, c_i64]),
    "wealy_loss_dp_forward_local": (c_int, [ctypes.POINTER(LossCfg), c_vp, c_i64, c_i64, c_i64, c_int, c_vp, c_vp, c_i64,
                                            c_i64, c_vp, c_sz, c_vp]),
    "wealy_loss_dp_forward_phase": (c_int, [ctypes.POINTER(LossCfg), c_vp, c_i64, c_i64, c_i64, c_int, c_vp, c_vp, c_i64,
                                            c_i64, c_int, c_vp, c_sz, c_vp]),
    "wealy_loss_dp_buffers": (c_int, [ctypes.POINTER(LossCfg), c_vp, c_sz, c_i64, c_i64, c_i64, ctypes.POINTER(c_vp),
                                      ctypes.POINTER(c_i64), ctypes.POINTER(c_vp), ctypes.POINTER(c_vp)]),
    "wealy_loss_dp_record_bytes": (c_sz, [c_i64]),
    "wealy_loss_dp_pack": (c_int, [ctypes.POINTER(LossCfg), c_vp, c_sz, c_i64, c_i64, c_i64, c_i64, c_vp, c_vp]),
    "wealy_loss_dp_unpack": (c_int, [ctypes.POINTER(LossCfg), c_vp, c_sz, c_i64, c_i64, c_i64, c_vp, c_int, c_vp]),
    "wealy_loss_dp_forward_finish": (c_int, [ctypes.POINTER(LossCfg), c_i64, c_i64, c_i64, c_vp, c_vp, c_int, c_vp, c_sz,
                                             c_vp]),
    "wealy_loss_dp_backward": (c_int, [ctypes.POINTER(LossCfg), c_vp, c_i64, c_i64, c_i64, c_int, c_i64, c_i64, c_vp, c_vp,
                                       c_i64, c_vp, c_sz, c_vp]),
}
for _name, (_res, _args) in SIGNATURES.items():
    _fn = getattr(lib, _name)          # AttributeError here == a declared symbol is not exported
    _fn.restype = _res
    _fn.argtypes = _args


class WealyError(RuntimeError):
    pass


def last_error():
    msg = lib.wealy_last_error()
    return msg.decode("utf-8", "replace") if msg else ""


def check(status):
    """Map C status codes onto the exception types the reference raises (SURVEY.md 8(b))."""
    if status == OK:
        return
    msg = last_error()
    if status == ERR_BAD_ARG:
        raise AssertionError(msg)
    if status == ERR_UNSUPPORTED:
        raise NotImplementedError(msg)
    if status == ERR_ID_RANGE:
        raise ValueError(msg)
    raise WealyError(f"wealy_b200 native call failed (status {status}): {msg}")


def dtype_code(t, allow_f64=False):
    import torch
    table = {torch.float32: F32, torch.float16: F16, torch.bfloat16: BF16}
    if allow_f64:
        table[torch.float64] = F64
    try:
        return table[t]
    except KeyError:
        raise NotImplementedError(f"wealy_b200: dtype {t} is not supported by this CUDA entry point "
                                  "(float32 / float16 / bfloat16" + (" / float64" if allow_f64 else "") + " only)") from None


def require_cuda(*tensors):
    for t in tensors:
        if not t.is_cuda:
            raise RuntimeError("wealy_b200 computes on CUDA only (no CPU fallback): got a tensor on "
                               f"{t.device}; move it with .cuda() first")


def stream_ptr(device):
    import torch
    return ctypes.c_void_p(torch.cuda.current_stream(device).cuda_stream)
