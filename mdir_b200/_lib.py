"""ctypes binding of libmdir_b200.so (include/mdir_b200.h).

There is NO fallback: if the shared library is missing or a call fails, this raises.
PyTorch is used only for device memory and streams; every kernel is reached through the
C ABI with raw pointers."""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libmdir_b200.so")
_lib = None
ABI_VERSION = 2


class ImageDesc(C.Structure):
    _fields_ = [("src_off", C.c_int64), ("dst_off", C.c_int64), ("H", C.c_int32), ("W", C.c_int32),
                ("src_pitch", C.c_int32), ("dst_pitch", C.c_int32)]


_vp, _i, _i64, _f, _d, _u32, _u64, _sz = C.c_void_p, C.c_int, C.c_int64, C.c_float, C.c_double, C.c_uint32, C.c_uint64, C.c_size_t

# name -> (restype, argtypes): must list every symbol declared in include/mdir_b200.h
PROTOTYPES = {
    "mdir_abi_version": (_i, []),
    "mdir_last_error": (C.c_char_p, []),
    "mdir_device_check": (_i, []),
    "mdir_launch_count": (_u64, []),
    "mdir_tune": (_i, [_i, _i]),
    "mdir_pool": (_i, [_i, _vp, _vp, _vp, _i, _i, _i, _f, _f, _vp, _vp]),
    "mdir_l2n": (_i, [_vp, _i, _i, _i, _f, _vp, _vp]),
    "mdir_ms_aggregate": (_i, [_vp, _i, _i, _i, _f, _f, _vp, _vp, _vp]),
    "mdir_whiten_project": (_i, [_vp, _vp, _i, _i, _vp, _i, _f, _vp, _vp]),
    "mdir_whiten_tc_workspace_bytes": (_sz, [_i, _i, _i]),
    "mdir_whiten_project_tc": (_i, [_vp, _vp, _i, _i, _vp, _i, _f, _vp, _vp, _vp]),
    "mdir_clahe_workspace_bytes": (_sz, [_i, _i, _i]),
    "mdir_clahe_u8": (_i, [_vp, _vp, _vp, _i, _i, _i, _d, _i, _i, _vp, _vp]),
    "mdir_rgb_to_l_u8": (_i, [_vp, _vp, _i, _i64, _vp, _vp, _vp]),
    "mdir_lab_clahe_to_rgb": (_i, [_vp, _vp, _i, _i64, _vp, _vp, _vp, _vp, _vp]),
    "mdir_pack_bf16": (_i, [_vp, _i64, _i, _i, _vp, _vp]),
    "mdir_sim_scan_bf16": (_i, [_vp, _i64, _vp, _i, _i, _i, _i, _i, _vp, _i64, _vp, _u32, _vp, _vp, _i, _i, _vp]),
    "mdir_sim_scan_dense_bf16": (_i, [_vp, _i64, _vp, _i, _i, _vp, _i64, _vp]),
    "mdir_sim_scan_wide_bf16": (_i, [_vp, _i64, _vp, _i, _i, _i, _i, _i, _vp, _i64, _vp, _u32, _vp, _vp, _i, _i, _vp]),
    "mdir_sim_scan_fused_workspace_bytes": (_sz, [_i]),
    "mdir_sim_scan_fused_bf16": (_i, [_vp, _i64, _vp, _i, _i, _i, _vp, _u32, _vp, _vp, _i, _i, _vp, _vp]),
    "mdir_sim_scan_fused_i8": (_i, [_vp, _vp, _i64, _vp, _vp, _i, _i, _i, _vp, _u32, _vp, _vp, _i, _i, _vp, _vp]),
    "mdir_sim_scan_tf32": (_i, [_vp, _i64, _vp, _i, _i, _i, _i, _i, _vp, _i64, _vp, _u32, _vp, _vp, _i, _i, _vp]),
    "mdir_split_tf32x3": (_i, [_vp, _i64, _i, _i, _vp, _vp]),
    "mdir_make_key": (_u64, [_f, _u32]),
    "mdir_key_score": (_f, [_u64]),
    "mdir_select_kth": (_i, [_vp, _i64, _i64, _i, _i, _i, _u32, _vp, _vp, _i64, _vp, _i, _i, _i, _vp]),
    "mdir_topk_finalize": (_i, [_vp, _i64, _vp, _i, _i, _i, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp]),
    "mdir_topk_finalize_rescore": (_i, [_vp, _i64, _vp, _i, _i, _i, _i, _i, _i, _vp, _i64, _u32, _vp, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "mdir_topk_finalize_rescore_eps": (_i, [_vp, _i64, _vp, _i, _i, _i, _i, _i, _i, _vp, _i64, _u32, _vp, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "mdir_pack_stats": (_i, [_vp, _vp, _i64, _i, _vp, _vp]),
    "mdir_pack_stats_i8": (_i, [_vp, _vp, _i64, _i, _vp, _vp, _vp, _vp]),
    "mdir_pack_q_i8": (_i, [_vp, _i, _i, _vp, _vp, _vp, _vp, _vp]),
    "mdir_rescore_f32": (_i, [_vp, _i64, _u32, _vp, _i, _i, _vp, _i, _vp, _vp]),
    "mdir_qe_accumulate": (_i, [_vp, _i64, _u32, _i, _vp, _vp, _i, _i, _f, _vp, _vp]),
    "mdir_add_l2n": (_i, [_vp, _vp, _i, _i, _vp, _vp]),
    "mdir_map_workspace_bytes": (_sz, [_i64, _i]),
    "mdir_compute_ap": (_i, [_vp, _i64, _i, _vp, _vp, _vp, _i64, _vp, _vp, _i, _vp, _vp, _vp, _vp]),
    "mdir_topk_plan": (_i, [_i64, _i, _i, _vp, _vp, _vp]),
    "mdir_sim_topk_workspace_bytes": (_sz, [_i]),
    "mdir_sim_topk_bf16": (_i, [_vp, _vp, _vp, _i64, _vp, _i, _i, _i, _i, _u32, _i, _vp, _vp, _vp, _vp, _vp, _vp]),
    "mdir_gem_head_workspace_bytes": (_sz, [_i, _i, _i, _i]),
    "mdir_gem_head": (_i, [_i, _vp, _vp, _vp, _i, _i, _i, _i, _f, _f, _f, _vp, _vp, _vp, _i, _vp, _vp, _vp]),
    "mdir_shard_mailbox_bytes": (_sz, [_i, _i, _i]),
    "mdir_p2p_alloc": (_i, [_sz, _vp, _vp]),
    "mdir_p2p_open": (_i, [_vp, _vp]),
    "mdir_p2p_close": (_i, [_vp]),
    "mdir_p2p_free": (_i, [_vp]),
    "mdir_shard_exchange_merge": (_i, [_vp, _i, _i, _i, _i, _i, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp]),
    "mdir_shard_status": (_i, [_vp, _vp]),
    "mdir_mine_negatives": (_i, [_vp, _i64, _i64, _i, _vp, _vp, _i, _vp, _vp, _vp]),
    "mdir_pair_l2dist": (_i, [_vp, _vp, _vp, _i, _i, _i, _f, _vp, _vp]),
    "mdir_gemm_f64_workspace_bytes": (_sz, [_i, _i, _i64]),
    "mdir_gemm_f64": (_i, [_vp, _i64, _vp, _vp, _i64, _vp, _i, _i, _i, _i64, _d, _vp, _i64, _vp, _vp]),
    "mdir_pair_diff_f64": (_i, [_vp, _i64, _i, _i64, _vp, _vp, _i64, _vp, _vp]),
    "mdir_cols_mean_f64": (_i, [_vp, _i64, _i, _i64, _vp, _i64, _vp, _vp]),
    "mdir_f32_to_f64": (_i, [_vp, _i64, _vp, _vp]),
    "mdir_rank_workspace_bytes": (_sz, [_i64, _i]),
    "mdir_rank_scores": (_i, [_vp, _i64, _i, _i, _vp, _i64, _vp, _vp]),
    "mdir_rank_fast_workspace_bytes": (_sz, [_i64, _i]),
    "mdir_rank_scores_fast": (_i, [_vp, _i64, _i, _i, _vp, _i64, _vp, _vp, _vp]),
    "mdir_rank_hist_workspace_bytes": (_sz, [_i64, _i]),
    "mdir_rank_scores_hist": (_i, [_vp, _i64, _i, _i, _vp, _i64, _vp, _vp, _vp]),
}


class MdirError(RuntimeError):
    pass


def lib():
    """The loaded library; raises MdirError when it has not been built (no fallback)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise MdirError("%s is missing: run `python -m mdir_b200.build` (nvcc, sm_100a). "
                            "mdir_b200 has no CPU or PyTorch fallback." % LIB_PATH)
        l = C.CDLL(LIB_PATH)
        for name, (res, args) in PROTOTYPES.items():
            fn = getattr(l, name)
            fn.restype = res
            fn.argtypes = args
        if l.mdir_abi_version() != ABI_VERSION:
            raise MdirError("libmdir_b200.so ABI mismatch")
        _lib = l
    return _lib


def check(rc, what=""):
    if rc != 0:
        msg = lib().mdir_last_error()
        raise MdirError("%s failed (code %d): %s" % (what or "libmdir_b200 call", rc, (msg or b"").decode()))


def stream():
    import torch
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def ptr(t):
    """Device pointer of a torch tensor (None -> NULL)."""
    return C.c_void_p(t.data_ptr()) if t is not None else C.c_void_p(0)


def require_cuda(t, name="tensor"):
    if not t.is_cuda:
        raise MdirError("%s must live on a CUDA device (mdir_b200 has no CPU path); got %s" % (name, t.device))
    return t
