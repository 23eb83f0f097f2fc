"""ctypes binding of `libfoodrec_b200.so` (the C ABI in include/foodrec_b200.h).

The product path has no fallback: if the library is missing this module raises, and every wrapper
raises `FoodRecError` on a non-zero return code.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libfoodrec_b200.so")


class FoodRecError(RuntimeError):
    pass


def _load():
    if not os.path.exists(LIB_PATH):
        raise FoodRecError(
            f"{LIB_PATH} is not built: run `make` (or `python -c 'import __graft_entry__ as g; g.build()'`) "
            "at the repo root. foodrec_b200 has no CPU or eager fallback.")
    import torch  # noqa: F401  (loads the CUDA runtime the library links against)
    return C.CDLL(LIB_PATH, mode=C.RTLD_GLOBAL)


lib = _load()

_p, _i32, _i64, _f32 = C.c_void_p, C.c_int32, C.c_int64, C.c_float

SIGNATURES = {
    "fr_version": (C.c_int, []),
    "fr_last_error": (C.c_char_p, []),
    "fr_launch_count": (_i64, []),
    "fr_profile_enable": (C.c_int, [C.c_int]),
    "fr_profile_dump": (C.c_int, [C.c_char_p, _i64]),
    "fr_spmm_plan_sizes": (C.c_int, [_p, _i32, _i32, C.POINTER(_i64), C.POINTER(_i64), C.POINTER(_i64)]),
    "fr_spmm_plan_fill": (C.c_int, [_p, _i32, _i32, _p, _p]),
    "fr_spmm_csr_f32": (C.c_int, [_p, _i64, _p, _i64, _p, _p, _i32, _p, _p, _f32, _f32, _p, _i32, _p, _p, _p, _p]),
    "fr_spmm_csr_f32_split": (C.c_int, [_p, _i64, _p, _i64, _p, _p, _i32, _p, _p, _i32, _p, _p, _i32, _f32, _f32, _p, _i32,
                                        _p, _p, _p, _p]),
    "fr_spmm_task_blocks": (_i64, [_i64]),
    "fr_spmm_csr_f32_grouped": (C.c_int, [_p, _i32, _i32, _p, _i64, _p]),
    "fr_adam_step": (C.c_int, [_p, _i32, C.c_double, C.c_double, C.c_double, C.c_double, _p, _p, _p]),
    "fr_rank_loss_ws_floats": (_i64, []),
    "fr_rank_loss_fwd": (C.c_int, [_p, _i32, _i64, _p, _p, _p, _i32, _f32, _i32, _p, _p, _p, _f32, _p, _p, _p, _p, _p]),
    "fr_rank_loss_bwd": (C.c_int, [_p, _i32, _i64, _p, _p, _p, _i32, _p, _p, _p, _i32, _p, _p, _p, _p, _f32, _p, _p, _p, _p]),
    "fr_bpr_scores_fwd": (C.c_int, [_p, _p, _i64, _f32, _p, _p, _p]),
    "fr_l2_norm_f32": (C.c_int, [_p, _i64, _p, _p]),
    "fr_spmm_csr_f32_masked": (C.c_int, [_p, _i64, _p, _i64, _p, _p, _i32, _p, _p, _f32, _f32, _p, _p, _p, _p, _p, _p]),
    "fr_dcor_ws_floats": (_i64, [_i32]),
    "fr_dcor_fwd": (C.c_int, [_p, _i32, _i32, _p, _i32, _p, _i32, _f32, _p, _p, _p, _p, _p, _p, _p]),
    "fr_sum_rows": (C.c_int, [_p, _i32, _i32, _i64, _p, _p]),
    "fr_spread_rows": (C.c_int, [_p, _i32, _i64, _p, _p, _i32, _i32, _p, _p, _p]),
    "fr_dcor_bwd": (C.c_int, [_p, _i32, _i32, _p, _i32, _p, _i32, _p, _p, _p, _p, _p, _p, _p, _p, _p]),
    "fr_dcor_bwd_ws_floats": (_i64, [_i32]),
    "fr_f32_to_bf16": (C.c_int, [_p, _p, _i64, _i32, _i32, _p]),
    "fr_gemm_topk_ws_bytes": (_i64, [_i32]),
    "fr_gemm_topk_bf16": (C.c_int, [_p, _i32, _p, _i32, _i32, _f32, _p, _p, _p, _p, _i32, _p, _p, _p, _i64, _p]),
    "fr_max_row_norm": (C.c_int, [_p, _i64, _i32, _p, _p]),
    "fr_rescore_topk_f32": (C.c_int, [_p, _p, _p, _i32, _f32, _p, _i32, _p, _p, _i32, _i32, _i32, _p, _p, _i32, _p, _p, _p]),
    "fr_exact_topk_f32": (C.c_int, [_p, _p, _i32, _p, _i32, _i32, _f32, _p, _i32, _p, _p, _p, _i32, _p, _p, _p, _p]),
    "fr_exact_topk_thr_ws_bytes": (_i64, [_i32]),
    "fr_exact_topk_thr_f32": (C.c_int, [_p, _p, _i32, _p, _i32, _i32, _f32, _p, _i32, _p, _p, _p, _i32, _p, _p, _p, _p, _p, _p]),
    "fr_csr_from_coo": (C.c_int, [_p, _i64, _i32, _p, _p, _p]),
    "fr_cosine_mean_fwd": (C.c_int, [_p, _p, _p, _i64, _i32, _p, _p, _p, _p, _p]),
    "fr_cosine_mean_bwd": (C.c_int, [_p, _p, _p, _i64, _i32, _p, _p, _p, _p, _p, _p, _p]),
    "fr_infonce_ws_floats": (_i64, [_i32]),
    "fr_infonce_fwd": (C.c_int, [_p, _i32, _i32, _f32, _i32, _p, _p, _p, _p, _p, _p, _p]),
    "fr_infonce_bwd": (C.c_int, [_p, _p, _p, _p, _i32, _i32, _f32, _i32, _p, _p, _p]),
    "fr_gather_rows": (C.c_int, [_p, _i32, _p, _i64, _p, _p]),
    "fr_scatter_add_rows": (C.c_int, [_p, _i32, _p, _i64, _p, _p]),
    "fr_pair_scores": (C.c_int, [_p, _p, _i32, _p, _p, _i64, _p, _p]),
    "fr_comm_version": (C.c_int, []),
    "fr_comm_unique_id": (C.c_int, [_p]),
    "fr_comm_init": (C.c_int, [_p, _i32, _i32, _p]),
    "fr_comm_destroy": (C.c_int, [_p]),
    "fr_allgather_rows": (C.c_int, [_p, _p, _i64, _i32, _p, _p]),
    "fr_reduce_scatter_rows": (C.c_int, [_p, _p, _i64, _i32, _p, _p]),
    "fr_peer_alloc": (C.c_int, [_i64, _p, _p]),
    "fr_peer_open": (C.c_int, [_p, _p]),
    "fr_peer_close": (C.c_int, [_p]),
    "fr_peer_free": (C.c_int, [_p]),
    "fr_push_rows": (C.c_int, [_p, _i64, _i32, _p, _i32, _i64, _p]),
    "fr_spmm_csr_f32_push": (C.c_int, [_p, _i64, _p, _i64, _p, _p, _i32, _p, _p, _f32, _f32, _p, _p, _p, _p, _i32, _i64, _p]),
    "fr_probe_gather": (C.c_int, [_p, _i32, _p, _i64, _i32, _i32, _p, _p]),
    "fr_sample_negatives": (C.c_int, [_p, _p, _p, _i64, _i32, C.c_uint64, C.c_uint64, _p, _p, _p]),
    "fr_schgn_attend": (C.c_int, [_p, _p, _i32, _p, _i32, _p, _i32, _p, _p, _p, _p, _p, _p, _p, _i32, _p, _p, _p]),
    "fr_schgn_score": (C.c_int, [_p, _p, _i32, _p, _p, _p, _p, _p, _p, _i32, _i32, _p, _p]),
    "fr_schgn_score_topk_ws_bytes": (_i64, [_i32, _i32, _i32]),
    "fr_schgn_score_topk": (C.c_int, [_p, _p, _i32, _p, _p, _p, _p, _p, _p, _i32, _i32, _p, _p, _p, _i32, _p, _p, _p, _p]),
    "fr_schgn_attend_pairs_ws_bytes": (_i64, [_i32, _i64, _i32]),
    "fr_schgn_attend_pairs": (C.c_int, [_p, _p, _i32, _p, _p, _i64, _p, _i32, _p, _i32, _p, _p, _p, _p, _p, _p, _p, _i32,
                                        _p, _i64, _p, _p, _p, _p]),
    "fr_schgn_score_pairs": (C.c_int, [_p, _p, _i32, _p, _p, _i64, _p, _p, _p, _p, _p, _p, _i32, _i32, _p, _p]),
    "fr_eval_metrics_ws_bytes": (_i64, []),
    "fr_topk_metrics": (C.c_int, [_p, _i32, _i64, _i32, _p, _p, _p, _p, _i32, _p, _p, _p, _p, _p, _p]),
    "fr_by_user_metrics": (C.c_int, [_p, _p, _p, _i64, _i32, _p, _i32, _p, _p, _p, _p]),
}

class SpmmTask(C.Structure):
    """`fr_spmm_task` of include/foodrec_b200.h (one propagation of a grouped launch)."""
    _fields_ = [("seg", _p), ("n_seg", _i64), ("long_rows", _p), ("n_long", _i64), ("col_idx", _p), ("val", _p),
                ("X0", _p), ("X1", _p), ("x_split", _i32), ("Z0", _p), ("Z1", _p), ("z_split", _i32),
                ("alpha", _f32), ("beta", _f32), ("Y", _p), ("partial", _p), ("counters", _p)]


class AdamTensor(C.Structure):
    """`fr_adam_tensor` of include/foodrec_b200.h."""
    _fields_ = [("param", _p), ("grad", _p), ("exp_avg", _p), ("exp_avg_sq", _p), ("n", _i64)]


for _name, (_res, _args) in SIGNATURES.items():
    _fn = getattr(lib, _name)
    _fn.restype = _res
    _fn.argtypes = _args


def check(rc: int, what: str = ""):
    if rc != 0:
        msg = lib.fr_last_error().decode("utf-8", "replace")
        raise FoodRecError(f"{what or 'foodrec_b200'} failed (rc={rc}): {msg}")


def ptr(t):
    """Device (or host) address of a torch tensor / numpy array, or None."""
    if t is None:
        return None
    if hasattr(t, "data_ptr"):
        return t.data_ptr()
    return t.ctypes.data


def stream_ptr():
    import torch
    return torch.cuda.current_stream().cuda_stream


def launch_count() -> int:
    return int(lib.fr_launch_count())


class kernel_profile:
    """`with kernel_profile() as prof: ...` -> `prof.result` = {kernel: (launches, total_us)} for the
    launches of this library inside the block (CUDA events on the launch stream; eager launches only)."""

    def __enter__(self):
        lib.fr_profile_dump(None, 0)
        lib.fr_profile_enable(1)
        self.result = {}
        return self

    def __exit__(self, *exc):
        lib.fr_profile_enable(0)
        buf = C.create_string_buffer(1 << 16)
        lib.fr_profile_dump(buf, len(buf))
        for line in buf.value.decode().splitlines():
            name, n, us = line.rsplit(",", 2)
            self.result[name] = (int(n), float(us))
        return False
