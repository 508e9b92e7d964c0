"""ctypes binding of libdiffmm_b200.so (the C ABI declared in include/diffmm_b200.h).

The product path has no CPU or PyTorch fallback: if the shared library is missing, or a call
returns a non-zero status, this module raises.  PyTorch is used only for device memory, streams
and torch.distributed.
"""
from __future__ import annotations

import ctypes as C
import os
import threading

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libdiffmm_b200.so")

c_i64, c_i32, c_f32, c_vp = C.c_int64, C.c_int32, C.c_float, C.c_void_p


class GemmEpilogue(C.Structure):
    """Mirror of struct dmm_gemm_epilogue."""
    _fields_ = [
        ("bias", c_vp), ("act", c_i32), ("alpha", c_f32), ("beta", c_f32),
        ("residual", c_vp), ("ld_res", c_i64),
        ("out_f32", c_vp), ("ld_out", c_i64),
        ("out_hi", c_vp), ("out_lo", c_vp), ("ld_out16", c_i64),
        ("res_hi", c_vp), ("res_lo", c_vp), ("ld_res16", c_i64),
        ("res_pre_act", c_i32), ("post_act", c_i32), ("post_bias", c_vp),
        ("cmax", c_vp), ("ld_cmax", c_i64),
    ]


class NceProblem(C.Structure):
    """Mirror of struct dmm_nce_problem."""
    _fields_ = [("v1", c_vp), ("ld1", c_i64), ("v2", c_vp), ("ld2", c_i64), ("idx", c_vp), ("row_offset", c_i64),
                ("temperature", c_f32), ("weight", c_f32)]


class BprProblem(C.Structure):
    """Mirror of struct dmm_bpr_problem."""
    _fields_ = [("emb", c_vp), ("ld_emb", c_i64), ("item_offset", c_i64), ("users", c_vp), ("pos", c_vp), ("neg", c_vp)]


# name -> (restype, argtypes); every symbol of include/diffmm_b200.h must appear here
PROTOTYPES = {
    "dmm_version": (C.c_int, []),
    "dmm_last_error": (C.c_char_p, []),
    "dmm_init": (C.c_int, [C.c_int, C.POINTER(c_vp)]),
    "dmm_destroy": (None, [c_vp]),
    "dmm_num_sms": (C.c_int, [c_vp]),
    "dmm_pack_bf16": (C.c_int, [c_vp, c_vp, c_i64, c_i64, c_i64, c_vp, c_vp, c_i64, C.c_int, c_vp]),
    "dmm_pack_bf16_pair": (C.c_int, [c_vp, c_vp, c_i64, c_i64, c_i64, c_vp, c_vp, c_i64, c_vp, c_vp, c_i64, c_vp]),
    "dmm_csr_rows_to_dense": (C.c_int, [c_vp, c_vp, c_vp, c_vp, c_i64, c_i64, c_i64, c_vp, c_i64, c_vp, c_i64, c_vp]),
    "dmm_time_embedding": (C.c_int, [c_vp, c_vp, c_i64, c_i64, C.c_int, c_vp, c_vp, c_vp, c_vp, c_i64, c_i64, c_vp, c_vp]),
    "dmm_time_bias": (C.c_int, [c_vp, c_i64, c_i64, C.c_int, c_vp, c_vp, c_vp, c_i64, c_i64, c_vp, c_i64, c_vp, c_vp]),
    "dmm_csr_gather_act": (C.c_int, [c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_i64, c_i64, c_i64, c_vp, c_vp, c_i64, c_vp, C.c_int,
                                     c_i64, c_vp, c_vp, c_i64, c_vp, c_i64, c_vp]),
    "dmm_csr_gather_act_split": (C.c_int, [c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_i64, c_i64, c_i64, c_i64, c_vp, c_vp, c_i64,
                                           c_vp, C.c_int, c_i64, c_vp, c_vp, c_i64, c_vp, c_i64, c_vp]),
    "dmm_csr_qsample_values_rng": (C.c_int, [c_vp, c_vp, c_vp, c_vp, c_i64, c_i64, c_i64, c_vp, c_f32, c_f32, c_vp, C.c_int,
                                             c_vp]),
    "dmm_csr_qsample_values": (C.c_int, [c_vp, c_vp, c_vp, c_vp, c_i64, c_i64, c_i64, c_vp, c_i64, c_f32, c_f32, c_vp, c_vp]),
    "dmm_rows_long_first": (C.c_int, [c_vp, c_vp, c_i64, c_i64, c_i64, c_vp, c_vp, c_vp]),
    "dmm_gemv_f32": (C.c_int, [c_vp, c_vp, c_i64, c_i64, c_i64, c_vp, c_vp, c_vp]),
    "dmm_bias_act_pack": (C.c_int, [c_vp, c_vp, c_i64, c_vp, c_i64, c_i64, C.c_int, c_vp, c_vp, c_i64, c_vp]),
    "dmm_csr_axpy_bf16": (C.c_int, [c_vp, c_vp, c_vp, c_vp, c_i64, c_i64, c_i64, c_f32, c_vp, c_vp, c_i64, c_vp]),
    "dmm_q_sample": (C.c_int, [c_vp, c_vp, c_i64, c_vp, c_i64, c_vp, c_vp, c_i64, c_i64, C.c_int,
                               c_vp, c_i64, c_vp, c_vp, c_i64, c_vp]),
    "dmm_gemm_bf16_tn": (C.c_int, [c_vp, c_vp, c_vp, c_i64, c_vp, c_vp, c_i64, c_i64, c_i64, c_i64,
                                   C.POINTER(GemmEpilogue), c_vp]),
    "dmm_gemm_splitk_workspace_bytes": (c_i64, [c_vp, c_i64, c_i64, c_i64]),
    "dmm_gemm_bf16_tn_splitk": (C.c_int, [c_vp, c_vp, c_i64, c_vp, c_i64, c_i64, c_i64, c_i64, c_vp, c_i64, c_vp, c_vp, c_i64,
                                          c_vp, c_i64, c_vp]),
    "dmm_gemm_f32_tn": (C.c_int, [c_vp, c_vp, c_i64, c_vp, c_i64, c_i64, c_i64, c_i64, C.POINTER(GemmEpilogue), c_vp]),
    "dmm_topk_workspace_bytes": (c_i64, [c_i64, c_i64]),
    "dmm_topk_edges": (C.c_int, [c_vp, c_vp, c_i64, c_i64, c_i64, c_vp, c_i64, c_vp, c_vp, c_vp, c_vp, c_vp, c_i64, c_i64,
                                 c_vp]),
    "dmm_topk_pruned_workspace_bytes": (c_i64, [c_i64, c_i64, c_i64]),
    "dmm_topk_edges_pruned": (C.c_int, [c_vp, c_vp, c_i64, c_i64, c_i64, c_vp, c_i64, c_vp, c_i64, c_vp, c_vp, c_vp, c_vp,
                                        c_vp, c_i64, c_i64, c_vp]),
    "dmm_build_adj_workspace_bytes": (c_i64, [c_i64, c_i64, c_i64]),
    "dmm_build_norm_adj_csr": (C.c_int, [c_vp, c_vp, c_vp, c_i64, c_i64, c_i64, c_vp, c_vp, c_vp, c_vp, c_i64, c_vp, c_vp]),
    "dmm_spmm_plan_bytes": (c_i64, [c_i64, c_i64]),
    "dmm_spmm_plan": (C.c_int, [c_vp, c_vp, c_i64, c_i64, c_vp, c_i64, c_vp]),
    "dmm_spmm_workspace_bytes": (c_i64, [c_i64, c_i64]),
    "dmm_spmm_csr": (C.c_int, [c_vp, c_vp, c_vp, c_vp, c_i64, c_i64, c_vp, c_i64, c_i64, c_f32, c_f32,
                               c_vp, c_i64, c_vp, c_i64, c_vp, c_i64, c_vp, c_i64, c_vp]),
    "dmm_spmm_table_bf16": (C.c_int, [c_vp, c_vp, c_i64, c_i64, c_vp, c_i64, c_i64, c_vp, c_i64, c_vp, c_vp]),
    "dmm_spmm_norm_bf16": (C.c_int, [c_vp, c_vp, c_i64, c_i64, c_i64, c_vp, c_f32, c_f32, c_vp, c_i64, c_vp, c_i64, c_vp, c_i64,
                                     c_vp, c_i64, c_vp]),
    "dmm_sign_noise_": (C.c_int, [c_vp, c_vp, c_i64, c_vp, c_i64, c_i64, c_i64, c_f32, c_vp]),
    "dmm_adam_step": (C.c_int, [c_vp, C.c_int32, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, C.c_double, C.c_double, C.c_double,
                                c_vp]),
    "dmm_adam_step_host": (C.c_int, [c_vp, C.c_int32, c_vp, c_vp, c_vp, c_vp, c_vp, C.c_double, C.c_double, C.c_double, C.c_double,
                                     C.c_double, c_vp]),
    "dmm_rownorm_fwd": (C.c_int, [c_vp, c_vp, c_i64, c_i64, c_i64, c_f32, c_vp, c_i64, c_vp, c_vp]),
    "dmm_rownorm_bwd": (C.c_int, [c_vp, c_vp, c_i64, c_vp, c_vp, c_i64, c_i64, c_i64, c_vp, c_i64, c_vp]),
    "dmm_modal_mix_fwd": (C.c_int, [c_vp, c_vp, c_vp, c_vp, C.c_int32, c_f32, c_i64, c_vp, c_vp]),
    "dmm_modal_mix_partial_rows": (c_i64, [c_i64]),
    "dmm_modal_mix_bwd": (C.c_int, [c_vp, c_vp, c_vp, c_vp, c_vp, C.c_int32, c_f32, c_i64, c_vp, c_vp, c_vp, c_vp]),
    "dmm_bpr_fwd_bwd": (C.c_int, [c_vp, c_vp, c_i64, c_vp, c_i64, c_vp, c_vp, c_vp, c_i64, c_i64, c_f32,
                                  c_vp, c_vp, c_vp, c_vp, c_vp, c_vp]),
    "dmm_infonce_workspace_floats": (c_i64, [c_i64, c_i64, C.c_int]),
    "dmm_infonce_fwd": (C.c_int, [c_vp, c_vp, c_i64, c_vp, c_i64, c_vp, c_i64, c_i64, c_f32,
                                  c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp]),
    "dmm_infonce_bwd": (C.c_int, [c_vp, c_vp, c_i64, c_vp, c_i64, c_vp, c_i64, c_i64, c_f32,
                                  c_vp, c_vp, c_vp, c_f32, c_vp, c_vp, c_vp, c_vp]),
    "dmm_train_prep": (C.c_int, [c_vp, c_vp, c_i64, c_vp, c_i64, c_vp, c_vp, c_vp, c_i64, c_i64, C.c_int, c_vp, c_vp, c_vp, c_vp,
                                 c_i64, c_vp, c_i64, c_vp, c_vp]),
    "dmm_gate_fwd": (C.c_int, [c_vp, c_vp, c_i64, c_i64, c_vp, c_vp, c_vp, c_vp, c_vp, c_i64, c_vp]),
    "dmm_gate_bwd_pre": (C.c_int, [c_vp, c_vp, c_i64, c_vp, c_i64, c_vp, c_i64, c_vp, c_vp]),
    "dmm_diff_loss_fwd": (C.c_int, [c_vp, c_vp, c_i64, c_i64, c_i64, c_vp, c_i64, c_vp, c_i64, c_vp, c_i64, c_vp, c_vp, c_f32,
                                    c_vp, c_vp, c_vp, c_vp, c_vp]),
    "dmm_diff_loss_bwd": (C.c_int, [c_vp, c_vp, c_vp, c_vp, c_i64, c_vp, c_vp, c_vp, c_f32, c_i64, c_i64, c_vp, c_vp, c_vp,
                                    c_i64, c_vp, c_vp]),
    "dmm_hidden_bwd": (C.c_int, [c_vp, c_vp, c_i64, c_vp, c_i64, c_vp, c_vp, c_i64, c_vp, c_i64, c_i64, c_vp, c_i64, c_vp, c_vp, c_i64,
                                 c_vp, c_vp, c_vp, c_vp, c_i64, c_vp]),
    "dmm_transpose_bf16": (C.c_int, [c_vp, c_vp, c_vp, c_i64, c_i64, c_i64, c_vp, c_vp, c_i64, c_vp]),
    "dmm_colsum": (C.c_int, [c_vp, c_vp, c_i64, c_i64, c_i64, c_vp, c_vp, c_vp]),
    "dmm_atb_small_workspace_floats": (c_i64, [c_i64, c_i64]),
    "dmm_atb_small": (C.c_int, [c_vp, c_vp, c_i64, c_i64, c_vp, c_i64, c_i64, c_i64, c_vp, c_vp, c_vp]),
    "dmm_eval_mask_scores": (C.c_int, [c_vp, c_vp, c_vp, c_vp, c_i64, c_i64, c_vp, c_i64, c_f32, c_vp]),
    "dmm_eval_metrics": (C.c_int, [c_vp, c_vp, c_i64, c_i64, c_vp, c_i64, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp]),
    "dmm_eval_mask_scores_cmax": (C.c_int, [c_vp, c_vp, c_vp, c_vp, c_i64, c_i64, c_vp, c_i64, c_f32, c_vp, c_i64, c_vp]),
    "dmm_topn_rank": (C.c_int, [c_vp, c_vp, c_i64, c_i64, c_vp, c_i64, c_i64, c_vp, c_i64, c_vp, c_i64, c_vp]),
    "dmm_eval_metrics_cutoffs": (C.c_int, [c_vp, c_vp, c_i64, c_i64, c_i64, C.POINTER(c_i32), c_i64, c_vp, c_vp, c_vp, c_vp,
                                           c_vp, c_vp, c_vp]),
    "dmm_score_pairs": (C.c_int, [c_vp, c_vp, c_i64, c_i64, c_vp, c_i64, c_i64, c_i64, c_vp, c_vp, c_i64, C.c_int, c_vp, c_vp]),
    "dmm_rank_candidates": (C.c_int, [c_vp, c_vp, c_i64, c_vp, c_i64, c_i64, c_i64, c_vp, c_i64, c_i64, c_i64, c_i64, C.c_int,
                                      c_vp, c_i64, c_vp, c_i64, c_vp]),
    "dmm_bpr_infonce_workspace_floats":(c_i64, [c_i64, C.c_int, C.c_int]),
    "dmm_bpr_infonce_fwd": (C.c_int, [c_vp, C.POINTER(NceProblem), C.c_int, C.POINTER(BprProblem), c_i64, c_vp, c_vp, c_vp, c_vp,
                                      c_vp]),
    "dmm_bpr_infonce_bwd": (C.c_int, [c_vp, C.POINTER(NceProblem), C.c_int, C.POINTER(BprProblem), c_i64, c_vp, c_vp, c_vp, c_vp,
                                      c_vp, C.POINTER(c_vp), C.POINTER(c_i64), c_vp]),
    "dmm_host_neg_sampling": (C.c_int, [c_vp, c_vp, c_vp, c_i64, c_vp, c_i64, c_vp, c_vp]),
    "dmm_scatter_add_rows": (C.c_int, [c_vp, c_vp, c_i64, c_vp, c_i64, c_i64, c_vp, c_i64, c_vp]),
}

_lib = None
_lock = threading.Lock()
_ctx = {}          # device index -> dmm_ctx*
launch_count = 0   # kernels-launching C-ABI calls made by this process (bench.py's gpu_launches evidence)


class DiffMMError(RuntimeError):
    pass


def load():
    """Loads the shared library (no CUDA call is made). Raises if it has not been built."""
    global _lib
    with _lock:
        if _lib is not None:
            return _lib
        if not os.path.isfile(LIB_PATH):
            raise DiffMMError(
                f"{LIB_PATH} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "(diffmm_b200 has no CPU / PyTorch fallback)")
        lib = C.CDLL(LIB_PATH)
        for name, (res, args) in PROTOTYPES.items():
            fn = getattr(lib, name)          # AttributeError if the symbol is not exported
            fn.restype = res
            fn.argtypes = args
        _lib = lib
        return _lib


def last_error() -> str:
    return (load().dmm_last_error() or b"").decode()


def check(status: int, what: str):
    if status != 0:
        raise DiffMMError(f"{what} failed with status {status}: {last_error()}")


def ctx(device_index: int):
    """Per-device context handle (created on first use)."""
    lib = load()
    h = _ctx.get(device_index)
    if h is None:
        out = c_vp()
        check(lib.dmm_init(int(device_index), C.byref(out)), "dmm_init")
        h = out
        _ctx[device_index] = h
    return h


def call(name: str, *args):
    global launch_count
    lib = load()
    launch_count += 1
    check(getattr(lib, name)(*args), name)
