"""ctypes binding of the C ABI declared in include/uml_b200.h.

The library is looked up in-tree (``lib/libuml_b200.so``, built by ``build.py``).  A missing
library is a hard error - the product path never falls back to PyTorch or the CPU."""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("UML_LIB_PATH") or os.path.join(_HERE, "lib", "libuml_b200.so")  # override: A/B builds

c_i32, c_i64, c_f32, c_f64, c_vp = C.c_int32, C.c_int64, C.c_float, C.c_double, C.c_void_p


class Segment(C.Structure):
    """uml_segment"""
    _fields_ = [("rows", c_vp), ("idx", c_vp), ("labels", c_vp), ("n", c_i64), ("ld", c_i64),
                ("scale", c_f32), ("loss_weight", c_f32), ("label_idx", c_vp), ("scale_dev", c_vp), ("rows16", c_vp)]


class SegStats(C.Structure):
    """uml_seg_stats"""
    _fields_ = [("loss_mean", c_f32), ("dscale", c_f32), ("correct", c_i32), ("n", c_i32)]


class Update(C.Structure):
    """uml_update"""
    _fields_ = [("kind", c_i32), ("lr", c_f32), ("beta1", c_f32), ("beta2", c_f32), ("eps", c_f32),
                ("weight_decay", c_f32), ("momentum", c_f32), ("step", c_i64), ("m", c_vp), ("v", c_vp)]


class TcSegments(C.Structure):
    """uml_tc_segments"""
    _fields_ = [("seg_rows", c_i64 * 2), ("scale", c_f32 * 2), ("loss_weight", c_f32 * 2), ("nseg", c_i32),
                ("scale_dev", c_vp * 2)]


class LinearStepArgs(C.Structure):
    """uml_linear_step_args"""
    _fields_ = [("dim", c_i32), ("n_classes", c_i32), ("nseg", c_i32), ("precision", c_i32),
                ("seg", Segment * 2), ("W", c_vp), ("upd", Update), ("G", c_vp), ("ldg", c_i64),
                ("row_loss", c_vp), ("row_correct", c_vp), ("row_dscale", c_vp), ("stats", c_vp),
                ("X16", c_vp), ("W16", c_vp), ("labels32", c_vp), ("partials", c_vp), ("tile_ws", c_vp),
                ("max_splits", c_i32), ("w16_valid", c_i32), ("dW_out", c_vp), ("dW_scratch", c_vp),
                ("scale_param", c_vp * 2), ("scale_m", c_vp * 2), ("scale_v", c_vp * 2), ("scale_step", c_i64 * 2),
                ("ev", c_vp * 8), ("dp_allreduce", c_i32), ("X16_alt", c_vp), ("labels32_alt", c_vp), ("g_capacity_rows", c_i64),
                ("X16_alt2", c_vp), ("labels32_alt2", c_vp), ("idx_ready", c_vp)]


class RunStep(C.Structure):
    """uml_run_step"""
    _fields_ = [("idx", c_vp * 2), ("n", c_i64 * 2), ("loss_weight", c_f32 * 2), ("lr", c_f32), ("opt_step", c_i64),
                ("scale_step", c_i64 * 2), ("stats", c_vp), ("ev", c_vp * 8)]


SWEEP_MAX_HEADS = 32


class SweepArgs(C.Structure):
    """uml_sweep_args"""
    _fields_ = [("n_heads", c_i32), ("dim", c_i32), ("n_classes", c_i32), ("kind", c_i32),
                ("bank", c_vp * 2), ("bank_ld", c_i64 * 2), ("labels", c_vp * 2),
                ("perm", (c_vp * SWEEP_MAX_HEADS) * 2), ("perm_len", c_i64 * 2), ("pos", c_i64 * 2),
                ("scale", c_f32 * 2), ("W", c_vp), ("m", c_vp), ("v", c_vp), ("head_stride", c_i64),
                ("G", c_vp), ("ldg", c_i64), ("max_rows", c_i64), ("row_loss", c_vp), ("row_correct", c_vp),
                ("stats", c_vp), ("beta1", c_f32), ("beta2", c_f32), ("eps", c_f32), ("momentum", c_f32),
                ("step", c_i64), ("weight_decay", c_f32 * SWEEP_MAX_HEADS), ("alpha", c_f32 * SWEEP_MAX_HEADS),
                ("active", C.c_uint8 * SWEEP_MAX_HEADS), ("ev", c_vp * 8)]


class SweepAdapterArgs(C.Structure):
    """uml_sweep_adapter_args"""
    _fields_ = [("img_dim", c_i32), ("W", c_vp), ("m", c_vp), ("v", c_vp), ("adapter_stride", c_i64), ("Z", c_vp),
                ("dZ", c_vp), ("ldz", c_i64), ("max_img_rows", c_i64), ("scale_param", c_vp), ("scale_m", c_vp),
                ("scale_v", c_vp), ("row_dscale", c_vp), ("ev", c_vp * 10)]


# name -> argtypes; every function returns int except uml_last_error
PROTOTYPES = {
    "uml_abi_version": [],
    "uml_device_ok": [c_i32],
    "uml_gather_rows_f32": [c_vp, c_i64, c_i32, c_vp, c_i64, c_vp, c_vp],
    "uml_gather_rows_bf16": [c_vp, c_i64, c_i32, c_vp, c_i64, c_vp, c_i64, c_vp],
    "uml_gather_rows_labels_bf16": [c_vp, c_vp, c_i32, c_vp, c_i64, c_vp, c_i64, c_vp, c_vp],
    "uml_gather_labels_i32": [c_vp, c_vp, c_i64, c_vp, c_vp],
    "uml_gather2_rows_bf16": [c_vp, c_vp, c_vp, c_i64, c_vp, c_vp, c_vp, c_i64, c_i32, c_vp, c_i64, c_vp, c_vp],
    "uml_gather2_rows_bf16_light": [c_vp, c_vp, c_vp, c_i64, c_vp, c_vp, c_vp, c_i64, c_i32, c_vp, c_i64, c_vp, c_vp],
    "uml_cast_f32_to_bf16": [c_vp, c_vp, c_i64, c_vp],
    "uml_head_fwd_ce_f32": [C.POINTER(Segment), c_i32, c_i32, c_vp, c_i32, c_vp, c_i64, c_vp, c_vp, c_vp, c_vp, c_i64, c_vp],
    "uml_head_bwd_dw_f32": [C.POINTER(Segment), c_i32, c_i32, c_vp, c_i64, c_i32, c_vp, c_vp, C.POINTER(Update), c_vp],
    "uml_head_step_fused_count": [],
    "uml_sweep_launch_count": [],
    "uml_head_step_fused_f32": [C.POINTER(Segment), c_i32, c_i32, c_vp, c_i32, c_vp, c_i64, c_vp, c_vp, c_vp, c_vp,
                                C.POINTER(Update), C.POINTER(c_i32), c_vp],
    "uml_gemm_nt_f32": [c_vp, c_i64, c_vp, c_vp, c_i64, c_vp, c_i64, c_i64, c_i64, c_i64, c_f32, c_vp],
    "uml_gemm_nn_f32": [c_vp, c_i64, c_vp, c_i64, c_vp, c_i64, c_i64, c_i64, c_i64, c_f32, c_vp],
    "uml_gemm_tn_f32": [c_vp, c_i64, c_vp, c_i64, c_vp, c_vp, c_i64, c_i64, c_i64, c_i64, c_f32, c_vp,
                        C.POINTER(Update), c_vp],
    "uml_adamw_step": [c_vp, c_vp, c_vp, c_f32, c_vp, c_vp, c_i64, c_f64, c_f64, c_f64, c_f64, c_f64, c_i64, c_i32,
                       c_vp, c_vp],
    "uml_sgd_step": [c_vp, c_vp, c_vp, c_f32, c_vp, c_i64, c_f64, c_f64, c_f64, c_i64, c_vp, c_vp],
    "uml_eval_f32": [c_vp, c_i64, c_vp, c_i64, c_i32, c_vp, c_i32, c_f32, c_vp, c_vp, c_vp],
    "uml_eval_reduce": [c_vp, c_vp, c_vp, c_i64, c_i64, c_vp, c_vp, c_vp],
    "uml_cka_workspace_doubles": [c_i32, c_i32],
    "uml_cka_linear_f32": [c_vp, c_i64, c_i32, c_vp, c_i64, c_i32, c_i64, c_vp, c_vp, c_vp],
    "uml_mutual_knn_f32": [c_vp, c_i64, c_i32, c_vp, c_i64, c_i32, c_i64, c_i32, c_vp, c_vp, c_vp],
    "uml_gauss_embed": [c_vp, c_i32, c_i32, c_i32, c_vp, c_vp, c_i64, c_vp, c_vp, c_vp],
    "uml_eval_group_f32": [c_vp, c_i64, c_vp, c_i64, c_i32, c_vp, c_i64, c_vp, c_vp, c_i32, c_i32, c_vp, c_vp, c_vp],
    "uml_eval_reduce_group": [c_vp, c_vp, c_vp, c_i64, c_i64, c_i32, c_vp, c_vp, c_vp],
    "uml_grad_diag": [c_vp, c_vp, c_i64, c_vp, c_vp, c_vp],
    "uml_head_fwd_ce_bf16": [c_vp, c_i64, c_i32, c_vp, c_i32, c_vp, C.POINTER(TcSegments), c_vp, c_i64, c_vp, c_vp,
                             c_vp, c_vp, c_vp, c_vp, c_vp],
    "uml_head_bwd_dw_bf16": [c_vp, c_i64, c_vp, c_i64, c_i32, c_i32, c_vp, c_i32, c_vp],
    "uml_head_fwd_ce_deferred_bf16": [c_vp, c_i64, c_i32, c_vp, c_i32, c_vp, C.POINTER(TcSegments), c_vp, c_i64, c_vp, c_vp],
    "uml_head_bwd_dw_fix_bf16": [c_vp, c_i64, c_vp, c_i64, c_i32, c_i32, c_vp, c_i32, C.POINTER(TcSegments), c_vp, c_vp, c_vp,
                                 c_vp],
    "uml_tc_dw_splits": [c_i64, c_i32, c_i32],
    "uml_gemm_bf16": [c_vp, c_i64, c_i32, c_vp, c_i64, c_i32, c_i64, c_i64, c_i64, c_vp, c_i64, c_i32, c_i32, c_vp],
    "uml_gemm_bf16_splits": [c_i64, c_i64, c_i64],
    "uml_adamw_step_partials": [c_vp, c_vp, c_i32, c_i64, c_vp, c_vp, c_i64, c_f64, c_f64, c_f64, c_f64, c_f64, c_i64,
                                c_i32, c_vp, c_vp, c_vp],
    "uml_sum_partials": [c_vp, c_i32, c_i64, c_i64, c_vp, c_vp],
    "uml_reduce_seg_stats": [c_vp, c_vp, c_vp, C.POINTER(c_i64), c_i32, c_vp, c_vp],
    "uml_reduce_tile_stats": [c_vp, c_i64, c_i32, c_vp, c_vp],
    "uml_fwd_x_failed": [c_vp],
    "uml_linear_step": [C.POINTER(LinearStepArgs), c_vp],
    "uml_linear_run_reset": [],
    "uml_linear_run": [C.POINTER(LinearStepArgs), C.POINTER(RunStep), c_i32, c_vp],
    "uml_dp_unique_id": [c_vp],
    "uml_dp_init": [c_vp, c_i32, c_i32],
    "uml_dp_allreduce_f32": [c_vp, c_i64, c_vp],
    "uml_dp_shutdown": [],
    "uml_dp_p2p_alloc": [c_i64, c_vp],
    "uml_dp_p2p_open": [c_vp, c_i32, c_i32],
    "uml_dp_allreduce_p2p": [c_i64, c_vp],
    "uml_dp_fused_adam_update": [c_vp, c_i32, c_i64, c_i64, c_vp, c_vp, c_vp, c_f64, c_f64, c_f64, c_f64, c_f64, c_i64, c_i32,
                                 c_vp, c_vp],
    "uml_dp_p2p_failed": [],
    "uml_dp_p2p_close_peers": [],
    "uml_gauss_param_count": [c_i32, c_i32, c_i32],
    "uml_gauss_workspace_floats": [c_i32, c_i32, c_i32, c_i64],
    "uml_gauss_step": [c_vp, c_vp, c_vp, c_i32, c_i32, c_i32, c_vp, c_i64, c_vp, c_i64, c_vp, c_i64, c_i32, c_f32, c_f32,
                       c_f64, c_f64, c_f64, c_f64, c_i64, c_vp, c_vp, c_vp],
    "uml_gauss_run": [c_vp, c_vp, c_vp, c_i32, c_i32, c_i32, c_vp, c_i64, c_vp, c_i64, c_vp, c_i32, c_i64, c_i32, c_f32, c_f32,
                      c_f64, c_f64, c_f64, c_f64, c_i64, c_vp, c_vp, c_vp],
    "uml_gauss_eval": [c_vp, c_i32, c_i32, c_i32, c_vp, c_vp, c_i64, c_vp, c_vp, c_vp],
    "uml_sweep_run": [C.POINTER(SweepArgs), c_i32, c_vp, c_vp, c_vp],
    "uml_sweep_adapter_run": [C.POINTER(SweepArgs), C.POINTER(SweepAdapterArgs), c_i32, c_vp, c_vp, c_vp],
    "uml_randperm_i64": [C.c_uint64, c_i64, c_vp],
    "uml_randperm_begin": [c_vp, C.c_uint64, c_i64, c_vp],
    "uml_randperm_advance": [c_vp, c_i64],
    "uml_randperm_run": [c_vp, C.c_uint64, c_i64, c_vp, c_i64, c_i32, c_vp],
    "uml_randperm_next_filled": [c_vp],
    "uml_randperm_wait": [c_vp, c_i64],
}

_lib = None

# kernels launched per C-ABI call (bench.py reports the sum as "gpu_launches")
KERNELS_PER_CALL = {
    "uml_gather_rows_f32": 1, "uml_gather_rows_bf16": 1, "uml_gather_labels_i32": 1, "uml_cast_f32_to_bf16": 1,
    "uml_gather_rows_labels_bf16": 1, "uml_gather2_rows_bf16": 1, "uml_gather2_rows_bf16_light": 1, "uml_gauss_step": 2, "uml_gauss_eval": 2, "uml_head_fwd_ce_deferred_bf16": 1, "uml_head_bwd_dw_fix_bf16": 1,
    "uml_head_fwd_ce_f32": 3, "uml_head_bwd_dw_f32": 1, "uml_gemm_nt_f32": 1, "uml_gemm_nn_f32": 1,
    "uml_gemm_tn_f32": 1, "uml_adamw_step": 1, "uml_sgd_step": 1, "uml_eval_f32": 1, "uml_eval_reduce": 1, "uml_eval_group_f32": 1, "uml_eval_reduce_group": 1, "uml_cka_linear_f32": 3, "uml_mutual_knn_f32": 4, "uml_gauss_embed": 1,
    "uml_grad_diag": 2, "uml_head_fwd_ce_bf16": 2, "uml_reduce_tile_stats": 1, "uml_head_bwd_dw_bf16": 1, "uml_gemm_bf16": 1, "uml_adamw_step_partials": 1,
    "uml_sum_partials": 1, "uml_reduce_seg_stats": 1,
}  # uml_linear_step is counted by the caller (its kernel count depends on the path)
LAUNCH_COUNT = [0]


class _Counted:
    """Wraps a ctypes function so every successful call adds its kernel count to LAUNCH_COUNT."""

    def __init__(self, fn, n):
        self.fn, self.n = fn, n

    def __call__(self, *a):
        r = self.fn(*a)
        LAUNCH_COUNT[0] += self.n
        return r


class UmlLibraryError(RuntimeError):
    pass


def load() -> C.CDLL:
    """Load libuml_b200.so once and attach prototypes.  Raises if it is absent."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise UmlLibraryError(
            f"{LIB_PATH} not found - build it with `python unpaired-multimodal-learning_b200/build.py` "
            "(or __graft_entry__.build()).  There is no CPU/PyTorch fallback for the UML hot path.")
    lib = C.CDLL(LIB_PATH)
    lib.uml_last_error.restype = C.c_char_p
    lib.uml_last_error.argtypes = []
    for name, args in PROTOTYPES.items():
        fn = getattr(lib, name)  # AttributeError here means header and library disagree
        fn.restype = c_i32
        fn.argtypes = args
        if name in KERNELS_PER_CALL:
            setattr(lib, name, _Counted(fn, KERNELS_PER_CALL[name]))
    if lib.uml_abi_version() != 1:
        raise UmlLibraryError("libuml_b200.so ABI version mismatch")
    _lib = lib
    return lib


def check(status: int):
    if status != 0:
        msg = load().uml_last_error().decode("utf-8", "replace")
        raise RuntimeError(f"libuml_b200: {msg} (status {status})")
