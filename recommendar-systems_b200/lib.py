"""ctypes binding of libmmrec_b200.so (the C ABI declared in include/mmrec_b200.h).

There is no fallback: if the library is missing or a call fails, a RuntimeError is raised.
torch tensors cross the boundary as raw device pointers + sizes; kernels are enqueued on
torch's current CUDA stream so they compose with autograd, NCCL and CUDA-graph capture.
"""
from __future__ import annotations

import ctypes as C
import os

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libmmrec_b200.so")

_p, _i32, _i64, _f32, _sz = C.c_void_p, C.c_int32, C.c_int64, C.c_float, C.c_size_t

# name -> (restype, argtypes); must list every symbol of include/mmrec_b200.h
SIGNATURES = {
    "mmrec_abi_version": (C.c_int, []),
    "mmrec_last_error": (C.c_char_p, []),
    "mmrec_launch_count": (_i64, []),
    "mmrec_ui_adj_workspace_bytes": (_sz, [_i64, _i32, _i32]),
    "mmrec_ui_adj_build": (C.c_int, [_p, _p, _i64, _i32, _i32, _p, _i32, _i32, _p, _p, _p, _p, _p,
                                     _sz, _p]),
    "mmrec_csr_from_coo_workspace_bytes": (_sz, [_i64]),
    "mmrec_csr_from_coo": (C.c_int, [_p, _p, _p, _i64, _i32, _i32, _i32, _p, _p, _p, _p, _p, _sz,
                                     _p]),
    "mmrec_spmm_csr_f32": (C.c_int, [_p, _p, _p, _p, _i32, _p, _p, _p, _i32, _p, _i32, _p, _p, _p,
                                     _f32, _p, _p, _p, _p]),
    "mmrec_spmm_csr_ex_f32": (C.c_int, [_p, _p, _p, _p, _i32, _p, _p, _p, _i32, _p, _i32, _p, _p, _p,
                                        _f32, _p, _p, _p, _i32, _p]),
    "mmrec_spmm_csr_bf16_f32": (C.c_int, [_p, _p, _p, _p, _i32, _p, _p, _p, _i32, _p, _i32, _p, _p, _p, _p,
                                          _f32, _p, _p, _p, _i32, _p]),
    "mmrec_spmm_csr_multi_f32": (C.c_int, [_p, _i32, _i32, _p]),
    "mmrec_layergcn_cos_bwd_f32": (C.c_int, [_p, _p, _p, _p, _i32, _i32, _p, _p, _p]),
    "mmrec_bpr_fwd_f32": (C.c_int, [_p, _p, _i32, _p, _p, _p, _i32, _p, _p, _p, _p, _p]),
    "mmrec_bpr_bwd_f32": (C.c_int, [_p, _p, _i32, _p, _p, _p, _i32, _p, _p, _p, _p, _p]),
    "mmrec_lightgcn_loss_fwd_workspace_floats": (_sz, [_i32]),
    "mmrec_lightgcn_loss_fwd_f32": (C.c_int, [_p, _p, _p, _p, _i32, _p, _p, _p, _i32, _f32, _p, _p, _p, _p, _p]),
    "mmrec_lightgcn_loss_bwd_f32": (C.c_int, [_p, _p, _p, _p, _i32, _p, _p, _p, _i32, _p, _p, _p, _p, _p, _p, _p]),
    "mmrec_infonce_splits": (_i32, [_i32]),
    "mmrec_infonce_fwd_workspace_floats": (_sz, [_i32]),
    "mmrec_infonce_fwd_f32": (C.c_int, [_p, _p, _i32, _p, _i32, _f32, _p, _p, _p, _p, _p, _p, _p,
                                        _p]),
    "mmrec_infonce_bwd_f32": (C.c_int, [_p, _p, _p, _p, _i32, _p, _i32, _f32, _p, _i32, _p, _p, _p,
                                        _p, _p]),
    "mmrec_infonce_pair_supported": (C.c_int, [_i32]),
    "mmrec_infonce_pair_fwd_f32": (C.c_int, [_p, _p, _i32, _p, _i32, _f32, _p, _p, _p, _p, _p, _p, _p]),
    "mmrec_infonce_pair_bwd_f32": (C.c_int, [_p, _p, _p, _p, _i32, _p, _i32, _f32, _p, _i32, _p, _p, _p, _p, _p]),
    "mmrec_spectral_fwd_f32": (C.c_int, [_p, _p, _i32, _i32, _p, _p, _p, _i32, _p, _p, _p, _p, _p]),
    "mmrec_spectral_bwd_f32": (C.c_int, [_p, _p, _i32, _i32, _p, _p, _p, _i32, _p, _p, _p, _p, _p,
                                         _p, _p, _p, _p, _p, _p]),
    "mmrec_gemm_splits": (C.c_int, [_i32, _i32, _i32, _i32, _i32]),
    "mmrec_gemm_tf32x3_f32": (C.c_int, [_p, _i32, _p, _i32, _p, _p, _i32, _i32, _i32, _i32, _p, _p]),
    "mmrec_linear_act_tc_supported": (C.c_int, [_i32, _i32, _i32]),
    "mmrec_linear_act_tc_f32": (C.c_int, [_p, _p, _p, _p, _i32, _i32, _i32, _i32, _p]),
    "mmrec_act_bwd_f32": (C.c_int, [_p, _p, _i64, _i32, _p, _p]),
    "mmrec_activation_f32": (C.c_int, [_p, _i64, _i32, _p, _p]),
    "mmrec_dense_act_supported": (C.c_int, [_i32, _i32]),
    "mmrec_dense_act_bwd_workspace_bytes": (_sz, [_i32, _i32]),
    "mmrec_dense_act_fwd_f32": (C.c_int, [_p, _p, _p, _p, _i32, _i32, _i32, _i32, _p]),
    "mmrec_dense_act_bwd_f32": (C.c_int, [_p, _p, _p, _p, _p, _p, _p, _p, _i32, _i32, _i32, _i32, _p]),
    "mmrec_dense_act_batch_fwd_f32": (C.c_int, [_p, _p, _p, _p, _i32, _i32, _i32, _i32, _i32, _p]),
    "mmrec_dense_act_batch_bwd_f32": (C.c_int, [_p, _p, _p, _p, _p, _p, _p, _p, _i32, _i32, _i32, _i32, _i32, _p]),
    "mmrec_smore_side_supported": (C.c_int, [_i32]),
    "mmrec_smore_side_bwd_workspace_bytes": (_sz, [_i32, _i32]),
    "mmrec_smore_side_fwd_f32": (C.c_int, [_p, _p, _p, _p, _p, _p, _p, _p, _p, _p, _i32, _i32, _p]),
    "mmrec_smore_side_bwd_f32": (C.c_int, [_p, _p, _p, _p, _p, _p, _p, _p, _p, _p, _p, _p, _p, _p, _p, _p,
                                           _p, _i32, _i32, _p]),
    "mmrec_smore_side_fwd_drop_f32": (C.c_int, [_p, _p, _p, _p, _p, _p, _p, _p, _p, _p, _i32, _i32, _p]),
    "mmrec_smore_side_bwd_drop_f32": (C.c_int, [_p] * 17 + [_i32, _i32, _p]),
    "mmrec_smore_side_fwd_tc_workspace_bytes": (_sz, [_i32, _i32]),
    "mmrec_gather_batch_rows_f32": (C.c_int, [_p, _i32, _p, _p, _p, _i32, _i32, _i32, _p, _p, _p]),
    "mmrec_scatter_batch_rows_add_f32": (C.c_int, [_p, _i32, _p, _i32, _i32, _p, _p]),
    "mmrec_gather_batch_views_f32": (C.c_int, [_p, _p, _p, _i32, _p, _i32, _p, _p, _p, _p, _i32, _i32, _i32, _p, _p, _p, _p]),
    "mmrec_scatter_batch_views_add_f32": (C.c_int, [_p, _p, _p, _i32, _p, _i32, _p, _p, _p, _p, _i32, _i32, _i32, _p, _p, _p]),
    "mmrec_smore_side_fwd_tc_f32": (C.c_int, [_p] * 10 + [_i32, _i32, _p, _p]),
    "mmrec_dropout_mask_f32": (C.c_int, [_p, _i32, _i32, _i32, _p, _p]),
    "mmrec_smore_combine_fwd_drop_f32": (C.c_int, [_p] * 10 + [_i32, _i32, _p, _p, _p]),
    "mmrec_smore_combine_bwd_drop_f32": (C.c_int, [_p] * 11 + [_i32, _i32] + [_p] * 10),
    "mmrec_smore_combine_supported": (C.c_int, [_i32]),
    "mmrec_smore_combine_fwd_f32": (C.c_int, [_p] * 10 + [_i32, _i32, _p, _p, _p]),
    "mmrec_smore_combine_bwd_f32": (C.c_int, [_p] * 11 + [_i32, _i32] + [_p] * 10),
    "mmrec_mgcn_fuse_supported": (C.c_int, [_i32]),
    "mmrec_mgcn_fuse_bwd_blocks": (_i32, [_i32, _i32]),
    "mmrec_mgcn_fuse_fwd_f32": (C.c_int, [_p] * 8 + [_i32, _i32, _p, _p, _p, _p]),
    "mmrec_mgcn_fuse_bwd_f32": (C.c_int, [_p] * 10 + [_i32, _i32] + [_p] * 10),
    "mmrec_adam_step_f32": (C.c_int, [_p, _p, _p, _p, _p, _i32, _p, C.c_double, C.c_double, C.c_double,
                                      C.c_double, C.c_double, _p, _p, _i32, _p]),
    "mmrec_adam_tick": (C.c_int, [_p, _p]),
    "mmrec_mirror_coef_workspace_bytes": (_sz, [_p, _i32]),
    "mmrec_mirror_coef_f32": (C.c_int, [_p, _p, _p, _i32, _p, C.c_double, C.c_double, C.c_double, C.c_double,
                                        _p, _i32, _i32, _p, _p, _p]),
    "mmrec_table_lowrank_supported": (C.c_int, [_i32, _i32, _i32]),
    "mmrec_table_lowrank_workspace_bytes": (_sz, [_i32, _i32]),
    "mmrec_table_adam_lowrank_f32": (C.c_int, [_p, _p, _p, _p, _p, _i32, _i32, _i32, _p, C.c_double, C.c_double,
                                               C.c_double, C.c_double, C.c_double, _i32, _p, _p, _p]),
    "mmrec_table_lowrank_sumsq_f64": (C.c_int, [_p, _p, _i32, _i32, _i32, _p, _p, _p]),
    "mmrec_axpy_multi_f32": (C.c_int, [_p, _p, _p, _i32, _p, _f32, _p]),
    "mmrec_inject3_fwd_f32": (C.c_int, [_p, _p, _p, _p, _f32, _i64, _p, _p, _p, _p]),
    "mmrec_inject3_bwd_f32": (C.c_int, [_p, _p, _p, _f32, _i64, _p, _p, _p, _p, _p]),
    "mmrec_loss_head_fwd_f32": (C.c_int, [_p, _p, _f32, _f32, _f32, _f32, _p, _p]),
    "mmrec_loss_head_bwd_f32": (C.c_int, [_p, _f32, _f32, _f32, _f32, _p, _p, _p]),
    "mmrec_colsum_f32": (C.c_int, [_p, _i32, _i32, _p, _p]),
    "mmrec_colsum_workspace_bytes": (_sz, [_i32, _i32]),
    "mmrec_colsum_ws_f32": (C.c_int, [_p, _i32, _i32, _p, _p, _p]),
    "mmrec_row_normalize_f32": (C.c_int, [_p, _i32, _i32, _p, _p]),
    "mmrec_row_topk_f32": (C.c_int, [_p, _i32, _i32, _i64, _i32, _p, _p, _p]),
    "mmrec_knn_weights_f32": (C.c_int, [_p, _p, _i32, _i32, _i32, _p, _p, _p]),
    "mmrec_score_mask_topk_f32": (C.c_int, [_p, _p, _i32, _p, _i32, _i32, _i32, _p, _p, _i32, _i32,
                                            _p, _p, _p, _p, _p]),
    "mmrec_score_mask_topk_simt_f32": (C.c_int, [_p, _p, _i32, _p, _i32, _i32, _i32, _p, _p, _i32, _i32,
                                                 _p, _p, _p, _p, _p]),
    "mmrec_score_mask_topk_rows_f32": (C.c_int, [_p, _p, _i32, _p, _i32, _i32, _i32, _p, _p, _i32, _i32,
                                                 _p, _p, _p, _p, _p]),
    "mmrec_topk_metrics_workspace_bytes": (_sz, [_i32]),
    "mmrec_topk_metrics_f64": (C.c_int, [_p, _i32, _i32, _p, _p, _p, _p, _p, _p, _p, _p]),
    "mmrec_topk_merge": (C.c_int, [_p, _p, _i32, _i32, _i32, _p, _p, _p]),
    "mmrec_neg_sample_counter": (C.c_int, [_p, _i64, _p, _i64, _p, _p, C.c_uint64, C.c_uint64, _i32, _p, _p]),
    "mmrec_neg_sample_mt19937_host": (C.c_int, [_p, _p, _i64, _p, _p, _i64, _p, _i64, _p]),
}



class SpmmProblem(C.Structure):
    """MmrecSpmmProblem of include/mmrec_b200.h."""
    _fields_ = [("row_ptr", _p), ("col_idx", _p), ("vals", _p), ("tasks", _p), ("n_tasks", _i32),
                ("slot_base", _p), ("counters", _p), ("scratch", _p), ("col_offset", _i32), ("X", _p),
                ("Y", _p), ("acc_in", _p), ("acc_out", _p), ("acc_scale", _f32)]


class Dropout(C.Structure):
    """MmrecDropout of include/mmrec_b200.h: in-kernel nn.Dropout (no mask tensor)."""
    _fields_ = [("p", _f32), ("seed", C.c_uint64), ("counter", _p), ("row_ids", _p), ("n_total", _i32)]

    @classmethod
    def make(cls, p, seed, counter=None, row_ids=None, n_total=0):
        """`counter`: a 1-element float64 CUDA tensor read on the device (FusedAdam's update count) or None.
        `row_ids` (int64 CUDA tensor) / `n_total`: the call evaluates gathered rows of a dense [n_total, d]
        table and draws the multipliers of those rows (batch-row calls)."""
        if counter is not None and (counter.dtype != torch.float64 or not counter.is_cuda or counter.numel() < 1):
            raise RuntimeError("Dropout.counter must be a float64 CUDA tensor")
        if row_ids is not None and (row_ids.dtype != torch.int64 or not row_ids.is_cuda or not row_ids.is_contiguous()
                                    or int(n_total) <= 0):
            raise RuntimeError("Dropout.row_ids must be a contiguous int64 CUDA tensor with n_total > 0")
        return cls(float(p), int(seed) & 0xFFFFFFFFFFFFFFFF, ptr(counter), ptr(row_ids), int(n_total))


_lib = None


def load():
    """Load the shared library (once). Raises if it has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                f"{LIB_PATH} is missing: run `python -c 'import __graft_entry__ as g; g.build()'` "
                "(there is no CPU or PyTorch fallback for the hot path)")
        lib = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(lib, name)          # AttributeError if a declared symbol is absent
            fn.restype, fn.argtypes = res, args
        _lib = lib
    return _lib


def _check_device(t):
    """Kernels are enqueued on the CURRENT device's current stream (see `stream`): a tensor that
    lives on another GPU would be dereferenced by the wrong device, so that is an error here
    (torch ops switch devices by themselves; this library asks the caller to
    `torch.cuda.set_device` / `with torch.cuda.device(...)` first). A host tensor is an error too: its
    address would reach a kernel as a device pointer."""
    if not t.is_cuda:
        raise RuntimeError("mmrec_b200 operators need CUDA tensors; there is no CPU fallback")
    if t.device.index != torch.cuda.current_device():
        raise RuntimeError(f"mmrec_b200: tensor on {t.device} but the current CUDA device is "
                           f"cuda:{torch.cuda.current_device()}; wrap the call in torch.cuda.device(tensor.device)")


def ptr(t):
    """Device pointer of a tensor (None -> NULL); the tensor must live on the current device."""
    if t is None:
        return None
    _check_device(t)
    return t.data_ptr()


def ptr_array(tensors):
    """void*[n] of device pointers (None -> NULL) for the batched entry points."""
    for t in tensors:
        if t is not None:
            _check_device(t)
    return (C.c_void_p * len(tensors))(*[None if t is None else t.data_ptr() for t in tensors])


def stream():
    return torch.cuda.current_stream().cuda_stream


def call(name, *args):
    lib = load()
    rc = getattr(lib, name)(*args)
    if rc != 0:
        msg = lib.mmrec_last_error().decode(errors="replace")
        raise RuntimeError(f"{name} failed with code {rc}: {msg}")


def launch_count() -> int:
    return int(load().mmrec_launch_count())


def require_cuda(*tensors):
    for t in tensors:
        if t is not None and not t.is_cuda:
            raise RuntimeError("mmrec_b200 operators need CUDA tensors; there is no CPU fallback")
