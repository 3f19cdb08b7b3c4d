"""ctypes bindings to ``_lib/libdtf_kernels.so`` (hand-written sm_100a kernels, plain C ABI).

The library is built in-tree by ``python __graft_entry__.py build`` (explicit
``nvcc -gencode arch=compute_100a,code=sm_100a``).  On a machine with a CUDA
device the library MUST load: every entry point here raises if it is missing,
there is no silent eager fallback (DESIGN.md "no compatibility layers").
"""
from __future__ import annotations

import contextlib
import ctypes
import os
import threading
from ctypes import (POINTER, Structure, byref, c_float, c_int, c_longlong, c_uint, c_ulonglong, c_void_p)
from typing import Optional, Sequence, Tuple

import torch

MAX_WORKERS = 16
_LIB: Optional[ctypes.CDLL] = None
_LOCK = threading.Lock()


def lib_path() -> str:
    here = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    return os.path.join(here, "_lib", "libdtf_kernels.so")


class GemmArgs(Structure):
    _fields_ = [("a", c_void_p), ("b", c_void_p), ("c", c_void_p),
                ("M", c_longlong), ("N", c_longlong), ("K", c_longlong),
                ("lda", c_longlong), ("ldb", c_longlong), ("ldc", c_longlong),
                ("a_mn", c_int), ("b_mn", c_int), ("c_bf16", c_int),
                ("bias", c_void_p), ("relu", c_int),
                ("mask", c_void_p), ("ldmask", c_longlong),
                ("alpha", c_float), ("splits", c_int), ("accumulate", c_int),
                ("colsum", c_void_p),
                ("wait_flag", c_void_p), ("wait_target", c_ulonglong),
                ("signal", c_void_p), ("err", c_void_p), ("timeout_ns", c_ulonglong),
                ("block_n_override", c_int), ("wait_target_ptr", c_void_p), ("phase_trace", c_void_p),
                ("signal_gpu_scope", c_int), ("stamp_src", c_void_p), ("stamp_dst", c_void_p), ("persistent", c_int), ("cta_pair", c_int),
                ("tf32", c_int),
                ("conv", c_int), ("cv_n", c_int), ("cv_h", c_int), ("cv_w", c_int), ("cv_c", c_int), ("cv_kh", c_int),
                ("cv_kw", c_int), ("cv_pt", c_int), ("cv_pl", c_int)]


class PsApplyArgs(Structure):
    _fields_ = [("ctl", c_void_p), ("master", c_void_p), ("slot_m", c_void_p), ("slot_v", c_void_p),
                ("grad", c_void_p * MAX_WORKERS), ("shadow", c_void_p),
                ("replica", c_void_p * MAX_WORKERS), ("mailbox", c_void_p * MAX_WORKERS),
                ("n", c_longlong), ("num_workers", c_int), ("replicas_to_aggregate", c_int),
                ("ctas_per_push", c_uint), ("mode", c_int), ("kind", c_int),
                ("lr", c_float), ("momentum", c_float), ("beta1", c_float), ("beta2", c_float), ("eps", c_float),
                ("nesterov", c_int), ("publish_replicas", c_int),
                ("zero_begin", c_longlong * 4), ("zero_end", c_longlong * 4), ("num_zero", c_int),
                ("timeout_ns", c_ulonglong), ("trace", c_void_p), ("trace_cap", c_int), ("grid", c_int),
                ("system_scope", c_int), ("phase_trace", c_void_p), ("idle_ok", c_int),
                ("grad_mc", c_void_p), ("shadow_mc", c_void_p), ("master_mc", c_void_p), ("token_mc", c_void_p)]


class MlpHeadArgs(Structure):
    _fields_ = [("h", c_void_p), ("ldh", c_longlong), ("w2", c_void_p), ("ldw2", c_longlong),
                ("b2", c_void_p), ("labels", c_void_p), ("ldl", c_longlong),
                ("B", c_int), ("H", c_int), ("C", c_int), ("clip_min", c_float),
                ("loss_out", c_void_p), ("loss_hist", c_void_p), ("step_counter", c_void_p), ("hist_cap", c_int),
                ("dh", c_void_p), ("lddh", c_longlong), ("gw2", c_void_p), ("ldgw2", c_longlong),
                ("gb2", c_void_p), ("gb1", c_void_p), ("logits_out", c_void_p),
                ("mailbox", c_void_p), ("ctl", c_void_p), ("rank", c_int), ("stamp_from_version", c_int),
                ("phase_trace", c_void_p), ("h_acc", c_void_p), ("ld_acc", c_longlong), ("b1", c_void_p),
                ("sys_scope", c_int), ("ctas", c_int)]


class MlpStepArgs(Structure):
    """``csrc/mlp_step.cu: DtfMlpStepArgs`` -- one whole worker step of the MLP as one kernel (fp32 storage, TF32 MMAs)."""
    _fields_ = [("B", c_int), ("D", c_int), ("H", c_int), ("C", c_int), ("G", c_int), ("phase_mask", c_int),
                ("x", c_void_p), ("ldx", c_longlong), ("x_rows", c_longlong),
                ("labels", c_void_p), ("ldl", c_longlong),
                ("nbatches", c_longlong), ("bstride", c_longlong), ("boffset", c_longlong),
                ("w1", c_void_p), ("ldw1", c_longlong), ("b1", c_void_p), ("w2", c_void_p), ("ldw2", c_longlong),
                ("b2", c_void_p),
                ("hpart", c_void_p), ("dh", c_void_p), ("lddh", c_longlong), ("flags", c_void_p),
                ("gw1", c_void_p), ("ldgw1", c_longlong), ("gb1", c_void_p), ("gw2", c_void_p), ("ldgw2", c_longlong),
                ("gb2", c_void_p),
                ("clip_min", c_float), ("loss_out", c_void_p), ("logits_out", c_void_p), ("step_counter", c_void_p),
                ("forward_only", c_int), ("num_tokens", c_int), ("token", c_void_p * 4), ("token_scale", c_ulonglong * 4),
                ("token_base", c_ulonglong * 4), ("stamp_step", c_int), ("consumed", c_void_p * 4),
                ("num_signals", c_int), ("arrivals", c_void_p * 4), ("stamp_dst", c_void_p * 4), ("stamp_src", c_void_p * 4),
                ("sys_scope", c_int), ("timeout_ns", c_ulonglong), ("err", c_void_p), ("trace", c_void_p),
                ("no_cluster", c_int), ("dbg", c_int), ("ring", c_void_p), ("ring_cap", c_int),
                ("head_part", c_void_p)]


class StepOp(Structure):
    """One entry of a native step plan (``csrc/step_exec.cu``: ``DtfStepOp``)."""
    _fields_ = [("kind", c_int), ("is_kernel", c_int), ("p0", c_void_p), ("p1", c_void_p), ("p2", c_void_p),
                ("p3", c_void_p), ("p4", c_void_p), ("i0", c_longlong), ("i1", c_longlong), ("i2", c_longlong),
                ("i3", c_longlong), ("i4", c_longlong), ("i5", c_longlong), ("u0", c_ulonglong)]


class LoopArgs(Structure):
    """``csrc/step_exec.cu: DtfLoopArgs`` -- ``steps`` end-to-end training steps of one local worker in ONE native call
    (per step: H2D of that step's pinned batch one step ahead, the step's plan, the ps shard's plan, D2H of the loss row)."""
    _fields_ = [("device", c_int), ("steps", c_int), ("depth", c_int), ("parity", c_int), ("prefetched", c_int),
                ("prefetch_next", c_int), ("x_op", c_int), ("y_op", c_int), ("n_copy", c_int * 2), ("n_compute", c_int * 2), ("n_ps", c_int),
                ("copy_ops", c_void_p * 2), ("compute_ops", c_void_p * 2), ("ps_ops", c_void_p),
                ("copy_stream", c_void_p), ("stream", c_void_p), ("ps_stream", c_void_p),
                ("x_base", c_void_p), ("y_base", c_void_p), ("x_stride", c_longlong), ("y_stride", c_longlong),
                ("nbatches", c_longlong), ("first", c_longlong), ("batch_step", c_longlong),
                ("loss_src", c_void_p), ("loss_bytes", c_longlong), ("loss_host", c_void_p), ("loss_row_bytes", c_longlong),
                ("kernels", c_longlong), ("waited", c_longlong)]


OP_H2D, OP_D2H, OP_CONVERT, OP_GEMM, OP_HEAD, OP_PS_APPLY, OP_WAIT_TOKEN, OP_SIGNAL, OP_STAGE, OP_SYNC = range(1, 11)
OP_GRAPH = 13
OP_MLP_STEP = 14
_KERNEL_OPS = (OP_CONVERT, OP_GEMM, OP_HEAD, OP_PS_APPLY, OP_WAIT_TOKEN, OP_SIGNAL, OP_STAGE, OP_MLP_STEP)


class StepPlan:
    """A fixed op sequence executed by ONE native call (memcpys, kernel launches, optional stream sync)."""

    def __init__(self, ops: Sequence[StepOp], device: int, stream: int, keep=()):
        self.n = len(ops)
        self.ops = (StepOp * self.n)(*ops)
        self.device, self.stream = int(device), stream
        self.keep = list(keep)            # objects whose memory the ops point into
        self._kernels = c_int(0)

    def run(self) -> int:
        self._kernels.value = 0
        rc = load().dtf_run_ops(self.ops, self.n, self.device, self.stream, byref(self._kernels))
        if rc:
            raise RuntimeError("native step plan failed at op %d (kind %d) with code %d" % (
                rc // 100000 - 1, self.ops[rc // 100000 - 1].kind, rc % 100000))
        _bump(self._kernels.value)
        return self._kernels.value

    def graphed(self) -> "StepPlan":
        """Same plan with every maximal run of kernel ops replaced by ONE CUDA-graph launch.  Call after the plan
        has run eagerly at least once (first-launch attribute setup cannot be captured)."""
        lib = load()
        out, i, keep = [], 0, list(self.keep) + [self]
        while i < self.n:
            if self.ops[i].kind not in _KERNEL_OPS:
                out.append(self.ops[i])
                i += 1
                continue
            j = i
            while j < self.n and self.ops[j].kind in _KERNEL_OPS:
                j += 1
            sub = (StepOp * (j - i))(*[self.ops[k] for k in range(i, j)])
            ex, nk = c_void_p(), c_int(0)
            rc = lib.dtf_capture_ops(sub, j - i, self.device, self.stream, byref(ex), byref(nk))
            if rc or not ex.value:
                raise RuntimeError("CUDA-graph capture of ops [%d, %d) failed with code %d" % (i, j, rc))
            out.append(StepOp(kind=OP_GRAPH, p0=ex.value, i0=nk.value))
            keep.append(sub)
            i = j
        return StepPlan(out, self.device, self.stream, keep=keep)


def available() -> bool:
    return os.path.exists(lib_path())


class _Missing:
    """Stand-in for an entry point the loaded library does not have (the emulation build has no tcgen05 GEMM, VMM, step
    executor): declaring its signature is a no-op, calling it is an error."""

    def __call__(self, *a, **k):
        raise RuntimeError("this entry point is not part of the loaded kernel library (kernel-emulation build?)")


class _Tolerant:
    def __init__(self, lib):
        object.__setattr__(self, "_lib", lib)

    def __getattr__(self, name):
        try:
            return getattr(object.__getattribute__(self, "_lib"), name)
        except AttributeError:
            return _Missing()


def _declare(lib) -> None:
    """argtypes / restype of every entry point (``lib``: the CDLL, or a ``_Tolerant`` view of a partial library)."""
    lib.dtf_gemm_bf16.argtypes = [POINTER(GemmArgs), c_void_p]
    lib.dtf_gemm_bf16.restype = c_int
    lib.dtf_ps_apply.argtypes = [POINTER(PsApplyArgs), c_void_p]
    lib.dtf_ps_apply.restype = c_int
    if not isinstance(getattr(lib, "dtf_ps_apply_grid", _Missing()), _Missing):
        lib.dtf_ps_apply_grid.argtypes = [c_longlong]
        lib.dtf_ps_apply_grid.restype = c_int
    lib.dtf_mlp_head.argtypes = [POINTER(MlpHeadArgs), c_void_p]
    lib.dtf_mlp_head.restype = c_int
    lib.dtf_convert_f32_bf16.argtypes = [c_void_p, c_longlong, c_void_p, c_longlong, c_longlong, c_longlong,
                                         c_longlong, c_void_p]
    lib.dtf_convert_u8_bf16.argtypes = [c_void_p, c_void_p, c_longlong, c_float, c_void_p]
    lib.dtf_softmax_xent.argtypes = [c_void_p, c_longlong, c_void_p, c_longlong, c_int, c_int, c_float, c_void_p,
                                     c_void_p, c_void_p, c_longlong, c_void_p, c_longlong, c_int, c_void_p,
                                     c_longlong, c_float, c_void_p]
    lib.dtf_relu_grad.argtypes = [c_void_p, c_void_p, c_void_p, c_longlong, c_void_p]
    lib.dtf_colsum.argtypes = [c_void_p, c_longlong, c_int, c_int, c_void_p, c_void_p]
    lib.dtf_argmax_rows.argtypes = [c_void_p, c_longlong, c_int, c_int, c_void_p, c_void_p]
    lib.dtf_mean_of_n.argtypes = [c_void_p, c_int, c_void_p, c_longlong, c_void_p]
    lib.dtf_optimizer_apply.argtypes = [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_longlong, c_int, c_float,
                                        c_float, c_int, c_float, c_float, c_float, c_float, c_void_p]
    lib.dtf_im2col_nhwc.argtypes = [c_void_p, c_void_p] + [c_int] * 12 + [c_longlong, c_void_p]
    lib.dtf_col2im_nhwc.argtypes = [c_void_p, c_longlong, c_void_p] + [c_int] * 12 + [c_void_p]
    lib.dtf_gemm_ref.argtypes = [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_longlong, c_longlong,
                                 c_longlong, c_int, c_int, c_void_p, c_int, c_float, c_void_p]
    lib.dtf_ps_publish.argtypes = [c_void_p, c_void_p, c_longlong, c_void_p]
    lib.dtf_wait_token.argtypes = [c_void_p, c_ulonglong, c_void_p, c_ulonglong, c_void_p, c_void_p]
    lib.dtf_stage_from_dataset.argtypes = [c_void_p, c_void_p, c_longlong, c_int, c_int, c_int, c_longlong, c_longlong,
                                           c_void_p, c_void_p, c_void_p, c_void_p]
    lib.dtf_stage_from_dataset.restype = c_int
    lib.dtf_push_grad.argtypes = [c_void_p, c_void_p, c_longlong, c_void_p, c_void_p, c_int, c_int, c_int, c_int,
                                  c_void_p]
    lib.dtf_pull_shadow.argtypes = [c_void_p, c_void_p, c_longlong, c_int, c_void_p]
    lib.dtf_fabric_alloc.argtypes = [POINTER(c_void_p), c_longlong]
    lib.dtf_fabric_free.argtypes = [c_void_p]
    lib.dtf_fabric_export.argtypes = [c_void_p, c_void_p]
    lib.dtf_fabric_import.argtypes = [c_void_p, POINTER(c_void_p)]
    lib.dtf_fabric_close.argtypes = [c_void_p]
    lib.dtf_enable_peer.argtypes = [c_int]
    lib.dtf_can_access_peer.argtypes = [c_int, c_int]
    lib.dtf_memcpy_d2h.argtypes = [c_void_p, c_void_p, c_longlong]
    lib.dtf_memcpy_h2d.argtypes = [c_void_p, c_void_p, c_longlong]
    lib.dtf_memset.argtypes = [c_void_p, c_int, c_longlong, c_void_p]
    for name in ("dtf_convert_f32_bf16", "dtf_convert_u8_bf16", "dtf_softmax_xent", "dtf_relu_grad", "dtf_colsum",
                 "dtf_argmax_rows", "dtf_mean_of_n", "dtf_optimizer_apply", "dtf_im2col_nhwc", "dtf_col2im_nhwc",
                 "dtf_gemm_ref", "dtf_ps_publish", "dtf_wait_token", "dtf_push_grad", "dtf_pull_shadow",
                 "dtf_fabric_alloc", "dtf_fabric_free", "dtf_fabric_export", "dtf_fabric_import",
                 "dtf_fabric_close", "dtf_enable_peer", "dtf_can_access_peer", "dtf_memcpy_d2h", "dtf_memcpy_h2d",
                 "dtf_memset", "dtf_sizeof_ps_control", "dtf_sizeof_mailbox", "dtf_offsetof_ctl",
                 "dtf_ipc_handle_size"):
        getattr(lib, name).restype = c_int
    lib.dtf_offsetof_ctl.argtypes = [c_int]
    lib.dtf_fabric_bcast.argtypes = [c_void_p, c_void_p, c_void_p, c_int, c_longlong, c_int, c_void_p]
    lib.dtf_fabric_reduce.argtypes = [c_void_p, c_void_p, c_int, c_void_p, c_longlong, c_int, c_void_p]
    if not isinstance(getattr(lib, "dtf_fabric_reduce_ex", _Missing()), _Missing):
        lib.dtf_fabric_bcast_ex.argtypes = [c_void_p, c_void_p, c_void_p, c_int, c_longlong, c_int, c_int, c_void_p]
        lib.dtf_fabric_reduce_ex.argtypes = [c_void_p, c_void_p, c_int, c_void_p, c_longlong, c_int, c_int, c_void_p]
        lib.dtf_fabric_bcast_ex.restype = lib.dtf_fabric_reduce_ex.restype = c_int
    lib.dtf_vmm_support.argtypes = [c_int]
    lib.dtf_vmm_granularity.argtypes = [c_int, c_int, POINTER(c_longlong)]
    lib.dtf_vmm_create.argtypes = [c_int, c_longlong, POINTER(c_ulonglong)]
    lib.dtf_vmm_map.argtypes = [c_ulonglong, c_longlong, c_int, POINTER(c_void_p)]
    lib.dtf_vmm_unmap.argtypes = [c_void_p, c_longlong]
    lib.dtf_vmm_release.argtypes = [c_ulonglong]
    lib.dtf_vmm_export_fd.argtypes = [c_ulonglong, POINTER(c_int)]
    lib.dtf_vmm_import_fd.argtypes = [c_int, POINTER(c_ulonglong)]
    lib.dtf_mc_create.argtypes = [c_int, c_longlong, POINTER(c_ulonglong)]
    lib.dtf_mc_add_device.argtypes = [c_ulonglong, c_int]
    lib.dtf_mc_bind.argtypes = [c_ulonglong, c_ulonglong, c_longlong]
    lib.dtf_mc_unbind.argtypes = [c_ulonglong, c_int, c_longlong]
    for name in ("dtf_fabric_bcast", "dtf_fabric_reduce", "dtf_vmm_support", "dtf_vmm_granularity", "dtf_vmm_create",
                 "dtf_vmm_map", "dtf_vmm_unmap", "dtf_vmm_release", "dtf_vmm_export_fd", "dtf_vmm_import_fd",
                 "dtf_mc_create", "dtf_mc_add_device", "dtf_mc_bind", "dtf_mc_unbind"):
        getattr(lib, name).restype = c_int
    if not isinstance(getattr(lib, "dtf_mlp_step", _Missing()), _Missing):
        lib.dtf_mlp_step.argtypes = [POINTER(MlpStepArgs), c_void_p]
        lib.dtf_mlp_step.restype = c_int
        lib.dtf_mlp_step_slices.argtypes = [c_int, c_int, POINTER(c_int)]
        lib.dtf_mlp_step_slices.restype = c_int
        lib.dtf_mlp_step_scratch_floats.argtypes = [c_int, c_int, c_int]
        lib.dtf_mlp_step_scratch_floats.restype = c_longlong
        lib.dtf_sizeof_mlp_step_args.restype = c_int
        lib.dtf_mlp_step_head_part_floats.restype = c_int
        assert lib.dtf_sizeof_mlp_step_args() == ctypes.sizeof(MlpStepArgs), "MlpStepArgs layout mismatch"
    lib.dtf_run_ops.argtypes = [c_void_p, c_int, c_int, c_void_p, c_void_p]
    lib.dtf_run_ops.restype = c_int
    lib.dtf_capture_ops.argtypes = [c_void_p, c_int, c_int, c_void_p, POINTER(c_void_p), POINTER(c_int)]
    lib.dtf_capture_ops.restype = c_int
    lib.dtf_graph_destroy.argtypes = [c_void_p]
    lib.dtf_graph_destroy.restype = c_int
    lib.dtf_sizeof_step_op.restype = c_int
    lib.dtf_run_loop.argtypes = [POINTER(LoopArgs)]
    lib.dtf_run_loop.restype = c_int
    lib.dtf_sizeof_loop_args.restype = c_int
    if not isinstance(lib.dtf_sizeof_loop_args, _Missing):
        assert lib.dtf_sizeof_loop_args() == ctypes.sizeof(LoopArgs), "LoopArgs layout mismatch"
    if not isinstance(lib.dtf_sizeof_step_op, _Missing):
        assert lib.dtf_sizeof_step_op() == ctypes.sizeof(StepOp), "StepOp layout mismatch"
    if not isinstance(getattr(lib, "dtf_philox_fill", _Missing()), _Missing):    # random fills + element-wise graph ops (K13, K9)
        lib.dtf_philox_fill.argtypes = [c_void_p, c_longlong, c_ulonglong, c_ulonglong, c_ulonglong, c_int, c_float, c_float, c_void_p]
        lib.dtf_philox_fill.restype = c_int
        lib.dtf_ew_binary.argtypes = [c_void_p, c_void_p, c_void_p, c_longlong, c_int, c_int, c_int, c_longlong, c_void_p]
        lib.dtf_ew_binary.restype = c_int
        lib.dtf_ew_unary.argtypes = [c_void_p, c_void_p, c_longlong, c_int, c_void_p]
        lib.dtf_ew_unary.restype = c_int
        lib.dtf_copy_parts.argtypes = [c_int, c_longlong] + [c_void_p] * 7 + [c_void_p]
        lib.dtf_copy_parts.restype = c_int
        lib.dtf_ew_affine.argtypes = [c_void_p, c_void_p, c_longlong, c_int, c_float, c_float, c_void_p]
        lib.dtf_ew_affine.restype = c_int
        lib.dtf_ew_reduce_sum.argtypes = [c_void_p, c_longlong, c_float, c_int, c_void_p, c_void_p]
        lib.dtf_ew_reduce_sum.restype = c_int
    if not isinstance(getattr(lib, "dtf_bn_reduce", _Missing()), _Missing):    # csrc/nn_kernels.cu (a stale build lacks it)
        lib.dtf_bn_row_splits.argtypes = [c_longlong, c_int]
        lib.dtf_bn_row_splits.restype = c_int
        lib.dtf_bn_workspace_floats.argtypes = [c_longlong, c_int]
        lib.dtf_bn_workspace_floats.restype = c_longlong
        lib.dtf_bn_reduce.argtypes = [c_int] + [c_void_p] * 5 + [c_longlong, c_int] + [c_void_p] * 4 + [c_float, c_void_p]
        lib.dtf_bn_reduce.restype = c_int
        lib.dtf_bn_apply.argtypes = [c_void_p] * 7 + [c_longlong, c_int, c_int, c_void_p]
        lib.dtf_bn_apply.restype = c_int
        lib.dtf_bn_bwd_apply.argtypes = [c_void_p] * 10 + [c_longlong, c_int, c_void_p]
        lib.dtf_bn_bwd_apply.restype = c_int
        lib.dtf_im2col_nhwc_vec8.argtypes = [c_void_p, c_void_p] + [c_int] * 12 + [c_longlong, c_void_p]
        lib.dtf_im2col_nhwc_vec8.restype = c_int
        lib.dtf_col2im_nhwc_vec4.argtypes = [c_void_p, c_longlong, c_void_p] + [c_int] * 12 + [c_void_p]
        lib.dtf_col2im_nhwc_vec4.restype = c_int
        lib.dtf_maxpool_nhwc_fwd.argtypes = [c_void_p, c_void_p, c_void_p] + [c_int] * 12 + [c_void_p]
        lib.dtf_maxpool_nhwc_fwd.restype = c_int
        lib.dtf_maxpool_nhwc_bwd.argtypes = [c_void_p, c_void_p, c_void_p] + [c_int] * 12 + [c_void_p]
        lib.dtf_maxpool_nhwc_bwd.restype = c_int
        lib.dtf_global_avgpool_nhwc.argtypes = [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p]
        lib.dtf_global_avgpool_nhwc.restype = c_int


def load() -> ctypes.CDLL:
    global _LIB
    with _LOCK:
        if _LIB is not None:
            return _LIB
        p = lib_path()
        if not os.path.exists(p):
            raise RuntimeError("sm_100a kernel library %s is missing: run `python __graft_entry__.py build`" % p)
        lib = ctypes.CDLL(p)
        _declare(lib)
        _LIB = lib
        return lib


# ---------------------------------------------------------------------------------------------------
# kernel emulation: the op layer on HOST tensors (tests without a GPU)
# ---------------------------------------------------------------------------------------------------
EMULATION = False
_EMU_SOURCES = ("elementwise.cu", "ps_engine.cu", "nn_kernels.cu", "mlp_step.cu")


def enable_emulation(build_dir: Optional[str] = None) -> ctypes.CDLL:
    """Swap the kernel library for a g++ build of the SAME ``.cu`` sources against ``tests/emu/host_emu.h`` (threads +
    barriers emulate a thread block; docs/TESTING.md) and let the wrappers of this module -- and the autograd functions of
    ``ops/native.py`` on top -- accept host tensors.  The tcgen05 / TMA GEMM is hardware-only: ``gemm`` runs the CUDA-core
    reference GEMM kernel (same bf16-rounded operands, fp32 accumulate) instead.  Test tier only."""
    global _LIB, EMULATION
    import subprocess
    import tempfile
    root = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    csrc = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "csrc")
    emu_dir = os.path.join(root, "tests", "emu")
    out_dir = build_dir or tempfile.mkdtemp(prefix="dtf_emu_")
    so = os.path.join(out_dir, "libdtf_kernels_emu.so")
    if not os.path.exists(so):
        objs = []
        for src in _EMU_SOURCES:
            obj = os.path.join(out_dir, src + ".o")
            subprocess.run(["g++", "-O1", "-std=c++17", "-w", "-DDTF_HOST_EMU", "-I" + emu_dir, "-I" + csrc, "-x", "c++", "-fPIC",
                            "-pthread", "-c", os.path.join(csrc, src), "-o", obj], check=True)
            objs.append(obj)
        subprocess.run(["g++", "-shared", "-pthread", "-o", so] + objs, check=True)
    with _LOCK:
        lib = ctypes.CDLL(so)
        _declare(_Tolerant(lib))
        enable_emulation._saved = _LIB
        _LIB, EMULATION = lib, True
    return lib


def disable_emulation() -> None:
    global _LIB, EMULATION
    with _LOCK:
        _LIB, EMULATION = getattr(enable_emulation, "_saved", None), False


# csrc/nn_kernels.cu (fused batch norm, channel-vectorised im2col / col2im, NHWC pooling): validated on a B200 in round 2
# (tests/test_gpu_nn_fused.py; ResNet-18 step 14.6 -> 11.6 ms eager, 12.9 -> 5.4 ms CUDA-graphed) -> on by default.
# DTF_FUSED_NN=0 selects the element-wise PyTorch formulation again (DTF_FUSED_BN is the older name of the same switch).
FUSED_NN = os.environ.get("DTF_FUSED_NN", os.environ.get("DTF_FUSED_BN", "1")) == "1"

# launch counter: bench.py reports how many of OUR kernels ran in the timed region
_launches = 0


def launch_count() -> int:
    return _launches


def _bump(n: int = 1) -> None:
    global _launches
    _launches += n


def _check(rc: int, what: str) -> None:
    if rc != 0:
        raise RuntimeError("%s failed with code %d%s" % (what, rc, _cuda_err(rc)))


def _cuda_err(rc: int) -> str:
    if rc <= 0:
        return {-2: " (bad shape)", -3: " (leading dimension not a multiple of 8)", -4: " (pointer not 16-byte aligned)",
                -5: " (split-K with relu/bf16 output)", -6: " (bad BLOCK_N)", -7: " (cuTensorMapEncodeTiled unavailable)"
                }.get(rc, "")
    if rc >= 1000:
        return " (cuTensorMapEncodeTiled CUresult %d)" % (rc - 1000)
    return " (cudaError %d)" % rc


def _stream(t: Optional[torch.Tensor] = None) -> Optional[int]:
    if EMULATION:
        return None                       # host emulation: kernels run synchronously inside the call
    dev = t.device if t is not None else None
    return torch.cuda.current_stream(dev).cuda_stream


def _on(dev):
    """``torch.cuda.device(dev)`` for CUDA tensors; a no-op for the host tensors of the kernel-emulation mode."""
    dev = torch.device(dev) if not isinstance(dev, torch.device) else dev
    return torch.cuda.device(dev) if dev.type == "cuda" else contextlib.nullcontext()


def _on_device(t: torch.Tensor) -> bool:
    """May our kernels touch this tensor?  CUDA tensors always; host tensors only under the kernel emulation."""
    return t.is_cuda or EMULATION


def _ptr(t: Optional[torch.Tensor]) -> Optional[int]:
    return None if t is None else t.data_ptr()


def round_up(x: int, m: int) -> int:
    return (x + m - 1) // m * m


# ---------------------------------------------------------------------------------------------------
# conversions
# ---------------------------------------------------------------------------------------------------
def to_bf16_padded(x: torch.Tensor) -> Tuple[torch.Tensor, int]:
    """Row-major 2-D tensor -> (bf16 tensor whose row pitch is a multiple of 8 elements, pitch)."""
    assert x.dim() == 2 and _on_device(x)
    rows, cols = x.shape
    if x.dtype == torch.bfloat16 and x.stride(1) == 1 and x.stride(0) % 8 == 0 and x.data_ptr() % 16 == 0:
        return x, x.stride(0)
    ld = round_up(cols, 8)
    if x.dtype != torch.float32 or x.stride(1) != 1:
        x = x.float().contiguous()
    out = torch.empty((rows, ld), dtype=torch.bfloat16, device=x.device)
    lib = load()
    with _on(x.device):
        _check(lib.dtf_convert_f32_bf16(x.data_ptr(), x.stride(0), out.data_ptr(), ld, rows, cols, ld, _stream(x)),
               "convert_f32_bf16")
    _bump()
    return out, ld


def to_f32_padded(x: torch.Tensor) -> Tuple[torch.Tensor, int]:
    """Row-major 2-D tensor -> (fp32 tensor with a 16-byte row pitch and base, pitch): the TF32 GEMM's TMA reads fp32
    tensors in place; only odd pitches / other dtypes are copied."""
    assert x.dim() == 2 and _on_device(x)
    rows, cols = x.shape
    if x.dtype == torch.float32 and x.stride(1) == 1 and x.stride(0) % 4 == 0 and x.stride(0) >= cols and x.data_ptr() % 16 == 0:
        return x, x.stride(0)
    ld = round_up(cols, 4)
    out = torch.zeros((rows, ld), dtype=torch.float32, device=x.device) if ld != cols else \
        torch.empty((rows, ld), dtype=torch.float32, device=x.device)
    out[:, :cols].copy_(x)
    return out, ld


# Operand precision of fp32 matmuls on /gpu devices.  "tf32": fp32 tensors stay fp32 in memory and are multiplied by
# tcgen05.mma.kind::tf32 (the reference model is fp32: /root/reference/distributed_mnist.py:98-113); "bf16": operands
# are rounded to bf16 first (kind::f16, twice the tensor throughput).  Accumulation is fp32 either way.
MATMUL_PRECISION = os.environ.get("DTF_MATMUL_PRECISION", "tf32")


def set_matmul_precision(p: str) -> str:
    global MATMUL_PRECISION
    assert p in ("tf32", "bf16"), p
    old, MATMUL_PRECISION = MATMUL_PRECISION, p
    return old


# ---------------------------------------------------------------------------------------------------
# GEMM
# ---------------------------------------------------------------------------------------------------
def gemm_raw(a: torch.Tensor, lda: int, b: torch.Tensor, ldb: int, c: torch.Tensor, ldc: int, M: int, N: int, K: int,
             a_mn: bool, b_mn: bool, bias: Optional[torch.Tensor] = None, relu: bool = False,
             mask: Optional[torch.Tensor] = None, ldmask: int = 0, alpha: float = 1.0, splits: int = 1,
             accumulate: bool = False, colsum: Optional[torch.Tensor] = None, wait_flag: int = 0, wait_target: int = 0,
             signal: int = 0, err: int = 0, timeout_ns: int = 0, block_n: int = 0, stream: Optional[int] = None,
             a_ptr: Optional[int] = None, b_ptr: Optional[int] = None, c_ptr: Optional[int] = None,
             bias_ptr: Optional[int] = None, c_bf16: Optional[bool] = None, persistent: int = 0, tf32: bool = False) -> None:
    """Launch the tcgen05 GEMM on raw buffers (pointers may be peer memory).  ``tf32``: A and B are fp32."""
    g = GemmArgs()
    g.a = a_ptr if a_ptr is not None else a.data_ptr()
    g.b = b_ptr if b_ptr is not None else b.data_ptr()
    g.c = c_ptr if c_ptr is not None else c.data_ptr()
    g.M, g.N, g.K, g.lda, g.ldb, g.ldc = M, N, K, lda, ldb, ldc
    g.a_mn, g.b_mn = int(a_mn), int(b_mn)
    g.c_bf16 = int(c_bf16 if c_bf16 is not None else (c is not None and c.dtype == torch.bfloat16))
    g.bias = bias_ptr if bias_ptr is not None else _ptr(bias)
    g.relu = int(relu)
    g.mask, g.ldmask = _ptr(mask), ldmask
    g.alpha, g.splits, g.accumulate = alpha, splits, int(accumulate)
    g.colsum = _ptr(colsum)
    g.wait_flag, g.wait_target = wait_flag or None, wait_target
    g.signal, g.err, g.timeout_ns = signal or None, err or None, timeout_ns
    g.block_n_override = block_n
    g.persistent = persistent
    g.tf32 = int(tf32)
    lib = load()
    st = stream if stream is not None else torch.cuda.current_stream().cuda_stream
    _check(lib.dtf_gemm_bf16(byref(g), st), "gemm_bf16_tcgen05")
    _bump()


AUTO_SPLIT_K = os.environ.get("DTF_AUTO_SPLIT_K", "1") == "1"
# implicit-GEMM convolution (4-D TMA boxes over the NHWC activation instead of a materialised patch matrix)
IMPLICIT_CONV = os.environ.get("DTF_IMPLICIT_CONV", "1") == "1"


def implicit_conv_ok(n: int, h: int, w: int, c: int, strides=(1, 1)) -> bool:
    """Shapes the implicit-GEMM path of ``dtf_gemm_bf16`` takes (csrc/gemm_tcgen05.cu, ``conv``): stride 1, whole
    64-channel chunks, and both tile sizes (128 pixels for fprop / dgrad, 64 for wgrad) made of whole rows / whole images."""
    if tuple(strides) != (1, 1) or c % 64 or w > 64 or 64 % w:
        return False
    hw = h * w
    for tile in (128, 64):
        if not (hw % tile == 0 or tile % hw == 0) or (n * hw) % tile:
            return False
    return (h if hw < 128 else 128 // w) <= 256


def conv_igemm(x16: torch.Tensor, b: torch.Tensor, kh: int, kw: int, pt: int, pl: int, wgrad: bool = False,
               splits: int = 0) -> torch.Tensor:
    """Implicit-GEMM convolution product on the tcgen05 GEMM; ``x16``: bf16 NHWC activation [n, h, w, c] (dense).

    ``wgrad=False``: ``patches(x16) @ b`` with ``b`` = filter matrix [kh*kw*c, cout] -> fp32 [n*h*w, cout] (the forward
    convolution; with dY as ``x16`` and the flipped, in/out-swapped filter, the data gradient).
    ``wgrad=True``: ``patches(x16)^T @ b`` with ``b`` = dY [n*h*w, cout] -> fp32 [kh*kw*c, cout] (split-K over the pixels).
    The patch matrix is never written: the kernel's TMA producer loads one shifted 4-D box per (tap, 64-channel chunk) and
    the box's out-of-bounds zero fill is the padding."""
    assert x16.dtype == torch.bfloat16 and x16.is_contiguous() and x16.dim() == 4
    n, h, w, c = x16.shape
    pixels, kdim = n * h * w, kh * kw * c
    with _on(x16.device):
        b16, ldb = to_bf16_padded(b)
        cout = b.shape[1]
        g = GemmArgs()
        g.a, g.b, g.lda, g.ldb = x16.data_ptr(), b16.data_ptr(), c, ldb
        if not wgrad:
            M, N, K = pixels, cout, kdim
            g.a_mn, g.conv = 0, 1
        else:
            M, N, K = kdim, cout, pixels
            g.a_mn, g.conv = 1, 2
        assert b.shape[0] == K, (tuple(b.shape), K)
        if splits <= 0:
            splits = auto_splits(M, N, K, True, False) if AUTO_SPLIT_K else 1
        out = (torch.zeros if splits > 1 else torch.empty)((M, N), dtype=torch.float32, device=x16.device)
        g.c, g.ldc, g.M, g.N, g.K = out.data_ptr(), N, M, N, K
        g.b_mn, g.alpha, g.splits = 1, 1.0, splits
        g.cv_n, g.cv_h, g.cv_w, g.cv_c, g.cv_kh, g.cv_kw, g.cv_pt, g.cv_pl = n, h, w, c, kh, kw, pt, pl
        _check(load().dtf_gemm_bf16(byref(g), torch.cuda.current_stream().cuda_stream), "conv_igemm")
        _bump()
    return out


def auto_splits(M: int, N: int, K: int, b_mn: bool, tf32: bool, sms: int = 148) -> int:
    """Split-K factor for a GEMM whose output tiles do not fill the GPU (the weight-gradient GEMMs of a convolution are the
    extreme: [9*Cin, pixels] x [pixels, Cout] is a handful of tiles with K in the tens of thousands -- 5 CTAs walking
    K = 65536 measured 469 us; the same work over 150 CTAs is ~20 us).  Mirrors the tile choice of ``dtf_gemm_bf16``:
    at least 8 K-blocks per split, at most one wave of CTAs, and the fp32 red.add traffic (splits x output) bounded."""
    kbk = 32 if tf32 else 64
    if b_mn:
        bn = 64 if N <= 64 else (128 if N <= 128 else (192 if N <= 192 else 256))
    else:
        bn = round_up(N, 16)
        if bn > 256:
            bn = 256 if (N % 256 == 0 or N > 1024) else 128
    tiles = -(-M // 128) * -(-N // bn)
    num_kb = -(-K // kbk)
    if tiles * 2 > sms or num_kb < 16:
        return 1
    s = min(sms // tiles, num_kb // 8, max(1, (64 << 20) // (M * N * 4)))
    return max(int(s), 1)


def gemm(a: torch.Tensor, b: torch.Tensor, ta: bool = False, tb: bool = False, bias: Optional[torch.Tensor] = None,
         relu: bool = False, out_dtype: torch.dtype = torch.float32, splits: int = 0, persistent: int = 0,
         block_n: int = 0, precision: Optional[str] = None) -> torch.Tensor:
    """``op(a) @ op(b)`` (+bias, ReLU) on the tensor cores, fp32 accumulate.  ``precision``: "bf16" (operands rounded to
    bf16) or "tf32" (fp32 operands read in place, TF32 multiply); default: bf16 inputs -> "bf16", otherwise
    ``MATMUL_PRECISION``.  ``splits``: split-K factor (fp32 output, no ReLU); 0 = :func:`auto_splits`."""
    assert _on_device(a) and _on_device(b) and a.dim() == 2 and b.dim() == 2
    if precision is None:
        precision = "bf16" if (a.dtype == torch.bfloat16 or b.dtype == torch.bfloat16) else MATMUL_PRECISION
    tf32 = precision == "tf32"
    if EMULATION:
        # the tcgen05 / TMA kernel is hardware-only.  Same contract (bf16-rounded operands, fp32 accumulate, fused bias /
        # ReLU) from the CUDA-core reference GEMM kernel while one emulated thread per output element is affordable,
        # from a plain matmul beyond that.
        Mo = a.shape[1] if ta else a.shape[0]
        No = b.shape[0] if tb else b.shape[1]
        if Mo * No <= 1 << 14 and not tf32:
            out = gemm_ref(a, b, ta, tb, bias=bias, relu=relu)
        else:
            rnd = (lambda t: t.float()) if tf32 else (lambda t: t.bfloat16().float())
            x = rnd(a.t() if ta else a)
            y = rnd(b.t() if tb else b)
            out = x @ y
            if bias is not None:
                out = out + bias.float()
            if relu:
                out = torch.relu(out)
        return out if out_dtype == torch.float32 else out.to(out_dtype)
    M, K = (a.shape[1], a.shape[0]) if ta else (a.shape[0], a.shape[1])
    Kb, N = (b.shape[1], b.shape[0]) if tb else (b.shape[0], b.shape[1])
    if K != Kb:
        raise ValueError("gemm: inner dimensions differ (%d vs %d)" % (K, Kb))
    if splits <= 0:
        splits = auto_splits(M, N, K, not tb, tf32) if (out_dtype == torch.float32 and not relu and block_n == 0
                                                        and AUTO_SPLIT_K) else 1
    with _on(a.device):
        a16, lda = to_f32_padded(a) if tf32 else to_bf16_padded(a)
        b16, ldb = to_f32_padded(b) if tf32 else to_bf16_padded(b)
        ldc = N if out_dtype == torch.float32 else round_up(N, 8)
        c = (torch.zeros if splits > 1 else torch.empty)((M, ldc), dtype=out_dtype, device=a.device)
        if bias is not None:
            bias = bias.float().contiguous()
        gemm_raw(a16, lda, b16, ldb, c, ldc, M, N, K, a_mn=ta, b_mn=not tb, bias=bias, relu=relu, splits=splits,
                 persistent=persistent, block_n=block_n, tf32=tf32)
    return c if ldc == N else c[:, :N]


def gemm_ref(a: torch.Tensor, b: torch.Tensor, ta: bool = False, tb: bool = False, bias=None, relu=False) -> torch.Tensor:
    """CUDA-core reference over the same bf16-rounded operands (tests)."""
    M, K = (a.shape[1], a.shape[0]) if ta else (a.shape[0], a.shape[1])
    N = b.shape[0] if tb else b.shape[1]
    with _on(a.device):
        a16, lda = to_bf16_padded(a)
        b16, ldb = to_bf16_padded(b)
        c = torch.empty((M, N), dtype=torch.float32, device=a.device)
        lib = load()
        _check(lib.dtf_gemm_ref(a16.data_ptr(), b16.data_ptr(), c.data_ptr(), M, N, K, lda, ldb, N, int(ta), int(not tb),
                                _ptr(bias), int(relu), 1.0, _stream(a)), "gemm_ref")
    _bump()
    return c


# ---------------------------------------------------------------------------------------------------
# softmax / xent, relu grad, column sums
# ---------------------------------------------------------------------------------------------------
def softmax_xent_fwd_bwd(logits: torch.Tensor, labels: torch.Tensor, clip_min: float, reduce_sum: bool
                         ) -> Tuple[torch.Tensor, torch.Tensor]:
    logits = logits.float().contiguous()
    labels = labels.float().contiguous()
    rows, cols = logits.shape
    dl = torch.empty_like(logits)
    with _on(logits.device):
        if reduce_sum:
            loss = torch.zeros((), dtype=torch.float32, device=logits.device)
            lsum, lrows = loss.data_ptr(), None
        else:
            loss = torch.empty((rows,), dtype=torch.float32, device=logits.device)
            lsum, lrows = None, loss.data_ptr()
        lib = load()
        _check(lib.dtf_softmax_xent(logits.data_ptr(), cols, labels.data_ptr(), cols, rows, cols, clip_min, lsum, lrows,
                                    dl.data_ptr(), cols, None, 0, 0, None, 0, 1.0, _stream(logits)), "softmax_xent")
    _bump()
    return loss, dl


# ---------------------------------------------------------------------------------------------------
# random fills (K13) and element-wise graph ops (K9): csrc/elementwise.cu
# ---------------------------------------------------------------------------------------------------
PHILOX_UNIFORM, PHILOX_NORMAL, PHILOX_TRUNCATED_NORMAL = 0, 1, 2
EW_BINARY = {"add": 0, "sub": 1, "mul": 2, "div": 3, "max": 4, "min": 5, "sqdiff": 6}
EW_UNARY = {"neg": 0, "square": 1, "sqrt": 2, "rsqrt": 3, "exp": 4, "log": 5, "abs": 6, "sigmoid": 7, "tanh": 8, "relu": 9}
_EW_FULL, _EW_SCALAR, _EW_INNER = 0, 1, 2


def philox_fill(out: torch.Tensor, kind: int, p0: float, p1: float, key: int, offset: int, stream_id: int = 0) -> torch.Tensor:
    """Fill the contiguous fp32 tensor ``out`` from the Philox stream ``(key, stream_id)`` starting at block ``offset``
    (``csrc/philox.h``: element i = word i % 4 of block offset + i // 4).  Returns ``out``."""
    assert out.dtype == torch.float32 and out.is_contiguous() and _on_device(out)
    with _on(out.device):
        _check(load().dtf_philox_fill(out.data_ptr(), out.numel(), key & (2 ** 64 - 1), offset & (2 ** 64 - 1),
                                      stream_id & (2 ** 64 - 1), int(kind), float(p0), float(p1), _stream(out)), "philox_fill")
    _bump()
    return out


def ew_broadcast_mode(shape: Sequence[int], other: Sequence[int], out_shape: Sequence[int]) -> Optional[Tuple[int, int]]:
    """How the kernel indexes an operand of ``shape`` against the broadcast result ``out_shape``: (mode, inner) with mode
    full / scalar / trailing-dims vector, or None when the pattern needs a general broadcast (the op layer then uses torch)."""
    shape, out_shape = tuple(shape), tuple(out_shape)
    n = 1
    for d in shape:
        n *= d
    if shape == out_shape:
        return (_EW_FULL, 1)
    if n == 1:
        return (_EW_SCALAR, 1)
    core = shape
    while core and core[0] == 1:
        core = core[1:]
    if core and len(core) <= len(out_shape) and tuple(out_shape[len(out_shape) - len(core):]) == core:
        return (_EW_INNER, n)
    return None


def ew_binary(op: str, a: torch.Tensor, b: torch.Tensor) -> Optional[torch.Tensor]:
    """``a (op) b`` with numpy broadcasting for the patterns the kernel indexes directly; None = not handled."""
    if a.dtype != torch.float32 or b.dtype != torch.float32 or a.device != b.device:
        return None
    try:
        out_shape = torch.broadcast_shapes(a.shape, b.shape)
    except RuntimeError:
        return None
    ma, mb = ew_broadcast_mode(a.shape, b.shape, out_shape), ew_broadcast_mode(b.shape, a.shape, out_shape)
    if ma is None or mb is None:
        return None
    a, b = a.contiguous(), b.contiguous()
    out = torch.empty(out_shape, dtype=torch.float32, device=a.device)
    inner = ma[1] if ma[0] == _EW_INNER else mb[1]
    if ma[0] == _EW_INNER and mb[0] == _EW_INNER and ma[1] != mb[1]:
        return None
    with _on(a.device):
        _check(load().dtf_ew_binary(a.data_ptr(), b.data_ptr(), out.data_ptr(), out.numel(), EW_BINARY[op], ma[0], mb[0], inner,
                                    _stream(a)), "ew_binary(%s)" % op)
    _bump()
    return out


def ew_unary(op: str, x: torch.Tensor) -> torch.Tensor:
    x = x.contiguous()
    out = torch.empty_like(x)
    with _on(x.device):
        _check(load().dtf_ew_unary(x.data_ptr(), out.data_ptr(), x.numel(), EW_UNARY[op], _stream(x)), "ew_unary(%s)" % op)
    _bump()
    return out


def _copy_parts(outer: int, srcs, dsts, src_stride, dst_stride, src_off, dst_off, row_len, device: torch.device) -> None:
    n = len(srcs)
    LL, VP = c_longlong * n, c_void_p * n
    with _on(device):
        _check(load().dtf_copy_parts(n, int(outer), VP(*srcs), VP(*dsts), LL(*src_stride), LL(*dst_stride), LL(*src_off), LL(*dst_off),
                                     LL(*row_len), None if EMULATION else torch.cuda.current_stream(device).cuda_stream),
               "copy_parts")
    _bump()


def concat(xs: Sequence[torch.Tensor], axis: int) -> Optional[torch.Tensor]:
    """``torch.cat(xs, axis)`` of 2..16 contiguous fp32 tensors in ONE gather kernel; None = not handled."""
    xs = list(xs)
    if not (2 <= len(xs) <= 16) or any(x.dtype != torch.float32 or x.device != xs[0].device or x.dim() != xs[0].dim() or x.dim() == 0
                                       for x in xs):
        return None
    nd = xs[0].dim()
    ax = axis % nd
    base = list(xs[0].shape)
    for x in xs:
        if [d for i, d in enumerate(x.shape) if i != ax] != [d for i, d in enumerate(base) if i != ax]:
            return None
    outer, inner = 1, 1
    for d in base[:ax]:
        outer *= d
    for d in base[ax + 1:]:
        inner *= d
    lens = [x.shape[ax] for x in xs]
    total = sum(lens)
    shape = base[:ax] + [total] + base[ax + 1:]
    out = torch.empty(shape, dtype=torch.float32, device=xs[0].device)
    xs = [x.contiguous() for x in xs]
    offs, acc = [], 0
    for l in lens:
        offs.append(acc * inner)
        acc += l
    _copy_parts(outer, [x.data_ptr() for x in xs], [out.data_ptr()] * len(xs), [l * inner for l in lens], [total * inner] * len(xs),
                [0] * len(xs), offs, [l * inner for l in lens], out.device)
    return out


def scatter_rows(x: torch.Tensor, outs: Sequence[torch.Tensor]) -> None:
    """Split the leading dimension of the contiguous fp32 ``x`` across ``outs`` (contiguous fp32, rows summing to x's) with ONE
    kernel launched on x's device; an ``out`` on another GPU is written through its peer mapping (peer access must be on)."""
    outs = list(outs)
    assert 1 <= len(outs) <= 16 and x.dtype == torch.float32 and x.is_contiguous() and x.dim() >= 1
    inner = x[0].numel() if x.shape[0] else 1
    rows = [o.shape[0] for o in outs]
    assert sum(rows) == x.shape[0] and all(o.dtype == torch.float32 and o.is_contiguous() and (o[0].numel() if o.shape[0] else inner) == inner
                                             for o in outs)
    offs, acc = [], 0
    for r in rows:
        offs.append(acc * inner)
        acc += r
    _copy_parts(1, [x.data_ptr()] * len(outs), [o.data_ptr() for o in outs], [0] * len(outs), [0] * len(outs), offs, [0] * len(outs),
                [r * inner for r in rows], x.device)


def ew_affine(x: torch.Tensor, alpha: float, beta: float = 0.0, out_shape: Optional[Sequence[int]] = None) -> torch.Tensor:
    """``alpha * x + beta``; with ``out_shape`` the one-element ``x`` is broadcast to that shape."""
    x = x.contiguous()
    if out_shape is None:
        out, mode = torch.empty_like(x), _EW_FULL
    else:
        assert x.numel() == 1
        out, mode = torch.empty(tuple(out_shape), dtype=torch.float32, device=x.device), _EW_SCALAR
    with _on(x.device):
        _check(load().dtf_ew_affine(x.data_ptr(), out.data_ptr(), out.numel(), mode, float(alpha), float(beta), _stream(x)), "ew_affine")
    _bump()
    return out


def ew_reduce_sum(x: torch.Tensor, scale: float = 1.0, square: bool = False) -> torch.Tensor:
    """0-d tensor ``scale * sum(x)`` (``square``: of the squares) over every element."""
    x = x.contiguous()
    out = torch.empty((), dtype=torch.float32, device=x.device)
    with _on(x.device):
        _check(load().dtf_ew_reduce_sum(x.data_ptr(), x.numel(), float(scale), int(bool(square)), out.data_ptr(), _stream(x)),
               "ew_reduce_sum")
    _bump()
    return out


def relu_grad(g: torch.Tensor, y: torch.Tensor) -> torch.Tensor:
    g = g.float().contiguous()
    y = y.float().contiguous()
    out = torch.empty_like(g)
    with _on(g.device):
        _check(load().dtf_relu_grad(g.data_ptr(), y.data_ptr(), out.data_ptr(), g.numel(), _stream(g)), "relu_grad")
    _bump()
    return out


def colsum(x: torch.Tensor) -> torch.Tensor:
    x = x.float().contiguous()
    rows, cols = x.shape
    out = torch.empty((cols,), dtype=torch.float32, device=x.device)
    with _on(x.device):
        _check(load().dtf_colsum(x.data_ptr(), cols, rows, cols, out.data_ptr(), _stream(x)), "colsum")
    _bump()
    return out


def argmax_rows(x: torch.Tensor) -> torch.Tensor:
    x = x.float().contiguous()
    rows, cols = x.shape
    out = torch.empty((rows,), dtype=torch.int64, device=x.device)
    with _on(x.device):
        _check(load().dtf_argmax_rows(x.data_ptr(), cols, rows, cols, out.data_ptr(), _stream(x)), "argmax_rows")
    _bump()
    return out


# ---------------------------------------------------------------------------------------------------
# optimizer applies (in place)
# ---------------------------------------------------------------------------------------------------
def _apply(var, m, v, g, kind, lr, momentum=0.0, nesterov=False, beta1=0.0, beta2=0.0, eps=0.0, shadow=None,
           grad_scale=1.0):
    assert var.is_contiguous() and var.dtype == torch.float32
    g = g.to(dtype=torch.float32).contiguous()
    with _on(var.device):
        _check(load().dtf_optimizer_apply(var.data_ptr(), _ptr(m), _ptr(v), g.data_ptr(), _ptr(shadow), var.numel(), kind,
                                          lr, momentum, int(nesterov), beta1, beta2, eps, grad_scale, _stream(var)),
               "optimizer_apply")
    _bump()


def apply_sgd_(var, g, lr, shadow=None):
    _apply(var, None, None, g, 0, lr, shadow=shadow)


def apply_momentum_(var, acc, g, lr, momentum, nesterov=False, shadow=None):
    _apply(var, acc, None, g, 1, lr, momentum=momentum, nesterov=nesterov, shadow=shadow)


def apply_adam_(var, m, v, g, lr_t, beta1, beta2, eps, shadow=None):
    _apply(var, m, v, g, 2, lr_t, beta1=beta1, beta2=beta2, eps=eps, shadow=shadow)


# ---------------------------------------------------------------------------------------------------
# convolution lowering
# ---------------------------------------------------------------------------------------------------
def im2col_nhwc(x: torch.Tensor, kh: int, kw: int, strides: Sequence[int], pads: Sequence[int]):
    x = x.float().contiguous()
    n, h, w, c = x.shape
    sh, sw = strides
    pt, pb, pl, pr = pads
    ho = (h + pt + pb - kh) // sh + 1
    wo = (w + pl + pr - kw) // sw + 1
    kdim = kh * kw * c
    ld = round_up(kdim, 8)
    cols = torch.empty((n * ho * wo, ld), dtype=torch.bfloat16, device=x.device)
    with _on(x.device):
        rc = load().dtf_im2col_nhwc_vec8(x.data_ptr(), cols.data_ptr(), n, h, w, c, kh, kw, sh, sw, pt, pl, ho, wo, ld,
                                         _stream(x)) if FUSED_NN and c % 8 == 0 else -1
        if rc >= 0:                       # -1: not eligible -> scalar kernel below
            _check(rc, "im2col_nhwc_vec8")
            _bump()
            return cols, (n, ho, wo)
        _check(load().dtf_im2col_nhwc(x.data_ptr(), cols.data_ptr(), n, h, w, c, kh, kw, sh, sw, pt, pl, ho, wo, ld,
                                      _stream(x)), "im2col_nhwc")
    _bump()
    return (cols if ld == kdim else cols[:, :kdim]), (n, ho, wo)


def col2im_nhwc(gcols: torch.Tensor, xshape, kh: int, kw: int, strides, pads) -> torch.Tensor:
    gcols = gcols.float().contiguous()
    n, h, w, c = xshape
    sh, sw = strides
    pt, pb, pl, pr = pads
    ho = (h + pt + pb - kh) // sh + 1
    wo = (w + pl + pr - kw) // sw + 1
    gx = torch.empty(tuple(xshape), dtype=torch.float32, device=gcols.device)
    with _on(gcols.device):
        rc = load().dtf_col2im_nhwc_vec4(gcols.data_ptr(), gcols.shape[1], gx.data_ptr(), n, h, w, c, kh, kw, sh, sw, pt, pl,
                                         ho, wo, _stream(gcols)) if FUSED_NN and c % 4 == 0 else -1
        if rc >= 0:
            _check(rc, "col2im_nhwc_vec4")
            _bump()
            return gx
        _check(load().dtf_col2im_nhwc(gcols.data_ptr(), gcols.shape[1], gx.data_ptr(), n, h, w, c, kh, kw, sh, sw, pt, pl,
                                      ho, wo, _stream(gcols)), "col2im_nhwc")
    _bump()
    return gx


# ---------------------------------------------------------------------------------------------------
# fused training-mode batch norm over [rows, C] fp32 (csrc/nn_kernels.cu); all launches on the current stream
# ---------------------------------------------------------------------------------------------------
_BN_WS: dict = {}


def _bn_workspace(dev: torch.device, floats: int):
    """Per-device scratch: partial sums (grown on demand) + the ticket counters (zeroed once; the kernel resets them).
    One workspace per device = calls must be stream-ordered, which they are (everything runs on the current stream)."""
    ws = _BN_WS.get(dev)
    if ws is None or ws[0].numel() < floats:
        tickets = ws[1] if ws is not None else torch.zeros(64, dtype=torch.int32, device=dev)
        ws = _BN_WS[dev] = (torch.empty(max(floats, 1 << 16), dtype=torch.float32, device=dev), tickets)
    return ws


def _aligned16(t: torch.Tensor) -> torch.Tensor:
    """Views into flat parameter buffers can start at any element: the float4 kernels need 16-byte alignment."""
    return t if t.data_ptr() % 16 == 0 else t.clone()


def bn_forward(x2d: torch.Tensor, scale: torch.Tensor, offset: torch.Tensor, residual: Optional[torch.Tensor], relu: bool,
               eps: float):
    """x2d: [rows, C] fp32 contiguous, C % 4 == 0, C <= 8192 -> (y, mean, rstd)."""
    lib = load()
    rows, C = x2d.shape
    assert x2d.dtype == torch.float32 and x2d.is_contiguous() and C % 4 == 0 and C <= 64 * 128
    dev = x2d.device
    mean = torch.empty(C, dtype=torch.float32, device=dev)
    rstd = torch.empty(C, dtype=torch.float32, device=dev)
    y = torch.empty_like(x2d)
    scale, offset = _aligned16(scale.float().contiguous()), _aligned16(offset.float().contiguous())
    if residual is not None:
        residual = _aligned16(residual.float().contiguous())
    with _on(dev):
        ws, tickets = _bn_workspace(dev, int(lib.dtf_bn_workspace_floats(rows, C)))
        st = _stream(x2d)
        _check(lib.dtf_bn_reduce(0, x2d.data_ptr(), None, None, None, None, rows, C, ws.data_ptr(), tickets.data_ptr(),
                                 mean.data_ptr(), rstd.data_ptr(), float(eps), st), "bn_reduce(stats)")
        _check(lib.dtf_bn_apply(x2d.data_ptr(), _ptr(residual), y.data_ptr(), mean.data_ptr(), rstd.data_ptr(),
                                scale.data_ptr(), offset.data_ptr(), rows, C, int(relu), st), "bn_apply")
    _bump(2)
    return y, mean, rstd


def bn_backward(dy: torch.Tensor, y_mask: Optional[torch.Tensor], x2d: torch.Tensor, mean: torch.Tensor, rstd: torch.Tensor,
                scale: torch.Tensor, want_dres: bool):
    """-> (dx, dscale, doffset, dres or None).  ``y_mask``: the forward output when ReLU was fused (gradient gate)."""
    lib = load()
    rows, C = x2d.shape
    dev = x2d.device
    dy = _aligned16(dy.float().contiguous())
    scale = _aligned16(scale.float().contiguous())
    doffset = torch.empty(C, dtype=torch.float32, device=dev)
    dscale = torch.empty(C, dtype=torch.float32, device=dev)
    dx = torch.empty_like(x2d)
    dres = torch.empty_like(x2d) if want_dres else None
    with _on(dev):
        ws, tickets = _bn_workspace(dev, int(lib.dtf_bn_workspace_floats(rows, C)))
        st = _stream(x2d)
        _check(lib.dtf_bn_reduce(1, x2d.data_ptr(), dy.data_ptr(), _ptr(y_mask), mean.data_ptr(), rstd.data_ptr(), rows, C,
                                 ws.data_ptr(), tickets.data_ptr(), doffset.data_ptr(), dscale.data_ptr(), 0.0, st),
               "bn_reduce(backward)")
        _check(lib.dtf_bn_bwd_apply(dy.data_ptr(), _ptr(y_mask), x2d.data_ptr(), mean.data_ptr(), rstd.data_ptr(),
                                    scale.data_ptr(), doffset.data_ptr(), dscale.data_ptr(), dx.data_ptr(), _ptr(dres),
                                    rows, C, st), "bn_bwd_apply")
    _bump(2)
    return dx, dscale, doffset, dres


# ---------------------------------------------------------------------------------------------------
# pooling (csrc/nn_kernels.cu), NHWC fp32, C % 4 == 0
# ---------------------------------------------------------------------------------------------------
def maxpool_nhwc(x: torch.Tensor, kh: int, kw: int, strides: Sequence[int], pads: Sequence[int]):
    """-> (y [n, ho, wo, c], argmax bytes [n, ho, wo, c]: position inside the window, consumed by the backward)."""
    x = _aligned16(x.float().contiguous())
    n, h, w, c = x.shape
    sh, sw = strides
    pt, pb, pl, pr = pads
    ho = (h + pt + pb - kh) // sh + 1
    wo = (w + pl + pr - kw) // sw + 1
    y = torch.empty((n, ho, wo, c), dtype=torch.float32, device=x.device)
    arg = torch.empty((n, ho, wo, c), dtype=torch.uint8, device=x.device)
    with _on(x.device):
        _check(load().dtf_maxpool_nhwc_fwd(x.data_ptr(), y.data_ptr(), arg.data_ptr(), n, h, w, c, kh, kw, sh, sw, pt, pl, ho, wo,
                                           _stream(x)), "maxpool_nhwc_fwd")
    _bump()
    return y, arg


def maxpool_nhwc_bwd(dy: torch.Tensor, arg: torch.Tensor, xshape, kh: int, kw: int, strides, pads) -> torch.Tensor:
    dy = _aligned16(dy.float().contiguous())
    n, h, w, c = xshape
    sh, sw = strides
    pt, pb, pl, pr = pads
    ho, wo = dy.shape[1], dy.shape[2]
    dx = torch.empty(tuple(xshape), dtype=torch.float32, device=dy.device)
    with _on(dy.device):
        _check(load().dtf_maxpool_nhwc_bwd(dy.data_ptr(), arg.data_ptr(), dx.data_ptr(), n, h, w, c, kh, kw, sh, sw, pt, pl, ho,
                                           wo, _stream(dy)), "maxpool_nhwc_bwd")
    _bump()
    return dx


def global_avgpool_nhwc(x: torch.Tensor) -> torch.Tensor:
    x = _aligned16(x.float().contiguous())
    n, h, w, c = x.shape
    out = torch.empty((n, c), dtype=torch.float32, device=x.device)
    with _on(x.device):
        _check(load().dtf_global_avgpool_nhwc(x.data_ptr(), out.data_ptr(), n, h * w, c, 0, _stream(x)), "global_avgpool_nhwc")
    _bump()
    return out


def global_avgpool_nhwc_bwd(dy: torch.Tensor, xshape) -> torch.Tensor:
    dy = _aligned16(dy.float().contiguous())
    n, h, w, c = xshape
    dx = torch.empty(tuple(xshape), dtype=torch.float32, device=dy.device)
    with _on(dy.device):
        _check(load().dtf_global_avgpool_nhwc(dy.data_ptr(), dx.data_ptr(), n, h * w, c, 1, _stream(dy)), "global_avgpool_nhwc_bwd")
    _bump()
    return dx
