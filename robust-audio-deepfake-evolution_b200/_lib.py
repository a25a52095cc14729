"""ctypes binding of libbimamba_sm100.so (the C ABI declared in include/bimamba.h).

There is deliberately NO fallback: if the library is missing or a call fails this raises.
"""
from __future__ import annotations

import ctypes as C
import os
import threading

HERE = os.path.dirname(os.path.abspath(__file__))
# BIMAMBA_LIB: an experiment build of the SAME library (build.py --variant, e.g. another -D flag) for A/B timing runs
LIB_PATH = os.environ.get("BIMAMBA_LIB") or os.path.join(HERE, "libbimamba_sm100.so")

F32, BF16, F16 = 0, 1, 2
FLAG_SOFTPLUS = 1
FLAG_DTR_PADDED = 2
FLAG_SILU = 1
ABI_VERSION = 12
CHUNK = 16

EXPORTS = (
    "bimamba_abi_version", "bimamba_last_error", "bimamba_scan_plan",
    "bimamba_selective_scan_fwd", "bimamba_selective_scan_bwd",
    "bimamba_causal_conv1d_fwd", "bimamba_causal_conv1d_bwd", "bimamba_conv_bwd_slices",
    "bimamba_reduce_partials", "bimamba_layernorm_fwd", "bimamba_layernorm_bwd_blocks", "bimamba_layernorm_bwd",
    "bimamba_gemm_nt_block_n", "bimamba_gemm_nt_block_n_k", "bimamba_gemm_nt", "bimamba_gemm_tn_splits", "bimamba_gemm_tn", "bimamba_adamw_chunk", "bimamba_adamw_step", "bimamba_head_fwd", "bimamba_colsum_slices", "bimamba_colsum", "bimamba_pack_weights", "bimamba_cast_transpose",
    "bimamba_gelu_fwd", "bimamba_gelu_bwd", "bimamba_reduce_rows32", "bimamba_finalize_param_grads", "bimamba_head_pool_bwd", "bimamba_set_tuning", "bimamba_get_tuning",
    "bimamba_scan_fwd_workspace_bytes", "bimamba_scan_bwd_workspace_bytes", "bimamba_split3_bf16", "bimamba_cast", "bimamba_sumsq_slices", "bimamba_sumsq", "bimamba_scale_by",
    "bimamba_scan_fwd_split_plan", "bimamba_scan_fwd_split_workspace_bytes", "bimamba_selective_scan_fwd_split",
    "bimamba_block_fwd_workspace_bytes", "bimamba_block_bwd_workspace_bytes", "bimamba_block_fwd", "bimamba_block_bwd",
    "bimamba_layer_fwd_workspace_bytes", "bimamba_layer_bwd_workspace_bytes", "bimamba_layer_fwd", "bimamba_layer_bwd",
    "bimamba_causal_conv1d_fwd_varlen", "bimamba_selective_scan_fwd_varlen", "bimamba_head_fwd_varlen",
    "bimamba_block_fwd_varlen", "bimamba_layer_fwd_varlen",
    "bimamba_selective_scan_fwd_varlen_train", "bimamba_selective_scan_bwd_varlen", "bimamba_causal_conv1d_bwd_varlen",
    "bimamba_head_pool_bwd_varlen", "bimamba_block_fwd_varlen_train", "bimamba_block_bwd_varlen",
    "bimamba_layer_fwd_varlen_train", "bimamba_layer_bwd_varlen", "bimamba_mask_frames",
    "bimamba_interp_frames_fwd", "bimamba_interp_frames_bwd", "bimamba_frame_mean", "bimamba_frame_mean_bwd",
    "bimamba_frame_scale", "bimamba_frame_scale_bwd_slices", "bimamba_frame_scale_bwd",
    "bimamba_block_bwd_side", "bimamba_layer_fwd_side", "bimamba_layer_bwd_side",
    "bimamba_amp_grad_stats", "bimamba_adamw_amp_step", "bimamba_amp_update",
    "bimamba_mixup_frames",
)


class ScanDesc(C.Structure):
    """Mirror of `struct bimamba_scan_desc` (include/bimamba.h)."""
    _fields_ = (
        [(n, C.c_void_p) for n in (
            "u", "z", "delta", "bc", "dtr", "Wdt", "A", "D", "delta_bias", "out", "ypre", "ckpt",
            "dout", "du", "ddelta", "dz", "dbc_part", "dA_part", "dD_part", "dbias_part")]
        + [(n, C.c_int32) for n in (
            "batch", "ndir", "dim", "seqlen", "dstate", "dt_rank", "io_dtype", "flags",
            "group_channels", "reserved0")]
        + [(n, C.c_int64) for n in (
            "u_bs", "u_ds", "u_ts", "z_bs", "z_ds", "z_ts", "delta_bs", "delta_ds", "delta_ts",
            "bc_bs", "bc_ds", "bc_ts", "dtr_bs", "dtr_ds", "dtr_ts", "out_bs", "out_ds", "out_ts",
            "dout_bs", "dout_ds", "dout_ts")]
    )


class BlockDesc(C.Structure):
    """Mirror of `struct bimamba_block_desc` (include/bimamba.h): the whole block, forward."""
    _fields_ = (
        [(n, C.c_void_p) for n in ("x", "out", "Wi", "Wxp", "Wo2", "Wdt", "A", "D", "dt_bias", "conv_w", "conv_b",
                                   "workspace")]
        + [("workspace_bytes", C.c_size_t)]
        + [(n, C.c_int32) for n in ("batch", "seqlen", "d_model", "d_inner", "dt_rank", "d_conv", "ndir", "io_dtype",
                                    "save_for_backward", "reserved0")]
    )


class BlockGrads(C.Structure):
    """Mirror of `struct bimamba_block_grads` (include/bimamba.h): the whole block, backward."""
    _fields_ = (
        [(n, C.c_void_p) for n in ("dout", "dx", "WiT", "WxpT", "WoT", "WdT", "dW_in", "dconv_w", "dconv_b", "dW_x",
                                   "dW_dt", "db_dt", "dA_log", "dD", "dW_out", "workspace")]
        + [("workspace_bytes", C.c_size_t)]
    )


class LayerDesc(C.Structure):
    """Mirror of `struct bimamba_layer_desc` (include/bimamba.h): the whole encoder layer, forward."""
    _fields_ = (
        [(n, C.c_void_p) for n in ("x", "out", "norm1_w", "norm1_b", "norm2_w", "norm2_b", "ff_w1", "ff_b1", "ff_w2", "ff_b2")]
        + [("block", BlockDesc), ("workspace", C.c_void_p), ("workspace_bytes", C.c_size_t),
           ("eps1", C.c_float), ("eps2", C.c_float), ("d_ff", C.c_int32), ("x_dtype", C.c_int32)]
    )


class LayerGrads(C.Structure):
    """Mirror of `struct bimamba_layer_grads` (include/bimamba.h): the whole encoder layer, backward."""
    _fields_ = (
        [(n, C.c_void_p) for n in ("dout", "dx", "dnorm1", "dnorm2", "dff_w1", "dff_b1", "dff_w2", "dff_b2")]
        + [("block", BlockGrads), ("workspace", C.c_void_p), ("workspace_bytes", C.c_size_t)]
    )


class SideStream(C.Structure):
    """Mirror of `struct bimamba_side_stream` (include/bimamba.h): the second stream of the *_side calls."""
    _fields_ = [("stream", C.c_void_p), ("events", C.c_void_p * 3)]


class BlockPack(C.Structure):
    """Mirror of `struct bimamba_block_pack` (include/bimamba.h): the block's weight pack inside bimamba_layer_fwd_side."""
    _fields_ = [(n, C.c_void_p) for n in ("W_in", "W_x", "W_dt", "A_log", "W_out", "Wi", "WiT", "Wxp", "WxpT", "Wo2", "WoT",
                                          "WdT", "A")]


class AmpRecord(C.Structure):
    """Mirror of `struct bimamba_amp` (include/bimamba.h): the loss-scaling record of the fp16 optimizer step."""
    _fields_ = [("scale", C.c_float), ("growth_tracker", C.c_int32), ("found_inf", C.c_float), ("total_norm", C.c_float),
                ("clip_coef", C.c_float), ("reserved", C.c_int32 * 3)]


_lib = None
_lock = threading.Lock()

# number of kernels this library has enqueued through the bindings in ops.py (bench.py reports it
# as `gpu_launches`); every successful entry-point call below enqueues exactly one kernel.
launch_count = 0
# optional hook: callable(name) -> context manager, wrapped around each enqueue (bench.py uses it to
# put CUDA events around individual kernels for the roofline figure)
kernel_timer = None


def load() -> C.CDLL:
    """Load (once) and type the library.  Raises if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    with _lock:
        if _lib is not None:
            return _lib
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                f"{LIB_PATH} is missing: build it with `python __graft_entry__.py` or "
                "`python robust-audio-deepfake-evolution_b200/build.py` (needs nvcc). "
                "There is no CPU fallback for the Bi-Mamba path.")
        lib = C.CDLL(LIB_PATH)
        i32, i64, vp = C.c_int, C.c_int64, C.c_void_p
        lib.bimamba_abi_version.restype = i32
        lib.bimamba_abi_version.argtypes = []
        lib.bimamba_last_error.restype = C.c_char_p
        lib.bimamba_last_error.argtypes = []
        lib.bimamba_scan_plan.restype = i32
        lib.bimamba_scan_plan.argtypes = [i32, i32, i32, i32, C.POINTER(i32), C.POINTER(i32)]
        for name in ("bimamba_selective_scan_fwd", "bimamba_selective_scan_bwd"):
            fn = getattr(lib, name)
            fn.restype = i32
            fn.argtypes = [C.POINTER(ScanDesc), vp]
        lib.bimamba_causal_conv1d_fwd.restype = i32
        lib.bimamba_causal_conv1d_fwd.argtypes = [vp, vp, vp, vp, i32, i32, i32, i32, i32,
                                                  i64, i64, i64, i64, i64, i32, i32, vp]
        lib.bimamba_selective_scan_fwd_varlen.restype = i32
        lib.bimamba_selective_scan_fwd_varlen.argtypes = [C.POINTER(ScanDesc), vp, vp]
        lib.bimamba_causal_conv1d_fwd_varlen.restype = i32
        lib.bimamba_causal_conv1d_fwd_varlen.argtypes = [vp, vp, vp, vp, vp, i32, i32, i32, i32, i32,
                                                         i64, i64, i64, i64, i64, i32, i32, vp]
        lib.bimamba_causal_conv1d_bwd.restype = i32
        lib.bimamba_causal_conv1d_bwd.argtypes = [vp, vp, vp, vp, vp, vp, vp, vp, i32, i32, i32, i32, i32,
                                                  i64, i64, i64, i64, i64, i64, i64, i32, i32, vp]
        lib.bimamba_conv_bwd_slices.restype = i32
        lib.bimamba_conv_bwd_slices.argtypes = [i32, i32, i32]
        lib.bimamba_reduce_partials.restype = i32
        lib.bimamba_reduce_partials.argtypes = [vp, vp, i64, i64, i64, i64, i64, i64, i32, i32, vp]
        f32 = C.c_float
        lib.bimamba_layernorm_fwd.restype = i32
        lib.bimamba_layernorm_fwd.argtypes = [vp, vp, vp, vp, vp, vp, i64, i32, f32, i32, i32, vp]
        lib.bimamba_layernorm_bwd_blocks.restype = i32
        lib.bimamba_layernorm_bwd_blocks.argtypes = [i64]
        lib.bimamba_layernorm_bwd.restype = i32
        lib.bimamba_layernorm_bwd.argtypes = [vp, vp, vp, vp, vp, vp, vp, vp, i64, i32, i32, i32, vp]
        lib.bimamba_gemm_nt_block_n.restype = i32
        lib.bimamba_gemm_nt_block_n.argtypes = [i32]
        lib.bimamba_pack_weights.restype = i32
        lib.bimamba_pack_weights.argtypes = [vp] * 13 + [i32] * 6 + [vp]
        lib.bimamba_cast_transpose.restype = i32
        lib.bimamba_cast_transpose.argtypes = [vp, vp, vp, i32, i32, i32, vp]
        lib.bimamba_colsum_slices.restype = i32
        lib.bimamba_colsum_slices.argtypes = [i64]
        lib.bimamba_colsum.restype = i32
        lib.bimamba_colsum.argtypes = [vp, vp, i64, i32, i64, i32, vp]
        lib.bimamba_gemm_nt_block_n_k.restype = i32
        lib.bimamba_gemm_nt_block_n_k.argtypes = [i32, i32]
        lib.bimamba_head_fwd.restype = i32
        lib.bimamba_head_fwd.argtypes = [vp, vp, vp, vp, vp, vp, vp, vp, vp, i32, i32, i32, i32, C.c_float, i32, vp]
        lib.bimamba_head_fwd_varlen.restype = i32
        lib.bimamba_head_fwd_varlen.argtypes = [vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, i32, i32, i32, i32, C.c_float, i32, vp]
        lib.bimamba_adamw_chunk.restype = i32
        lib.bimamba_adamw_chunk.argtypes = []
        lib.bimamba_adamw_step.restype = i32
        lib.bimamba_adamw_step.argtypes = [vp, vp, i32, vp, vp, vp]
        lib.bimamba_amp_grad_stats.restype = i32
        lib.bimamba_amp_grad_stats.argtypes = [vp, vp, i32, C.c_float, vp, vp, vp]
        lib.bimamba_adamw_amp_step.restype = i32
        lib.bimamba_adamw_amp_step.argtypes = [vp, vp, i32, vp, vp, vp, vp, vp, C.c_float, vp]
        lib.bimamba_amp_update.restype = i32
        lib.bimamba_amp_update.argtypes = [vp, C.c_double, C.c_double, i32, vp, vp]
        lib.bimamba_gemm_tn_splits.restype = i32
        lib.bimamba_gemm_tn_splits.argtypes = [i64, i32, i32]
        lib.bimamba_gemm_tn.restype = i32
        lib.bimamba_gemm_tn.argtypes = [vp, i64, vp, i64, vp, vp, i64, i32, i32, i32, vp]
        lib.bimamba_gemm_nt.restype = i32
        lib.bimamba_gemm_nt.argtypes = [vp, i64, vp, i64, vp, i64, vp, vp, i64, i32, i32, i32, i32, vp]
        lib.bimamba_gelu_fwd.restype = i32
        lib.bimamba_gelu_fwd.argtypes = [vp, vp, i64, i32, vp]
        lib.bimamba_gelu_bwd.restype = i32
        lib.bimamba_gelu_bwd.argtypes = [vp, vp, vp, i64, i32, vp]
        lib.bimamba_reduce_rows32.restype = i32
        lib.bimamba_reduce_rows32.argtypes = [vp, vp, i64, i32, i64, i64, i32, vp]
        lib.bimamba_finalize_param_grads.restype = i32
        lib.bimamba_finalize_param_grads.argtypes = [vp] * 12 + [i32] * 6 + [vp]
        lib.bimamba_head_pool_bwd.restype = i32
        lib.bimamba_head_pool_bwd.argtypes = [vp, vp, vp, vp, vp, vp, vp, vp, i32, i32, i32, C.c_float, i32, vp]
        lib.bimamba_set_tuning.restype = i32
        lib.bimamba_set_tuning.argtypes = [i32, i32]
        lib.bimamba_get_tuning.restype = i32
        lib.bimamba_get_tuning.argtypes = [i32]
        lib.bimamba_scan_fwd_workspace_bytes.restype = C.c_size_t
        lib.bimamba_scan_fwd_workspace_bytes.argtypes = [i32, i32, i32, i32, i32, i32]
        lib.bimamba_scan_bwd_workspace_bytes.restype = C.c_size_t
        lib.bimamba_scan_bwd_workspace_bytes.argtypes = [i32, i32, i32, i32]
        lib.bimamba_split3_bf16.restype = i32
        lib.bimamba_split3_bf16.argtypes = [vp, vp, i64, i32, i64, i64, i64, i32, vp]
        lib.bimamba_cast.restype = i32
        lib.bimamba_cast.argtypes = [vp, vp, i64, i32, i32, vp]
        lib.bimamba_sumsq_slices.restype = i32
        lib.bimamba_sumsq_slices.argtypes = [i64]
        lib.bimamba_sumsq.restype = i32
        lib.bimamba_sumsq.argtypes = [vp, vp, i64, C.c_float, i32, vp]
        lib.bimamba_scale_by.restype = i32
        lib.bimamba_scale_by.argtypes = [vp, vp, vp, i64, C.c_float, i32, vp]
        lib.bimamba_block_fwd_workspace_bytes.restype = C.c_size_t
        lib.bimamba_block_fwd_workspace_bytes.argtypes = [i32] * 7
        lib.bimamba_block_bwd_workspace_bytes.restype = C.c_size_t
        lib.bimamba_block_bwd_workspace_bytes.argtypes = [i32] * 7
        lib.bimamba_block_fwd.restype = i32
        lib.bimamba_block_fwd.argtypes = [C.POINTER(BlockDesc), vp]
        lib.bimamba_block_fwd_varlen.restype = i32
        lib.bimamba_block_fwd_varlen.argtypes = [C.POINTER(BlockDesc), vp, vp]
        lib.bimamba_block_bwd.restype = i32
        lib.bimamba_block_bwd.argtypes = [C.POINTER(BlockDesc), C.POINTER(BlockGrads), vp]
        lib.bimamba_scan_fwd_split_plan.restype = i32
        lib.bimamba_scan_fwd_split_plan.argtypes = [i32, i32, i32, i32, i32, C.POINTER(i32), C.POINTER(i32)]
        lib.bimamba_scan_fwd_split_workspace_bytes.restype = C.c_size_t
        lib.bimamba_scan_fwd_split_workspace_bytes.argtypes = [i32, i32, i32, i32]
        lib.bimamba_selective_scan_fwd_split.restype = i32
        lib.bimamba_selective_scan_fwd_split.argtypes = [C.POINTER(ScanDesc), i32, i32, vp, C.c_size_t, vp]
        lib.bimamba_layer_fwd_workspace_bytes.restype = C.c_size_t
        lib.bimamba_layer_fwd_workspace_bytes.argtypes = [i32] * 8
        lib.bimamba_layer_bwd_workspace_bytes.restype = C.c_size_t
        lib.bimamba_layer_bwd_workspace_bytes.argtypes = [i32] * 8
        lib.bimamba_layer_fwd.restype = i32
        lib.bimamba_layer_fwd.argtypes = [C.POINTER(LayerDesc), vp]
        lib.bimamba_layer_fwd_varlen.restype = i32
        lib.bimamba_layer_fwd_varlen.argtypes = [C.POINTER(LayerDesc), vp, vp]
        lib.bimamba_layer_bwd.restype = i32
        lib.bimamba_layer_bwd.argtypes = [C.POINTER(LayerDesc), C.POINTER(LayerGrads), vp]
        for name in ("bimamba_selective_scan_fwd_varlen_train", "bimamba_selective_scan_bwd_varlen"):
            fn = getattr(lib, name)
            fn.restype = i32
            fn.argtypes = [C.POINTER(ScanDesc), vp, vp]
        lib.bimamba_causal_conv1d_bwd_varlen.restype = i32
        lib.bimamba_causal_conv1d_bwd_varlen.argtypes = [vp, vp, vp, vp, vp, vp, vp, vp, vp, i32, i32, i32, i32, i32,
                                                         i64, i64, i64, i64, i64, i64, i64, i32, i32, vp]
        lib.bimamba_head_pool_bwd_varlen.restype = i32
        lib.bimamba_head_pool_bwd_varlen.argtypes = [vp, vp, vp, vp, vp, vp, vp, vp, vp, i32, i32, i32, C.c_float, i32, vp]
        lib.bimamba_block_fwd_varlen_train.restype = i32
        lib.bimamba_block_fwd_varlen_train.argtypes = [C.POINTER(BlockDesc), vp, vp]
        lib.bimamba_block_bwd_varlen.restype = i32
        lib.bimamba_block_bwd_varlen.argtypes = [C.POINTER(BlockDesc), C.POINTER(BlockGrads), vp, vp]
        lib.bimamba_layer_fwd_varlen_train.restype = i32
        lib.bimamba_layer_fwd_varlen_train.argtypes = [C.POINTER(LayerDesc), vp, vp]
        lib.bimamba_layer_bwd_varlen.restype = i32
        lib.bimamba_layer_bwd_varlen.argtypes = [C.POINTER(LayerDesc), C.POINTER(LayerGrads), vp, vp]
        lib.bimamba_block_bwd_side.restype = i32
        lib.bimamba_block_bwd_side.argtypes = [C.POINTER(BlockDesc), C.POINTER(BlockGrads), vp, C.POINTER(SideStream), vp]
        lib.bimamba_layer_fwd_side.restype = i32
        lib.bimamba_layer_fwd_side.argtypes = [C.POINTER(LayerDesc), C.POINTER(BlockPack), vp, C.POINTER(SideStream), vp]
        lib.bimamba_layer_bwd_side.restype = i32
        lib.bimamba_layer_bwd_side.argtypes = [C.POINTER(LayerDesc), C.POINTER(LayerGrads), vp, C.POINTER(SideStream), vp]
        lib.bimamba_mask_frames.restype = i32
        lib.bimamba_mask_frames.argtypes = [vp, vp, vp, i32, i32, i32, i32, vp]
        lib.bimamba_mixup_frames.restype = i32
        lib.bimamba_mixup_frames.argtypes = [vp, vp, vp, vp, vp, vp, i32, i32, i32, i32, vp]
        for name in ("bimamba_interp_frames_fwd", "bimamba_interp_frames_bwd"):
            fn = getattr(lib, name)
            fn.restype = i32
            fn.argtypes = [vp, vp, vp, vp, i32, i32, i32, i32, i32, vp]
        lib.bimamba_frame_mean.restype = i32
        lib.bimamba_frame_mean.argtypes = [vp, vp, vp, i32, i32, i32, i32, vp]
        lib.bimamba_frame_mean_bwd.restype = i32
        lib.bimamba_frame_mean_bwd.argtypes = [vp, vp, vp, i32, i32, i32, i32, vp]
        lib.bimamba_frame_scale.restype = i32
        lib.bimamba_frame_scale.argtypes = [vp, vp, vp, vp, i32, i32, i32, i32, vp]
        lib.bimamba_frame_scale_bwd_slices.restype = i32
        lib.bimamba_frame_scale_bwd_slices.argtypes = [i32]
        lib.bimamba_frame_scale_bwd.restype = i32
        lib.bimamba_frame_scale_bwd.argtypes = [vp, vp, vp, vp, vp, vp, i32, i32, i32, i32, vp]
        got = lib.bimamba_abi_version()
        if got != ABI_VERSION:
            raise RuntimeError(f"libbimamba ABI {got} != expected {ABI_VERSION}; rebuild the library")
        _lib = lib
    return _lib


def check(rc: int, what: str) -> None:
    global launch_count
    if rc != 0:
        msg = load().bimamba_last_error().decode("utf-8", "replace")
        raise RuntimeError(f"{what} failed (code {rc}): {msg}")
    launch_count += 1


def scan_split_plan(batch: int, ndir: int, seqlen: int, dim: int, io_dtype: int = BF16):
    """-> (nseg, seg_len) of the time-parallel forward scan; nseg == 1: do not split."""
    ns, sl = C.c_int(1), C.c_int(0)
    load().bimamba_scan_fwd_split_plan(int(batch), int(ndir), int(seqlen), int(dim), int(io_dtype), C.byref(ns), C.byref(sl))
    return ns.value, sl.value


def scan_plan(seqlen: int, dim: int, rows: int, backward: bool = False):
    """-> (group_channels, ngroups, nchunks)"""
    gc, ng = C.c_int(0), C.c_int(0)
    n = load().bimamba_scan_plan(int(seqlen), int(dim), int(rows), int(backward), C.byref(gc), C.byref(ng))
    g = gc.value
    return g, (dim + g - 1) // g, n


TUNE_SCAN_FWD, TUNE_CONV_BWD, TUNE_GEMM_KERNEL, TUNE_GEMM_BN, TUNE_GEMM_STAGES, TUNE_PDL, TUNE_SCAN_SPLIT = range(7)


class tuning:
    """Context manager that forces a kernel variant (parity tests of every shipped variant, tuning experiments):
    `with tuning(TUNE_SCAN_FWD, 1): ...`.  0 = automatic choice."""

    def __init__(self, knob: int, value: int):
        self.knob, self.value = knob, value

    def __enter__(self):
        lib = load()
        self.old = lib.bimamba_get_tuning(self.knob)
        if lib.bimamba_set_tuning(self.knob, self.value) != 0:
            raise RuntimeError("bimamba_set_tuning: unknown knob")
        return self

    def __exit__(self, *a):
        load().bimamba_set_tuning(self.knob, self.old)
        return False
