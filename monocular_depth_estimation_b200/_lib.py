"""ctypes binding of libcrf_sm100.so (C ABI declared in include/crf_sm100.h).

The library is the product: there is no CPU or PyTorch fallback.  `lib()` raises if the shared object has not been
built (run `python -c "import __graft_entry__ as g; g.build()"` or `make -C monocular_depth_estimation_b200/csrc`).
"""
from __future__ import annotations

import ctypes as C
import os
import threading

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "csrc", "libcrf_sm100.so")

CRF_DT_F32 = 0
CRF_DT_BF16 = 1

PREC_BF16, PREC_FP32 = 0, 1   # crf_block_desc.precision (BASELINE.json: rel 2e-2 / rel 1e-3 tiers)
EPI_STORE_F32 = 0
EPI_STORE_BF16 = 1
EPI_BIAS_RES_F32 = 2
EPI_BIAS_GELU = 3
EPI_MUL_DGELU = 4
EPI_SPLITK_F32 = 5

ACT_NONE, ACT_RELU, ACT_HARDSWISH = 0, 1, 2   # crf_bn_fwd / crf_bn_bwd activation

# every symbol include/crf_sm100.h declares (checked by tests/test_abi.py)
EXPORTED_SYMBOLS = (
    "crf_last_error", "crf_abi_version", "crf_kernel_launches", "crf_timing_enable", "crf_timing_report", "crf_block_sizes", "crf_block_fwd", "crf_block_bwd", "crf_convert_v",
    "crf_layer_sizes", "crf_layer_fwd", "crf_layer_bwd",
    "crf_window_gather", "crf_window_scatter", "crf_shift_mask", "crf_gemm", "crf_mlp_fwd", "crf_gemm_workspace_bytes", "crf_ln_fwd", "crf_ln_bwd", "crf_dgrad_ln_bwd",
    "crf_layernorm_fwd", "crf_layernorm_bwd", "crf_layernorm_ps_fwd", "crf_layernorm_ps_bwd", "crf_depth_loss_fwd", "crf_depth_loss_bwd", "crf_pixel_shuffle_nhwc",
    "crf_colsum_bf16", "crf_cast_bf16", "crf_attn_fwd", "crf_attn_bwd", "crf_adam_step",
    "crf_bn_workspace_bytes", "crf_bn_fwd", "crf_bn_bwd",
)


class AdamTensor(C.Structure):          # include/crf_sm100.h: crf_adam_tensor
    _fields_ = [("p", C.c_void_p), ("g", C.c_void_p), ("m", C.c_void_p), ("v", C.c_void_p), ("n", C.c_int64)]


class BlockDesc(C.Structure):
    _fields_ = [
        ("B", C.c_int32), ("H", C.c_int32), ("W", C.c_int32), ("C", C.c_int32),
        ("num_heads", C.c_int32), ("window", C.c_int32), ("shift", C.c_int32),
        ("training", C.c_int32), ("device", C.c_int32),
        ("x_dtype", C.c_int32), ("v_dtype", C.c_int32), ("v_preconverted", C.c_int32),
        ("x_stride_b", C.c_int64), ("x_stride_t", C.c_int64), ("x_stride_c", C.c_int64),
        ("v_stride_b", C.c_int64), ("v_stride_h", C.c_int64), ("v_stride_w", C.c_int64), ("v_stride_c", C.c_int64),
        ("precision", C.c_int32), ("reserved", C.c_int32),
    ]


PARAM_NAMES = ("norm1_w", "norm1_b", "qk_w", "qk_b", "rpb_table", "proj_w", "proj_b", "norm2_w", "norm2_b",
               "fc1_w", "fc1_b", "fc2_w", "fc2_b")


class BlockParams(C.Structure):
    _fields_ = ([(n, C.c_void_p) for n in PARAM_NAMES] + [("qk_scale", C.c_float), ("ln_eps", C.c_float)]
                + [("ext_mask", C.c_void_p), ("ext_mask_windows", C.c_int32), ("reserved", C.c_int32)])


class BlockGrads(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in PARAM_NAMES]


class LayerArgs(C.Structure):
    _fields_ = [("depth", C.c_int32), ("out_dtype", C.c_int32), ("params", C.POINTER(BlockParams)),
                ("norm_w", C.c_void_p), ("norm_b", C.c_void_p), ("out_shuffle", C.c_int32)]


class GemmArgs(C.Structure):
    _fields_ = [
        ("A", C.c_void_p), ("B", C.c_void_p),
        ("a_major", C.c_int32), ("b_major", C.c_int32),
        ("M", C.c_int32), ("N", C.c_int32), ("K", C.c_int32),
        ("epilogue", C.c_int32), ("split_k", C.c_int32),
        ("out0", C.c_void_p), ("out1", C.c_void_p),
        ("bias", C.c_void_p), ("aux1", C.c_void_p),
        ("ld_out", C.c_int64),
        ("scale", C.c_float), ("scale_cols", C.c_int32),
        ("device", C.c_int32),
        ("workspace", C.c_void_p), ("workspace_bytes", C.c_size_t),
        ("colsum", C.c_void_p),
        ("split3", C.c_int32),
    ]


class MlpArgs(C.Structure):              # include/crf_sm100.h: crf_mlp_args
    _fields_ = [
        ("x1", C.c_void_p), ("y", C.c_void_p),
        ("w1_bf16", C.c_void_p), ("w2_bf16", C.c_void_p),
        ("b1", C.c_void_p), ("b2", C.c_void_p), ("norm_w", C.c_void_p), ("norm_b", C.c_void_p),
        ("xn2", C.c_void_p), ("stats", C.c_void_p), ("pre", C.c_void_p), ("act", C.c_void_p),
        ("eps", C.c_float),
        ("T", C.c_int32), ("C", C.c_int32), ("training", C.c_int32), ("device", C.c_int32),
    ]


_lock = threading.Lock()
_lib = None


def _declare(lib):
    vp, i32, i64, f32, f64, sz = C.c_void_p, C.c_int, C.c_int64, C.c_float, C.c_double, C.c_size_t
    lib.crf_last_error.restype = C.c_char_p
    lib.crf_last_error.argtypes = []
    lib.crf_abi_version.restype = i32
    lib.crf_abi_version.argtypes = []
    lib.crf_block_sizes.argtypes = [C.POINTER(BlockDesc), C.POINTER(sz), C.POINTER(sz), C.POINTER(sz)]
    lib.crf_block_fwd.argtypes = [C.POINTER(BlockDesc), C.POINTER(BlockParams), vp, vp, vp, vp, vp, sz, vp]
    lib.crf_block_bwd.argtypes = [C.POINTER(BlockDesc), C.POINTER(BlockParams), vp, vp, vp, vp, vp, vp, i32,
                                  C.POINTER(BlockGrads), vp, sz, vp]
    lib.crf_convert_v.argtypes = [C.POINTER(BlockDesc), vp, vp, vp]
    lib.crf_layer_sizes.argtypes = [C.POINTER(BlockDesc), i32, i32, C.POINTER(sz), C.POINTER(sz)]
    lib.crf_layer_fwd.argtypes = [C.POINTER(BlockDesc), C.POINTER(LayerArgs), vp, vp, vp, vp, vp]
    lib.crf_layer_bwd.argtypes = [C.POINTER(BlockDesc), C.POINTER(LayerArgs), vp, vp, vp, vp, vp, vp,
                                  C.POINTER(BlockGrads), vp, vp, vp, sz, vp]
    lib.crf_window_gather.argtypes = [vp, vp, i32, i32, i32, i32, i32, i32, vp]
    lib.crf_window_scatter.argtypes = [vp, vp, i32, i32, i32, i32, i32, i32, vp]
    lib.crf_shift_mask.argtypes = [vp, i32, i32, i32, i32, vp]
    lib.crf_gemm.argtypes = [C.POINTER(GemmArgs), vp]
    lib.crf_mlp_fwd.argtypes = [C.POINTER(MlpArgs), vp]
    lib.crf_gemm_workspace_bytes.restype = sz
    lib.crf_gemm_workspace_bytes.argtypes = [i32, i32, i32, i32]
    lib.crf_ln_fwd.argtypes = [vp, i32, i64, i64, i64, i32, i32, i32, vp, vp, f32, vp, vp, vp, i32, vp]
    lib.crf_ln_bwd.argtypes = [vp, vp, vp, vp, vp, vp, vp, vp, vp, i32, i32, i32, vp]
    lib.crf_dgrad_ln_bwd.argtypes = [vp, vp, i32, vp, vp, vp, vp, vp, vp, vp, vp, i32, i32, i32, vp]
    lib.crf_layernorm_fwd.argtypes = [vp, vp, vp, f32, vp, i32, vp, i32, i32, i32, vp]
    lib.crf_layernorm_bwd.argtypes = [vp, i32, vp, vp, vp, vp, vp, vp, i32, i32, i32, vp]
    lib.crf_layernorm_ps_fwd.argtypes = [vp, vp, vp, f32, vp, i32, vp, i32, i32, i32, i32, i32, vp]
    lib.crf_layernorm_ps_bwd.argtypes = [vp, i32, vp, vp, vp, vp, vp, vp, i32, i32, i32, i32, i32, vp]
    lib.crf_depth_loss_fwd.argtypes = [vp, i32, vp, i32, i32, i32, vp, vp, i32, vp]
    lib.crf_depth_loss_bwd.argtypes = [vp, i32, vp, vp, vp, i32, i32, i32, vp, i32, vp]
    lib.crf_pixel_shuffle_nhwc.argtypes = [vp, vp, i32, i32, i32, i32, i32, i32, i32, vp]
    lib.crf_colsum_bf16.argtypes = [vp, vp, i32, i32, i32, vp]
    lib.crf_cast_bf16.argtypes = [vp, vp, i64, i32, vp]
    lib.crf_adam_step.argtypes = [C.POINTER(AdamTensor), i32, i32, f64, f64, f64, f64, f64, vp, i32, vp]
    lib.crf_attn_fwd.argtypes = [C.POINTER(BlockDesc), vp, vp, vp, f32, vp, vp, i32, vp, vp, vp]
    lib.crf_attn_bwd.argtypes = [C.POINTER(BlockDesc), vp, vp, vp, f32, vp, vp, i32, vp, vp, vp, vp, i32, vp, vp, vp]
    lib.crf_bn_workspace_bytes.restype = sz
    lib.crf_bn_workspace_bytes.argtypes = [i32, i32, i32]
    lib.crf_bn_fwd.argtypes = [vp, vp, vp, vp, vp, vp, vp, vp, vp, i32, i32, f32, f32, i32, vp, sz, vp, i32, vp]
    lib.crf_bn_bwd.argtypes = [vp, vp, vp, vp, vp, vp, vp, vp, vp, i32, i32, i32, vp, sz, vp, i32, vp]
    for name in EXPORTED_SYMBOLS:
        if name not in ("crf_last_error", "crf_kernel_launches", "crf_timing_report", "crf_gemm_workspace_bytes",
                        "crf_bn_workspace_bytes"):
            getattr(lib, name).restype = i32
    lib.crf_kernel_launches.restype = C.c_longlong
    lib.crf_kernel_launches.argtypes = []
    lib.crf_timing_enable.argtypes = [i32]
    lib.crf_timing_report.restype = sz
    lib.crf_timing_report.argtypes = [C.c_char_p, sz]


def lib():
    """Load (once) and return the C-ABI library.  Raises RuntimeError if it is missing -- no fallback exists."""
    global _lib
    if _lib is None:
        with _lock:
            if _lib is None:
                if not os.path.exists(LIB_PATH):
                    raise RuntimeError(
                        f"{LIB_PATH} is missing: the sm_100a CUDA extension has not been built "
                        "(python -c 'import __graft_entry__ as g; g.build()'). There is no CPU/PyTorch fallback.")
                handle = C.CDLL(LIB_PATH)
                _declare(handle)
                _lib = handle
    return _lib


def check(rc: int, what: str) -> None:
    if rc != 0:
        msg = lib().crf_last_error().decode("utf-8", "replace")
        raise RuntimeError(f"{what} failed: {msg}")
