"""ctypes binding of liblfsr_b200.so (C ABI declared in include/lfsr.h).

There is deliberately no fallback: if the shared library is missing or a CUDA device is not
present the product path raises. Build it with ``python -c "import __graft_entry__ as g; g.build()"``
(or ``make -C <package>/csrc``).
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

_PKG_DIR = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_PKG_DIR, "liblfsr_b200.so")
#: measurement scripts under profiles/ set LFSR_PROBE_LIB=1 to load the probe build instead: the same kernels compiled with
#: -DLFSR_DEBUG_HOOKS (cycle counters, LFSR_TC_* experiment switches) plus the rate probes of csrc/lfsr_debug.cu
PROBE_LIB_PATH = os.path.join(_PKG_DIR, "liblfsr_probe.so")
CSRC_DIR = os.path.join(_PKG_DIR, "csrc")

ACT_NONE, ACT_RELU, ACT_LRELU, ACT_SIGMOID, ACT_GELU, ACT_SILU = 0, 1, 2, 3, 4, 5
PERM_NONE, PERM_MACPI_OVER_SAI = 0, 1
SHUF_CHANNEL_MAJOR, SHUF_FACTOR_MAJOR = 0, 1
INTERP_BICUBIC, INTERP_BILINEAR = 0, 1
OUT_F32, OUT_BOTH, OUT_F16 = 0, 1, 2       # lfsr_conv_desc.out_mode


class LfsrError(RuntimeError):
    pass


class Tensor(C.Structure):
    _fields_ = [("ptr", C.c_void_p), ("n", C.c_int32), ("h", C.c_int32), ("w", C.c_int32),
                ("c", C.c_int32), ("ld", C.c_int32)]


class ConvDesc(C.Structure):
    _fields_ = [
        ("kh", C.c_int32), ("kw", C.c_int32), ("stride_h", C.c_int32), ("stride_w", C.c_int32),
        ("dil_h", C.c_int32), ("dil_w", C.c_int32), ("pad_h", C.c_int32), ("pad_w", C.c_int32),
        ("in_perm", C.c_int32), ("out_perm", C.c_int32), ("perm_a", C.c_int32),
        ("shuf_ry", C.c_int32), ("shuf_rx", C.c_int32), ("shuf_mode", C.c_int32),
        ("block_h", C.c_int32), ("block_w", C.c_int32),
        ("act", C.c_int32), ("act_slope", C.c_float), ("alpha", C.c_float), ("mul_act", C.c_int32),
        ("bias", C.c_void_p), ("in_scale", C.c_void_p), ("in_scale_ld", C.c_int64), ("w_batch_stride", C.c_int64),
        ("mul", Tensor), ("res", Tensor),
        ("tail_w", C.c_void_p), ("tail_taps", C.c_int32), ("tail_c", C.c_int32),
        ("in_f16", C.c_int32), ("out_mode", C.c_int32), ("out16", Tensor),
    ]


class DwBranch(C.Structure):
    _fields_ = [("w", C.c_void_p), ("scale", C.c_void_p), ("shift", C.c_void_p),
                ("kh", C.c_int32), ("kw", C.c_int32), ("dil_h", C.c_int32), ("dil_w", C.c_int32),
                ("in_c0", C.c_int32), ("out_c0", C.c_int32), ("c", C.c_int32),
                ("act", C.c_int32), ("act_slope", C.c_float)]


class EpiAttnDesc(C.Structure):
    _fields_ = [
        ("heads", C.c_int32), ("head_dim", C.c_int32), ("A", C.c_int32), ("S", C.c_int32),
        ("half_window", C.c_int32), ("nb", C.c_int32), ("np", C.c_int32), ("nq", C.c_int32),
        ("stride_a", C.c_int64), ("stride_s", C.c_int64), ("stride_b", C.c_int64),
        ("stride_p", C.c_int64), ("stride_q", C.c_int64),
    ]


class BasicTransDesc(C.Structure):
    _fields_ = [
        ("A", C.c_int32), ("S", C.c_int32), ("half_window", C.c_int32), ("heads", C.c_int32), ("E", C.c_int32), ("C", C.c_int32),
        ("nb", C.c_int32), ("np", C.c_int32), ("nq", C.c_int32),
        ("stride_a", C.c_int64), ("stride_s", C.c_int64), ("stride_b", C.c_int64), ("stride_p", C.c_int64),
        ("stride_q", C.c_int64),
        ("eps1", C.c_float), ("eps2", C.c_float),
        ("ln1_g", C.c_float * 128), ("ln1_b", C.c_float * 128), ("ln2_g", C.c_float * 128), ("ln2_b", C.c_float * 128),
    ]


# name -> (restype, argtypes); mirrors include/lfsr.h one to one (tests check the export list)
_P = C.c_void_p
_I = C.c_int
_TP = C.POINTER(Tensor)
SIGNATURES = {
    "lfsr_last_error": (C.c_char_p, []),
    "lfsr_abi_version": (_I, []),
    "lfsr_built_for_sm100a": (_I, []),
    "lfsr_launch_count": (C.c_uint64, []),
    "lfsr_conv_tc_lean_count": (C.c_uint64, []),
    "lfsr_divide": (_I, [_P, _P, _I, _I, _I, _I, _I, _P]),
    "lfsr_divide_rows": (_I, [_P, _P, _I, _I, _I, _I, _I, _I, _I, _P]),
    "lfsr_integrate_rows": (_I, [_P, _P, _I, _I, _I, _I, _I, _I, _I, _I, _I, _P]),
    "lfsr_divide_rows_d8": (_I, [_P, _P, _I, _I, _I, _I, _I, _I, _I, _P]),
    "lfsr_integrate_rows_d8": (_I, [_P, _P, _I, _I, _I, _I, _I, _I, _I, _I, _I, _P]),
    "lfsr_interp": (_I, [_P, _P, _I, _I, _I, _I, _I, _I, _I, _P]),
    "lfsr_ycbcr_to_rgb8": (_I, [_P, _P, _P, _P, _I, _I, _I, _P, _P, _P]),
    "lfsr_ycbcr_to_rgb8_uv": (_I, [_P, _P, _P, _P, _I, _I, _I, _I, _P, _P, _P]),
    "lfsr_resample_f64": (_I, [_P, _P, _P, _P, _I, _I, _I, _I, _I, _P]),
    "lfsr_rgb_to_ycbcr_mosaic": (_I, [_P, _I, _P, _P, _P, _I, _I, _I, _P]),
    "lfsr_rgb_to_ycbcr_mosaic_uv": (_I, [_P, _I, _P, _P, _P, _I, _I, _I, _I, _P]),
    "lfsr_window_accumulate": (_I, [_P, _P, _I, _I, _I, _I, _I, _I, _P, _P]),
    "lfsr_window_accumulate_uv": (_I, [_P, _P, _I, _I, _I, _I, _I, _I, _I, _P, _P]),
    "lfsr_conv2d_f32": (_I, [_TP, _P, _TP, C.POINTER(ConvDesc), _P]),
    "lfsr_dwconv_f32": (_I, [_TP, _P, _P, _P, _TP, _I, _I, _I, _I, _I, C.c_float, _P]),
    "lfsr_dwconv_multi": (_I, [_TP, _TP, C.POINTER(DwBranch), _I, _P]),
    "lfsr_tap_gather": (_I, [_TP, _I, _I, _P, _TP, _TP, _P]),
    "lfsr_conv2d_stem_supported": (_I, [_TP, _TP, C.POINTER(ConvDesc)]),
    "lfsr_conv2d_stem": (_I, [_TP, _P, _TP, C.POINTER(ConvDesc), _P]),
    "lfsr_conv2d_thin_supported": (_I, [_TP, _TP, C.POINTER(ConvDesc)]),
    "lfsr_conv2d_thin": (_I, [_TP, _P, _TP, C.POINTER(ConvDesc), _P]),
    "lfsr_conv1x1_few_supported": (_I, [_TP, _TP, C.POINTER(ConvDesc)]),
    "lfsr_conv1x1_few": (_I, [_TP, _P, _TP, C.POINTER(ConvDesc), _P]),
    "lfsr_conv2d_small_cout_supported": (_I, [_TP, _TP, C.POINTER(ConvDesc)]),
    "lfsr_conv2d_small_cout": (_I, [_TP, _P, _TP, C.POINTER(ConvDesc), _P]),
    "lfsr_mel_epi_branch": (_I, [_TP, _P, _TP, _I, _I, C.c_float, _P]),
    "lfsr_mel_epi_branch_tc": (_I, [_TP, _P, _TP, _I, _I, C.c_float, _P]),
    "lfsr_mel_epi_pack_bytes": (C.c_size_t, [_I]),
    "lfsr_mel_epi_pack": (_I, [_P, _P, _I]),
    "lfsr_mel_epi_branch_mma": (_I, [_TP, _TP, _P, _TP, _I, _I, C.c_float, _P]),
    "lfsr_conv2d_tc_packed_floats": (C.c_size_t, [_I, _I, _I, _I]),
    "lfsr_pack_conv_tc": (_I, [_P, _P, _I, _I, _I, _I]),
    "lfsr_to_f16": (_I, [_TP, _TP, _P]),
    "lfsr_split_tf32": (_I, [_P, _P, _P, C.c_longlong, _P]),
    "lfsr_macpi_unshuffle": (_I, [_TP, _P, _I, _I, _I, _P]),
    "lfsr_conv2d_tc16_packed_bytes": (C.c_size_t, [_I, _I, _I, _I]),
    "lfsr_pack_conv_tc16": (_I, [_P, _P, _I, _I, _I, _I]),
    "lfsr_scale_pack_tc": (_I, [_P, _P, C.c_int64, _P, _I, _I, _I, _I, _I, _P]),
    "lfsr_conv2d_tc": (_I, [_TP, _P, _TP, C.POINTER(ConvDesc), _P]),
    "lfsr_conv2d_tc_supported": (_I, [_TP, _TP, C.POINTER(ConvDesc)]),
    "lfsr_block_mean": (_I, [_TP, _TP, _I, _I, _P]),
    "lfsr_pooled_mlp": (_I, [_TP, _I, _P, _P, _I, _I, _P, _P, _I, _I, _TP, _P]),
    "lfsr_ang_expand": (_I, [_TP, _P, _TP, _TP, _I, _I, C.c_float, C.c_float, _P]),
    "lfsr_sa_modulate": (_I, [_TP, _P, _P, _P, _TP, C.c_float, C.c_float, _TP, _TP, _I, _P]),
    "lfsr_sa_modulate16": (_I, [_TP, _P, _P, _P, _TP, C.c_float, C.c_float, _TP, _TP, _TP, _I, _P]),
    "lfsr_sa_modulate16w": (_I, [_TP, _P, _P, _P, _TP, C.c_float, C.c_float, _TP, _TP, _TP, _I, _I, _I, _P]),
    "lfsr_scale_add": (_I, [_TP, _TP, _TP, _TP, _P]),
    "lfsr_scale_add16": (_I, [_TP, _TP, _TP, _TP, _P]),
    "lfsr_layernorm": (_I, [_TP, _P, _P, C.c_float, _TP, _P]),
    "lfsr_epi_attention": (_I, [_P, _P, _P, C.POINTER(EpiAttnDesc), _P]),
    "lfsr_basictrans_packed_bytes": (C.c_size_t, []),
    "lfsr_pack_basictrans": (_I, [_P, _P, _P, _P, _P, _P, _P]),
    "lfsr_basictrans_supported": (_I, [_TP, _TP, C.POINTER(BasicTransDesc)]),
    "lfsr_epit_basictrans": (_I, [_TP, _P, _TP, C.POINTER(BasicTransDesc), _P]),
    "lfsr_metric_sums": (_I, [_P, _P, _I, _I, _I, _P, _P]),
    "lfsr_metric_sums_batched": (_I, [_P, _P, _I, _I, _I, _I, _P, _P]),
    "lfsr_metric_sums_uv": (_I, [_P, _P, _I, _I, _I, _I, _P, _P]),
}

_lib = None


def build_native(verbose: bool = False) -> str:
    """Compile csrc/*.cu for sm_100a into liblfsr_b200.so (nvcc cross-compiles without a GPU)."""
    proc = subprocess.run(["make", "-C", CSRC_DIR, "-j", str(os.cpu_count() or 4)], capture_output=True, text=True)
    if verbose or proc.returncode != 0:
        print(proc.stdout)
        print(proc.stderr)
    if proc.returncode != 0:
        raise LfsrError("nvcc build of liblfsr_b200.so failed")
    return LIB_PATH


def load():
    """Return the loaded library; raise loudly when it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    path = PROBE_LIB_PATH if os.environ.get("LFSR_PROBE_LIB") == "1" else LIB_PATH
    if not os.path.exists(path):
        raise LfsrError(
            f"{path} is missing: the sm_100a CUDA extension has not been built "
            "(run __graft_entry__.build()); there is no CPU fallback for this path")
    lib = C.CDLL(path)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if the export is missing - intended
        fn.restype = res
        fn.argtypes = args
    if lib.lfsr_abi_version() != 1:
        raise LfsrError("liblfsr_b200.so ABI version mismatch; rebuild")
    _lib = lib
    return lib


def check(status: int, what: str) -> None:
    if status != 0:
        msg = load().lfsr_last_error().decode("utf-8", "replace")
        raise LfsrError(f"{what} failed ({status}): {msg}")
