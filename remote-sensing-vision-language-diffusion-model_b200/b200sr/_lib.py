"""ctypes binding of libb200sr.so (the C ABI declared in include/b200sr.h).

The shared library is built in-tree by ``csrc/build.sh`` (or ``__graft_entry__.build()``) and
lives next to this file.  There is deliberately no fallback: if the library is missing or an
entry point is absent, importing/using the ops raises.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
# B200SR_LIB selects another in-tree build of the same ABI (A/B kernel experiments); default = the product library
LIB_PATH = os.path.join(_HERE, os.environ.get("B200SR_LIB", "libb200sr.so"))

ABI_VERSION = 8

c_void_p, c_int, c_i64, c_float, c_size_t = C.c_void_p, C.c_int32, C.c_int64, C.c_float, C.c_size_t


class Epilogue(C.Structure):
    """Mirror of ``b200sr_epilogue`` (include/b200sr.h)."""

    _fields_ = [
        ("bias", c_void_p),
        ("rowvec", c_void_p),
        ("rows_per_group", c_int),
        ("ld_rowvec", c_i64),
        ("residual", c_void_p),
        ("ldr", c_i64),
        ("out", c_void_p),
        ("ldc", c_i64),
        ("out_fp32", c_int),
        ("geglu", c_int),
        ("alpha", c_float),
        ("act", c_int),
        ("softmax_valid", c_int),
        ("w_dynamic", c_int),
        ("w_rows_per_group", c_int),
        ("w_group_stride", c_i64),
        ("a_gn_stats", c_void_p),
        ("a_gn_weight", c_void_p),
        ("a_gn_bias", c_void_p),
        ("a_gn_groups", c_int),
        ("a_gn_silu", c_int),
        ("ln_stats", c_void_p),
        ("ln_parts", c_int),
        ("ln_colsum", c_void_p),
        ("ln_shift", c_void_p),
        ("ln_eps", c_float),
        ("ln_stats_out", c_void_p),
        ("row_softmax", c_int),
        ("row_softmax_valid", c_int),
    ]


class Copy(C.Structure):
    """Mirror of ``b200sr_copy``."""

    _fields_ = [("src", c_void_p), ("dst", c_void_p), ("bytes", c_i64)]


def binding_snippet() -> str:
    """The struct declarations of this binding as the ctypes source a maintainer would paste (INTEGRATION.md
    section 1 embeds exactly this text; tests/test_abi_cpu.py diffs the two so the document cannot go stale)."""
    names = {c_void_p: "C.c_void_p", c_int: "C.c_int32", c_i64: "C.c_int64", c_float: "C.c_float"}
    out = []
    for cls, cname in ((Epilogue, "b200sr_epilogue"), (Copy, "b200sr_copy")):
        out.append(f"class {cls.__name__}(C.Structure):  # {cname} (ABI version {ABI_VERSION})")
        out.append("    _fields_ = [")
        for fname, ftype in cls._fields_:
            out.append(f'        ("{fname}", {names[ftype]}),')
        out.append("    ]")
        out.append("")
    return "\n".join(out).rstrip() + "\n"


P = c_void_p
# name -> (restype, argtypes); must list every symbol include/b200sr.h declares.
SIGNATURES = {
    "b200sr_abi_version": (c_int, []),
    "b200sr_num_sms": (c_int, []),
    "b200sr_gemm_bf16": (c_int, [P, c_i64, P, c_int, c_int, c_int, C.POINTER(Epilogue), c_int, P]),
    "b200sr_gemm_n_tile": (c_int, [c_int, c_int, c_int]),
    "b200sr_row_softmax_fold": (c_int, [P, c_int, c_i64, P, P]),
    "b200sr_conv3x3_bf16": (c_int, [P, P, c_int, c_int, c_int, c_int, c_int, c_int, c_int, C.POINTER(Epilogue), c_int, P]),
    "b200sr_pointwise_small": (c_int, [P, P, P, P, c_int, c_int, c_i64, c_int, c_int, c_float, P]),
    "b200sr_diag_gaussian": (c_int, [P, P, P, c_int, c_int, c_int, c_float, P]),
    "b200sr_group_norm_workspace_bytes": (c_size_t, [c_int, c_int, c_int, c_int]),
    "b200sr_group_norm_launches": (c_int, [c_int, c_int, c_int, c_int]),
    "b200sr_group_norm_nhwc": (
        c_int,
        [P, P, P, P, c_int, c_int, c_int, c_int, c_float, c_int, P, P, P, c_float, P, P],
    ),
    "b200sr_group_norm_stats": (c_int, [P, c_int, c_int, c_int, c_int, c_float, P, P, P]),
    "b200sr_layer_norm": (c_int, [P, P, P, P, c_int, c_int, c_float, P]),
    "b200sr_attention_d64": (
        c_int,
        [P, c_i64, c_int, P, c_i64, c_int, P, c_i64, c_int, P, c_i64, c_int, c_int, c_int, c_int, c_float, c_int, P, P],
    ),
    "b200sr_attention_d64_workspace_bytes": (C.c_size_t, [c_int, c_int, c_int, c_int]),
    "b200sr_nchw_f32_to_nhwc_bf16": (c_int, [P, P, c_int, c_int, c_int, c_float, P]),
    "b200sr_nhwc_bf16_to_nchw_f32_strided": (c_int, [P, P, c_int, c_int, c_int, c_int, P]),
    "b200sr_upsample2x_nhwc": (c_int, [P, P, c_int, c_int, c_int, c_int, P]),
    "b200sr_concat_add": (c_int, [P, c_int, P, c_int, P, P, c_i64, P]),
    "b200sr_axpy_bf16": (c_int, [P, P, P, c_float, c_i64, P]),
    "b200sr_silu_bf16": (c_int, [P, P, c_i64, P]),
    "b200sr_pad_channels": (c_int, [P, P, c_int, c_int, c_i64, P]),
    "b200sr_embed_tokens": (c_int, [P, P, P, P, c_int, c_int, c_int, c_int, P]),
    "b200sr_sinusoid_embedding": (c_int, [P, P, c_int, c_int, c_float, c_int, P]),
    "b200sr_sampler_pre": (c_int, [P, P, P, P, P, c_int, c_int, c_int, c_int, P]),
    "b200sr_sampler_post": (c_int, [P, P, P, P, P, c_int, c_int, c_int, c_int, P, P, P]),
    "b200sr_euler_from_denoised": (c_int, [P, P, P, P, c_i64, P, P, P]),
    "b200sr_tile_accumulate": (c_int, [P, P, P, P, c_int, c_int, c_int, c_int, c_int, c_int, c_int, P]),
    "b200sr_tile_normalize": (c_int, [P, P, P, c_i64, P]),
    "b200sr_rel_l1_similarity": (c_int, [P, P, c_i64, P, P, P, P]),
    "b200sr_sr3_update": (c_int, [P, P, P, P, P, c_i64, P]),
    "b200sr_wavelet_level": (c_int, [P, P, P, c_int, c_int, c_int, c_int, c_int, P]),
    "b200sr_add_f32": (c_int, [P, P, P, c_i64, P]),
    "b200sr_image_to_u8": (c_int, [P, P, c_int, c_int, c_int, c_int, c_int, P]),
    "b200sr_tensor2img_u8": (c_int, [P, P, c_int, c_int, c_int, P]),
    "b200sr_resample_u8": (c_int, [P, P, c_int, c_int, c_int, c_int, P, P, c_int, P]),
    "b200sr_img_u8_to_tensor": (c_int, [P, P, c_int, c_int, c_int, P]),
    "b200sr_copy_batch": (c_int, [C.POINTER(Copy), c_int, P]),
    "b200sr_tile_weighted_strip": (c_int, [P, P, P, c_int, c_int, c_int, c_int, c_int, c_int, c_int, P]),
    "b200sr_strip_add": (c_int, [P, P, c_int, c_int, c_int, c_int, c_int, c_int, c_int, P]),
}

_ERRORS = {-22: "EINVAL (bad shape / alignment / flags)", -19: "ENODEV (no sm_100 device / driver)", -5: "EIO (CUDA launch error)"}

_lib = None


class B200SRError(RuntimeError):
    pass


def load() -> C.CDLL:
    """Load libb200sr.so, bind every declared symbol, verify the ABI version."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise B200SRError(
            f"{LIB_PATH} not found: build the sm_100a extension first "
            "(python -c 'import __graft_entry__ as g; g.build()' or csrc/build.sh). There is no CPU fallback."
        )
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if the .so is stale
        fn.restype = res
        fn.argtypes = args
    if lib.b200sr_abi_version() != ABI_VERSION:
        raise B200SRError(f"libb200sr.so ABI {lib.b200sr_abi_version()} != binding ABI {ABI_VERSION}; rebuild")
    _lib = lib
    return lib


LAUNCHES = [0]  # number of b200sr kernels enqueued so far (each C-ABI call reports its kernel count here)


TRACE = None  # optional list: one entry per kernel enqueued ("what" of the C-ABI call), for joining with ncu launch lists


def check(rc: int, what: str, kernels: int = 1) -> None:
    LAUNCHES[0] += kernels
    if TRACE is not None:
        TRACE.extend([what] * kernels)
    if rc != 0:
        raise B200SRError(f"{what} failed: {_ERRORS.get(rc, rc)}")
