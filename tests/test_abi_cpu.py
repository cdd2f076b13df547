"""The drop-in boundary without a GPU: libb200sr.so loads, exports every entry point include/b200sr.h declares,
the ctypes binding lists exactly those, and the epilogue struct has the layout a C compiler gives the header.
No kernel is launched."""
import ctypes
import json
import os
import re
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "b200sr.h")
PKG = os.path.join(ROOT, "remote-sensing-vision-language-diffusion-model_b200")


@pytest.fixture(scope="module")
def lib():
    from b200sr import _lib

    if not os.path.exists(_lib.LIB_PATH):  # fresh checkout: nvcc cross-compiles without a GPU
        sys.path.insert(0, ROOT)
        import __graft_entry__

        __graft_entry__.build()
    return ctypes.CDLL(_lib.LIB_PATH)


def header_code():
    return re.sub(r"/\*.*?\*/", "", open(HEADER).read(), flags=re.S)


def declared_symbols():
    return sorted(set(re.findall(r"\b(b200sr_[a-z0-9_]+)\s*\(", header_code())))


def prototypes():
    """name -> (return type, [(parameter type, parameter name), ...]) of every function the header declares."""
    out = {}
    for ret, name, params in re.findall(r"(\w+)\s+(b200sr_[a-z0-9_]+)\s*\(([^)]*)\)\s*;", header_code()):
        params = [" ".join(p.split()) for p in params.split(",")]
        out[name] = (ret, [re.fullmatch(r"(.*?)\s*\b(\w+)", p).groups() for p in params if p != "void"])
    return out


def ctype_of(decl):
    from b200sr import _lib

    if "*" in decl:
        base = decl.replace("const", "").replace("*", "").strip()
        return {"b200sr_epilogue": ctypes.POINTER(_lib.Epilogue), "b200sr_copy": ctypes.POINTER(_lib.Copy)}.get(
            base, ctypes.c_void_p)
    return {"int32_t": ctypes.c_int32, "int": ctypes.c_int32, "int64_t": ctypes.c_int64, "float": ctypes.c_float,
            "size_t": ctypes.c_size_t}[decl]


def test_header_declares_the_path():
    names = declared_symbols()
    for must in ("b200sr_gemm_bf16", "b200sr_conv3x3_bf16", "b200sr_attention_d64", "b200sr_group_norm_nhwc",
                 "b200sr_layer_norm", "b200sr_sampler_post", "b200sr_tile_accumulate", "b200sr_rel_l1_similarity",
                 "b200sr_sr3_update"):
        assert must in names


def test_library_exports_every_declared_symbol(lib):
    missing = [n for n in declared_symbols() if not hasattr(lib, n)]
    assert not missing, f"declared in include/b200sr.h but not exported: {missing}"


def test_binding_covers_exactly_the_header(lib):
    from b200sr import _lib

    declared = set(declared_symbols())
    bound = set(_lib.SIGNATURES) | {"b200sr_abi_version", "b200sr_num_sms"}
    assert declared - bound == set(), f"no ctypes signature for {sorted(declared - bound)}"
    assert bound - declared == set(), f"bound but not declared in the header: {sorted(bound - declared)}"
    lib.b200sr_abi_version.restype = ctypes.c_int
    assert lib.b200sr_abi_version() == _lib.ABI_VERSION


def test_binding_types_match_the_header():
    """Every ctypes signature has the header's types: a parameter of the wrong width (c_int32 for an int64_t count)
    would make the library read undefined upper register bits, and no other check notices it."""
    from b200sr import _lib

    protos = prototypes()
    assert sorted(protos) == declared_symbols()
    for name, (res, args) in _lib.SIGNATURES.items():
        ret, params = protos[name]
        assert res == ctype_of(ret), name
        assert args == [ctype_of(t) for t, _ in params], name


def test_abi_version_matches_the_header():
    from b200sr import _lib

    m = re.search(r"^#define\s+B200SR_ABI_VERSION\s+(\d+)\b", open(HEADER).read(), flags=re.M)
    assert m is not None and int(m.group(1)) == _lib.ABI_VERSION


# Every entry point with pointer parameters: the pointers it rejects as NULL, and valid values for its other parameters.
# Pointers not listed may be NULL (optional operands such as bias, noise, cnt or high; the attention workspace).
NULL_REJECTED = {
    "b200sr_gemm_bf16": ("A W epi", dict(lda=64, M=128, N=64, K=64, force_bn=0)),
    "b200sr_conv3x3_bf16": ("x w epi", dict(N=1, H=16, W=16, Cin=64, Cout=64, stride=1, pad_lo=1, force_bn=0)),
    "b200sr_conv3x3_small": ("x w y", dict(N=1, H=8, W=8, Cin=4, Cout=64, out_nchw_f32=0)),
    "b200sr_group_norm_nhwc": ("x y", dict(N=1, HW=64, C=64, groups=32, eps=1e-5, silu=0, control_scale=1.0)),
    "b200sr_group_norm_stats": ("x", dict(N=1, HW=64, C=64, groups=32, eps=1e-5)),
    "b200sr_layer_norm": ("x y", dict(M=8, C=64, eps=1e-5)),
    "b200sr_attention_d64": ("q k v out", dict(ldq=64, q_col=0, ldk=64, k_col=0, ldv=64, v_col=0, ldo=64, B=1, H=1,
                                               Nq=128, Nk=128, scale=0.125, causal=0)),
    "b200sr_row_softmax_fold": ("parts out", dict(n_parts=2, rows=128)),
    "b200sr_softmax_rows": ("x y", dict(rows=8, cols=128, valid_cols=77, scale=0.125)),
    "b200sr_nchw_f32_to_nhwc_bf16": ("x y", dict(N=1, C=4, HW=64, scale=1.0)),
    "b200sr_nhwc_bf16_to_nchw_f32": ("x y", dict(N=1, C=4, HW=64)),
    "b200sr_nhwc_bf16_to_nchw_f32_strided": ("x y", dict(N=1, C=4, Cs=8, HW=64)),
    "b200sr_upsample2x_nhwc": ("x y", dict(N=1, H=8, W=8, C=64)),
    "b200sr_concat_add": ("a b out", dict(Ca=64, Cb=64, rows=64)),
    "b200sr_axpy_bf16": ("a b y", dict(alpha=1.0, n=64)),
    "b200sr_pad_channels": ("x y", dict(C=4, Cpad=64, rows=64)),
    "b200sr_silu_bf16": ("x y", dict(n=64)),
    "b200sr_embed_tokens": ("ids tok pos out", dict(B=1, T=77, C=768, vocab=49408)),
    "b200sr_sinusoid_embedding": ("t out", dict(B=2, dim=320, max_period=10000.0, sin_first=0)),
    "b200sr_sampler_pre": ("x scalars x_hat net_in", dict(B=1, C=4, HW=64, cfg_copies=2)),
    "b200sr_sampler_post": ("eps x_hat scalars x_next", dict(B=1, C=4, HW=64, use_cfg=1)),
    "b200sr_euler_from_denoised": ("denoised x_hat scalars x_next", dict(n=256)),
    "b200sr_tile_accumulate": ("tile weight acc", dict(BC=4, th=8, tw=8, H=16, W=16, h0=0, w0=8)),
    "b200sr_tile_normalize": ("acc cnt out", dict(n=256)),
    "b200sr_tile_weighted_strip": ("tile weight strip", dict(BC=4, th=8, tw=8, y0=0, x0=4, sh=8, sw=4)),
    "b200sr_strip_add": ("strip acc", dict(BC=4, sh=8, sw=4, H=16, W=16, h0=0, w0=4)),
    "b200sr_pointwise_small": ("x w y", dict(Cin=4, Cout=4, rows=64, HW=64, out_nchw_f32=0, scale=1.0)),
    "b200sr_diag_gaussian": ("moments z", dict(N=1, C=4, HW=64, scale=0.13025)),
    "b200sr_wavelet_level": ("img low", dict(first=1, BC=3, H=16, W=16, radius=1)),
    "b200sr_add_f32": ("a b out", dict(n=256)),
    "b200sr_image_to_u8": ("x out", dict(C=3, H=16, W=16, OH=32, OW=32)),
    "b200sr_tensor2img_u8": ("x out", dict(C=3, H=16, W=16)),
    "b200sr_resample_u8": ("src dst bounds coeffs", dict(outer=16, in_len=16, out_len=32, inner=3, ksize=4)),
    "b200sr_img_u8_to_tensor": ("in out", dict(C=3, H=16, W=16)),
    "b200sr_rel_l1_similarity": ("prev cur threshold workspace result", dict(n=64)),
    "b200sr_sr3_update": ("x eps scalars out", dict(n=256)),
    "b200sr_copy_batch": ("copies", dict(n=1)),
}

# Runs the calls in a process that sees no GPU, so that a missing check fails with a CUDA error code instead of
# launching a kernel on a NULL pointer.  "epi" / "copies" stand for one valid host-side struct.
_NULL_CALLS = r"""
import ctypes, json, sys
sys.path.insert(0, sys.argv[1])
from b200sr import _lib
lib = _lib.load()
structs = {"epi": ctypes.byref(_lib.Epilogue(out=1 << 20, ldc=64)),
           "copies": ctypes.byref(_lib.Copy(src=1 << 20, dst=2 << 20, bytes=64))}
calls = json.loads(sys.argv[2])
print(json.dumps([getattr(lib, name)(*[structs.get(a, a) if isinstance(a, str) else a for a in args])
                  for name, args in calls]))
"""


def test_null_pointers_are_rejected_before_any_cuda_call(lib):
    """Each pointer an entry point rejects as NULL gives -22 (EINVAL) with every other argument valid, checked before
    the entry point touches the CUDA runtime: the calls run without a device."""
    protos = prototypes()
    takes_pointers = {n for n, (_, ps) in protos.items() if any("*" in t and p != "stream" for t, p in ps)}
    assert takes_pointers == set(NULL_REJECTED)
    calls = []
    for name, (rejected, values) in NULL_REJECTED.items():
        params = protos[name][1]
        assert set(rejected.split()) <= {p for _, p in params}, name
        for nulled in rejected.split():
            args = []
            for i, (t, p) in enumerate(params):
                if p == nulled or p == "stream":
                    args.append(None)
                elif p in ("epi", "copies"):
                    args.append(p)
                elif "*" in t:
                    args.append((i + 1) << 20)  # distinct, aligned, never dereferenced
                else:
                    args.append(values[p])
            calls.append((name, args))
    res = subprocess.run([sys.executable, "-c", _NULL_CALLS, PKG, json.dumps(calls)],
                         env={**os.environ, "CUDA_VISIBLE_DEVICES": ""}, capture_output=True, text=True)
    assert res.returncode == 0, res.stderr
    rcs = json.loads(res.stdout)
    wrong = [(name, args, rc) for (name, args), rc in zip(calls, rcs) if rc != -22]
    assert not wrong, f"NULL pointer not rejected with EINVAL: {wrong}"


def test_epilogue_struct_layout_matches_a_c_compiler(tmp_path):
    from b200sr import _lib

    fields = [f[0] for f in _lib.Epilogue._fields_]
    prog = '#include <stdio.h>\n#include <stddef.h>\n#include "b200sr.h"\nint main(void) {\n'
    prog += '  printf("%zu\\n", sizeof(b200sr_epilogue));\n'
    for f in fields:
        prog += f'  printf("%zu\\n", offsetof(b200sr_epilogue, {f}));\n'
    prog += "  return 0;\n}\n"
    src, exe = tmp_path / "layout.c", tmp_path / "layout"
    src.write_text(prog)
    subprocess.run(["gcc", "-std=c11", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)], check=True)
    out = [int(x) for x in subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout.split()]
    assert out[0] == ctypes.sizeof(_lib.Epilogue)
    for name, off in zip(fields, out[1:]):
        assert getattr(_lib.Epilogue, name).offset == off, name


def test_integration_doc_embeds_the_current_binding():
    """INTEGRATION.md section 1 shows the struct declarations a maintainer pastes: they must be the binding's own
    (generated) text, field for field — a stale snippet mis-lays the struct silently."""
    from b200sr import _lib

    doc = open(os.path.join(ROOT, "INTEGRATION.md")).read()
    assert _lib.binding_snippet() in doc, "INTEGRATION.md struct snippet differs from b200sr._lib (regenerate it)"
    assert f"`b200sr_abi_version()` ({_lib.ABI_VERSION})" in doc


def test_copy_struct_layout_matches_a_c_compiler(tmp_path):
    from b200sr import _lib

    prog = ('#include <stdio.h>\n#include <stddef.h>\n#include "b200sr.h"\nint main(void) {\n'
            '  printf("%zu %zu %zu %zu\\n", sizeof(b200sr_copy), offsetof(b200sr_copy, src), offsetof(b200sr_copy, dst), '
            'offsetof(b200sr_copy, bytes));\n  return 0;\n}\n')
    src, exe = tmp_path / "copy.c", tmp_path / "copy"
    src.write_text(prog)
    subprocess.run(["gcc", "-std=c11", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)], check=True)
    out = [int(x) for x in subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout.split()]
    assert out == [ctypes.sizeof(_lib.Copy), _lib.Copy.src.offset, _lib.Copy.dst.offset, _lib.Copy.bytes.offset]


def test_size_queries_work_without_a_device(lib):
    lib.b200sr_group_norm_workspace_bytes.restype = ctypes.c_size_t
    lib.b200sr_attention_d64_workspace_bytes.restype = ctypes.c_size_t
    assert lib.b200sr_group_norm_workspace_bytes(2, 1024, 1280, 32) > 1024
    assert lib.b200sr_attention_d64_workspace_bytes(2, 20, 1024, 77) == 0  # one key block: nothing to split
    assert lib.b200sr_attention_d64_workspace_bytes(0, 20, 1024, 1024) == 0
