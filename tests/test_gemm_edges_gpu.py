"""The GEMM and the 3x3 convolution against float64, element by element, at every tile edge and epilogue family: N tiles
from 32 to 256 on CTA pairs and single CTAs, phantom M blocks, N tails on the 16-byte store path, ragged K, CTAs that
change N block between tiles, the plain / general / GEGLU / fp32 (direct and TMA-stored) epilogues, per-group weights
with gap rows, guarded output / residual / rowvec / A windows, CUDA-graph replay, the three convolution modes at the
widths the any-size restore reaches, and the env-switched alternative paths.  References, bounds (derived in gemm_ref's
docstring), the geometry ports and the generators live in tests/gemm_ref.py; each case prints its worst err / bound.

Epilogue families of gemm_conv.cu and the suite that owns each: EPI_GENERAL, EPI_PLAIN, EPI_GEGLU here; EPI_XFORM
(fused-input GroupNorm) and EPI_LN_PLAIN / EPI_LN_GEGLU in test_norm_edges_gpu.py; EPI_SOFTMAX, EPI_LN_SOFTMAX,
EPI_RS_STATS and EPI_RS_APPLY in test_softmax_edges_gpu.py."""
import ctypes
import os
import subprocess
import sys
import textwrap

import pytest
import torch

import gemm_ref as gr

pytestmark = pytest.mark.gpu
bf16, f32 = torch.bfloat16, torch.float32
TESTS = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(TESTS)
PKG = os.path.join(ROOT, "remote-sensing-vision-language-diffusion-model_b200")
NAN = float("nan")


@pytest.fixture(scope="module")
def ops():
    from b200sr import ops as _ops

    return _ops


@pytest.fixture(scope="module")
def lib():
    from b200sr import _lib

    return _lib.load()


@pytest.fixture(scope="module")
def num_sms():
    return torch.cuda.get_device_properties(torch.cuda.current_device()).multi_processor_count


def _report(what, worst):
    print(f"\n[err/bound] {what}: {worst:.3f}")


# ---------------------------------------------------------------------------------------------------------------------
# one GEMM through the C ABI, every operand in a guarded window
# ---------------------------------------------------------------------------------------------------------------------
class GemmCase:
    """Operands of one b200sr_gemm_bf16 call placed in sentinel-filled buffers: A [M, K] at row stride lda = K + 8 with NaN
    in columns K..lda; per-group weights with NaN gap rows; rowvec a column window of a NaN-padded matrix; residual and
    out windows at column offset ``col`` of rows ``ld`` wide (NaN around them)."""

    device = "cuda"

    def __init__(self, M, N, K, *, bias=True, alpha=1.0, rowvec=False, rpg=0, residual=False, act=0, geglu=False,
                 out_fp32=False, w_rpg=0, w_gap=0, col=16, ld_pad=48, force_bn=0, seed=0):
        self.M, self.N, self.K, self.force_bn = M, N, K, force_bn
        dev = self.device
        self.alpha, self.act, self.geglu, self.out_fp32, self.rpg, self.w_rpg = alpha, act, geglu, out_fp32, rpg, w_rpg
        groups = -(-M // w_rpg) if w_rpg else 1
        a, w, b, rv, res = gr.gemm_inputs(M, N, K, groups=groups, seed=seed)
        self.lda = K + 8
        self.a = gr.Guarded(M, K, self.lda, bf16, dev, values=a.to(dev), before=0, after=0)
        self.w3 = (w if w.dim() == 3 else w[None]).to(dev)
        self.w_stride = N + w_gap if w_rpg else 0
        rows = (groups - 1) * self.w_stride + N if w_rpg else N
        self.w = torch.full((rows, K), NAN, dtype=bf16, device=dev)
        for g in range(groups):
            self.w[g * self.w_stride:g * self.w_stride + N] = self.w3[g]
        self.bias = b.to(dev) if bias else None
        n_rv = -(-M // rpg) if rpg else 1
        self.rv = gr.Guarded(n_rv, N, N + 24, f32, dev, col=4, values=rv[:n_rv].to(dev), before=1, after=1) \
            if rowvec else None
        self.res = gr.Guarded(M, N, N + ld_pad, bf16, dev, col=col, values=res.to(dev)) if residual else None
        n_out = N // 2 if geglu else N
        esz = 4 if out_fp32 else 2
        self.out = gr.Guarded(M, n_out, n_out + ld_pad, f32 if out_fp32 else bf16, dev, col=col * 2 // esz)

    def plan(self, sms, **kw):
        return gr.gemm_plan(self.M, self.N, self.K, force_bn=self.force_bn, geglu=self.geglu, out_fp32=self.out_fp32,
                            residual=self.res is not None, rowvec=self.rv is not None, ldc=self.out.ld,
                            ldr=self.res.ld if self.res else 0, out_align=self.out.view.data_ptr() % 256 or 256,
                            res_align=(self.res.view.data_ptr() % 256 or 256) if self.res else 256, sms=sms, **kw)

    def epilogue(self):
        from b200sr import _lib

        e = _lib.Epilogue()
        e.bias = self.bias.data_ptr() if self.bias is not None else None
        if self.rv is not None:
            e.rowvec, e.ld_rowvec, e.rows_per_group = self.rv.view.data_ptr(), self.rv.ld, self.rpg
        if self.res is not None:
            e.residual, e.ldr = self.res.view.data_ptr(), self.res.ld
        e.out, e.ldc, e.out_fp32, e.geglu, e.alpha, e.act = self.out.view.data_ptr(), self.out.ld, int(self.out_fp32), \
            int(self.geglu), self.alpha, self.act
        e.w_rows_per_group, e.w_group_stride = self.w_rpg, self.w_stride
        return e

    def run(self, lib, ops):
        e = self.epilogue()
        rc = lib.b200sr_gemm_bf16(self.a.view.data_ptr(), self.lda, self.w.data_ptr(), self.M, self.N, self.K,
                                  ctypes.byref(e), self.force_bn, ops._stream())
        assert rc == 0, rc
        return self.out.view

    def reference(self):
        return gr.gemm(self.a.view, self.w3 if self.w_rpg else self.w3[0], bias=self.bias, alpha=self.alpha,
                       rowvec=None if self.rv is None else self.rv.view, rows_per_group=self.rpg,
                       residual=None if self.res is None else self.res.view, act=self.act, geglu=self.geglu,
                       w_rows_per_group=self.w_rpg, out_fp32=self.out_fp32)

    def check(self, what):
        torch.cuda.synchronize()
        for g in (self.out, self.res, self.rv, self.a):
            if g is not None:
                g.check(what, window_finite=g is self.out)
        ref, bound = self.reference()
        return gr.assert_within(self.out.view, ref, bound, what)


def _edges(p, case, claims):
    """Assert every edge a case claims to reach, from the geometry port."""
    M, N = case.M, case.N
    checks = {
        "phantom": p["phantom"] == 1,
        "cluster1": p["cluster"] == 1,
        "partial_m": M % 128 != 0,
        "partial_n": N % p["BN"] != 0,
        "store16": not p["wide_io"],
        "wide": p["wide_io"],
        "n_change": bool(gr.n_block_changes(p)),
        "multi_tile": p["work"] > p["grid"] // p["cluster"],
        "tma": p["epi_tma"],
        "ragged_k": case.K % 64 != 0,
        "k_not16": case.K % 16 != 0,
        "group_in_tile": case.rpg % 128 != 0,
        "partial_w_group": case.w_rpg and M % case.w_rpg != 0,
    }
    bad = [c for c in claims if not checks[c]]
    assert not bad, f"edges not reached: {bad} (plan {p})"


GEMM_CASES = [
    # id, (M, N, K), kwargs, claimed edges
    ("bn32-pair-phantom", (300, 200, 72), dict(force_bn=32, residual=True, alpha=0.75), ["phantom", "partial_n", "k_not16"]),
    ("bn64", (300, 200, 8), dict(force_bn=64, residual=True), ["phantom", "partial_n", "ragged_k"]),
    ("bn96", (1000, 200, 200), dict(force_bn=96, residual=True), ["partial_m", "partial_n", "ragged_k"]),
    ("bn128", (1000, 1000, 4104), dict(force_bn=128), ["partial_m", "partial_n", "ragged_k"]),
    ("bn160-store16", (640, 424, 136), dict(force_bn=160, residual=True, ld_pad=40, col=8),
     ["partial_n", "store16", "phantom"]),
    ("bn192", (640, 520, 72), dict(force_bn=192, residual=True, alpha=-2.0), ["partial_n", "phantom"]),
    ("bn224", (256, 1000, 72), dict(force_bn=224), ["partial_n"]),
    ("bn256-cluster1", (100, 520, 200), dict(force_bn=256, residual=True), ["cluster1", "partial_n", "partial_m"]),
    ("picked-cluster1", (77, 40, 72), dict(residual=True), ["cluster1", "store16"]),
    ("picked", (2048, 1280, 640), dict(residual=True), []),
    ("n-block-changes", (8192, 2560, 200), dict(force_bn=256, residual=True), ["n_change", "multi_tile"]),
    ("n-block-changes-partial", (4100, 1288, 72), dict(force_bn=128, residual=True), ["n_change", "partial_n", "phantom"]),
    ("general-rowvec-silu", (1000, 200, 200), dict(rowvec=True, rpg=100, residual=True, act=1, alpha=0.5),
     ["group_in_tile", "partial_m"]),
    ("general-gelu", (384, 264, 72), dict(rowvec=True, rpg=200, act=2), ["group_in_tile", "store16"]),
    ("general-quick-gelu", (130, 96, 4104), dict(rowvec=True, act=3, alpha=1.5), ["ragged_k"]),
    ("general-fp32", (1000, 200, 200), dict(out_fp32=True, rowvec=True, rpg=300, residual=True), ["partial_n"]),
    ("general-fp32-tma", (4096, 2048, 72), dict(out_fp32=True, force_bn=128, alpha=0.25), ["tma", "multi_tile"]),
    ("general-fp32-tma-silu", (4224, 1000, 72), dict(out_fp32=True, act=1, force_bn=64), ["tma", "partial_n"]),
    ("geglu", (260, 512, 136), dict(geglu=True), ["partial_m"]),
    ("geglu-store16", (1000, 2080, 200), dict(geglu=True, col=8, ld_pad=40), ["store16", "partial_m"]),
    ("geglu-big", (2048, 10240, 1280), dict(geglu=True), ["multi_tile"]),
    ("w-groups-gap", (612, 200, 72), dict(w_rpg=256, w_gap=24, residual=True), ["partial_w_group", "partial_n"]),
    ("w-groups-general", (1100, 320, 200), dict(w_rpg=512, w_gap=8, rowvec=True, rpg=100, act=1),
     ["partial_w_group", "group_in_tile"]),
]


@pytest.mark.parametrize("name,shape,kw,claims", GEMM_CASES, ids=[c[0] for c in GEMM_CASES])
def test_gemm_per_element(ops, lib, num_sms, name, shape, kw, claims):
    c = GemmCase(*shape, seed=sum(shape), **kw)
    p = c.plan(num_sms)
    if c.force_bn == 0 and not c.w_rpg:
        assert p["BN"] == ops.gemm_n_tile(*shape)
    _edges(p, c, claims)
    c.run(lib, ops)
    what = (f"gemm {name} {shape} BN={p['BN']} cluster={p['cluster']} wide={int(p['wide_io'])} "
            f"tma={int(p['epi_tma'])}")
    _report(what, c.check(what))


@pytest.mark.parametrize("fam", ["plain", "general", "geglu", "fp32-tma"])
def test_gemm_graph_replay_bit_equal(ops, lib, fam):
    """One capture per family, replayed on new operand values: bit-equal to an eager call on the same values."""
    kw = {"plain": dict(residual=True, alpha=0.5), "general": dict(rowvec=True, rpg=100, act=1, residual=True),
          "geglu": dict(geglu=True), "fp32-tma": dict(out_fp32=True, force_bn=128)}[fam]
    shape = (4096, 2048, 72) if fam == "fp32-tma" else (1000, 512, 200)
    c = GemmCase(*shape, **kw)
    c.run(lib, ops)
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        c.run(lib, ops)
    fresh = GemmCase(*shape, seed=7, **kw)
    c.a.view.copy_(fresh.a.view)
    if c.res is not None:
        c.res.view.copy_(fresh.res.view)
    graph.replay()
    torch.cuda.synchronize()
    replayed = c.out.view.clone()
    c.out.view.fill_(NAN)
    c.run(lib, ops)
    torch.cuda.synchronize()
    assert torch.equal(replayed, c.out.view), f"graph replay {fam}: differs from the eager call"
    _report(f"graph replay {fam} {shape}", c.check(f"graph replay {fam}"))


# ---------------------------------------------------------------------------------------------------------------------
# convolution
# ---------------------------------------------------------------------------------------------------------------------
def _conv(ops, NB, H, W, Cin, Cout, stride=1, pad_lo=1, *, force_bn=0, terms=True, col=0, ld_pad=0, seed=0):
    """ops.conv3x3 with every epilogue term (rowvec per image, residual, alpha, SiLU) into a guarded channel window of a
    wider NHWC buffer; returns (out view, reference, bound, the out Guarded)."""
    x, wp, b, rv, res = (t.cuda() for t in gr.conv_inputs(NB, H, W, Cin, Cout, stride=stride, seed=seed))
    OH, OW = H // stride, W // stride
    ld = Cout + ld_pad
    g = gr.Guarded(NB * OH * OW, Cout, ld, bf16, "cuda", col=col)
    out = g.view.unflatten(0, (NB, OH, OW))
    kw = dict(bias=b, rowvec=rv, residual=res, alpha=0.75, act=1) if terms else dict(bias=b)
    ops.conv3x3(x, wp, stride=stride, pad_lo=pad_lo, out=out, force_bn=force_bn, **kw)
    torch.cuda.synchronize()
    g.check("conv out window")
    ref, bound = gr.conv3x3(x, wp, stride=stride, pad_lo=pad_lo, **kw)
    return out, ref, bound


CONV_CASES = [
    # (NB, H, W, Cin, Cout, stride, pad_lo, force_bn), claim
    ((6, 17, 17, 64, 64, 1, 1, 0), "mode 1, W = 17: 1 x 32 x 4 box, second image block 2 real + 2 masked"),
    ((1, 17, 17, 128, 96, 1, 1, 0), "mode 1, one image in a 4-image box"),
    ((2, 34, 34, 64, 96, 1, 1, 0), "mode 1, W = 34: 2 x 64 box"),
    ((3, 12, 24, 64, 64, 1, 1, 0), "mode 1, H < 16"),
    ((3, 5, 12, 128, 72, 1, 1, 0), "mode 1, 4 x 8 x 4 box, H = 5"),
    ((5, 40, 5, 64, 64, 1, 1, 0), "mode 1, W = 5, H = 40"),
    ((2, 34, 34, 64, 64, 2, 1, 0), "mode 2, 34 -> 17, pad_lo = 1"),
    ((2, 34, 34, 128, 64, 2, 0, 0), "mode 2, 34 -> 17, pad_lo = 0"),
    ((1, 68, 100, 64, 200, 2, 0, 0), "mode 2, 68 x 100 -> 34 x 50, pad_lo = 0"),
    ((2, 64, 64, 192, 128, 2, 1, 0), "mode 2, even"),
    ((2, 40, 24, 64, 200, 1, 1, 0), "mode 3, partial H tile, Cout not a multiple of BN"),
    ((3, 48, 8, 320, 256, 1, 1, 0), "mode 3, odd tile count: a phantom M block"),
    ((1, 16, 16, 2560, 320, 1, 1, 0), "mode 3, Cin = 2560"),
    ((1, 16, 8, 64, 256, 1, 1, 256), "mode 3, single M block, BN = 256"),
    ((2, 32, 24, 128, 384, 1, 1, 192), "mode 3, BN = 192"),
    ((2, 64, 64, 64, 32, 1, 1, 0), "mode 3, resident weights"),
]


@pytest.mark.parametrize("case,claim", CONV_CASES, ids=["x".join(map(str, c[0])) for c in CONV_CASES])
def test_conv3x3_per_element(ops, num_sms, case, claim):
    NB, H, W, Cin, Cout, stride, pad_lo, bn = case
    p = gr.conv_plan(NB, H, W, Cin, Cout, stride, force_bn=bn, sms=num_sms)
    assert f"mode {p['mode']}" in claim
    if "resident" in claim:
        assert p["w_resident"]
    if "masked" in claim or "4-image" in claim:
        assert p["bn"] == 4 and p["tiles_n"] * 4 > NB
    if "phantom" in claim:
        assert p["phantom"] == 1
    if "single M block" in claim:
        assert p["cluster"] == 1 and p["m_blocks"] == 1
    if "Cout not a multiple" in claim:
        assert Cout % p["BN"] != 0
    out, ref, bound = _conv(ops, NB, H, W, Cin, Cout, stride, pad_lo, force_bn=bn, col=16, ld_pad=48, seed=H + Cout)
    what = (f"conv3x3 {NB}x{H}x{W} {Cin}->{Cout} s{stride} pad_lo={pad_lo} ({claim}; box {p['bw']}x{p['bh']}x{p['bn']}, "
            f"BN={p['BN']}, cluster {p['cluster']})")
    _report(what, gr.assert_within(out, ref, bound, what))


# The convolutions a 1088 x 1600 stage-2 input reaches (latent 136 x 200 -> 68 x 100 -> 34 x 50; widths 100 and 50 are not
# multiples of 8, so those levels leave the halo path), the VAE and SR3 levels at 136 x 200 and 68 x 100, and the
# benchmark's 128^2 latent (CFG batch 2).
PRODUCTION = [
    ("unet 136x200", (1, 136, 200, 320, 320, 1)), ("unet down 136x200", (1, 136, 200, 320, 320, 2)),
    ("unet 68x100", (1, 68, 100, 640, 640, 1)), ("unet cat 68x100", (1, 68, 100, 1280, 640, 1)),
    ("unet down 68x100", (1, 68, 100, 640, 640, 2)), ("unet 34x50", (1, 34, 50, 1280, 1280, 1)),
    ("unet cat 34x50", (1, 34, 50, 2560, 1280, 1)), ("vae 136x200", (1, 136, 200, 512, 512, 1)),
    ("sr3 68x100", (1, 68, 100, 512, 512, 1)),
    ("bench 128^2", (2, 128, 128, 320, 320, 1)), ("bench 64^2", (2, 64, 64, 640, 640, 1)),
    ("bench 32^2", (2, 32, 32, 1280, 1280, 1)), ("bench down 64^2", (2, 64, 64, 640, 640, 2)),
]


@pytest.mark.parametrize("name,case", PRODUCTION, ids=[c[0] for c in PRODUCTION])
def test_conv3x3_production_geometry(ops, num_sms, name, case):
    NB, H, W, Cin, Cout, stride = case
    p = gr.conv_plan(NB, H, W, Cin, Cout, stride, sms=num_sms)
    out, ref, bound = _conv(ops, NB, H, W, Cin, Cout, stride, seed=Cin)
    what = f"conv3x3 {name} {case}: mode {p['mode']}, box {p['bw']}x{p['bh']}x{p['bn']}, BN={p['BN']}"
    _report(what, gr.assert_within(out, ref, bound, what))


# ---------------------------------------------------------------------------------------------------------------------
# env-switched paths (each switch is read once per process: the alternative runs in a child)
# ---------------------------------------------------------------------------------------------------------------------
_CHILD = textwrap.dedent("""
    import sys
    sys.path[:0] = [{root!r}, {pkg!r}, {tests!r}]
    import torch
    import test_gemm_edges_gpu as t
    from b200sr import _lib, ops
    lib = _lib.load()
    torch.save(t._switch_outputs(lib, ops, {which!r}), {path!r})
""")

SWITCHES = {
    "B200SR_EPI_TMA": ("gemm", [((4096, 2048, 72), dict(out_fp32=True, force_bn=128)),
                                ((4224, 1000, 200), dict(out_fp32=True, act=3, force_bn=64))]),
    "B200SR_WIDE_IO": ("gemm", [((1000, 512, 200), dict(residual=True)), ((1000, 1024, 72), dict(geglu=True)),
                                ((1000, 256, 72), dict(rowvec=True, rpg=100, act=2, residual=True))]),
    "B200SR_CONV_RESIDENT": ("conv", [(2, 64, 64, 64, 32, 1), (1, 32, 32, 128, 32, 1)]),
    "B200SR_CONV_HALO": ("conv", [(2, 32, 32, 64, 64, 1), (2, 40, 24, 128, 96, 1)]),
}


def _switch_outputs(lib, ops, which):
    kind, cases = SWITCHES[which]
    outs = []
    for case in cases:
        if kind == "gemm":
            shape, kw = case
            c = GemmCase(*shape, seed=3, **kw)
            c.run(lib, ops)
            torch.cuda.synchronize()
            outs.append(c.out.view.cpu())
        else:
            outs.append(_conv(ops, *case, seed=5)[0].cpu())
    return outs


@pytest.mark.parametrize("which", list(SWITCHES))
def test_env_switched_path(ops, lib, num_sms, which, tmp_path):
    """The path a switch turns off, against the bound and against the default path.  EPI_TMA, WIDE_IO and CONV_RESIDENT
    change how data moves, not the arithmetic: bit for bit.  CONV_HALO=0 sends a stride-1 convolution to mode 1, whose K
    loop runs tap-major where the halo path runs chunk-major: with one 64-channel chunk (Cin = 64) both orders are the
    same and the outputs must be equal; with Cin = 128 they need only agree within the bound."""
    kind, cases = SWITCHES[which]
    for case in cases:    # the switch must change the path of each case
        if kind == "gemm":
            shape, kw = case
            p = GemmCase(*shape, seed=3, **kw).plan(num_sms)
            assert p["epi_tma"] if which == "B200SR_EPI_TMA" else p["wide_io"]
        else:
            p = gr.conv_plan(*case, sms=num_sms)
            assert p["mode"] == 3 and (p["w_resident"] or which == "B200SR_CONV_HALO")
    path = str(tmp_path / "switched.pt")
    code = _CHILD.format(root=ROOT, pkg=PKG, tests=TESTS, which=which, path=path)
    flags = ["-s"] if sys.flags.no_user_site else []
    r = subprocess.run([sys.executable, *flags, "-c", code], env=dict(os.environ, **{which: "0"}), capture_output=True,
                       text=True, timeout=900)
    assert r.returncode == 0, r.stderr[-4000:]
    switched = torch.load(path)
    default = _switch_outputs(lib, ops, which)
    for case, s, d in zip(cases, switched, default):
        if kind == "gemm":
            shape, kw = case
            c = GemmCase(*shape, seed=3, **kw)
            ref, bound = c.reference()
        else:
            x, wp, b, rv, res = (t.cuda() for t in gr.conv_inputs(*case[:5], stride=case[5], seed=5))
            ref, bound = gr.conv3x3(x, wp, stride=case[5], bias=b, rowvec=rv, residual=res, alpha=0.75, act=1)
        what = f"{which}=0 {case}"
        _report(what, gr.assert_within(s.cuda(), ref, bound, what))
        equal = torch.equal(s, d)
        if which != "B200SR_CONV_HALO" or case[3] == 64:
            assert equal, f"{what}: differs from the default path"
        print(f"[bitwise] {what}: {'equal to' if equal else 'differs from'} the default path")
