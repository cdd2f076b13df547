"""Every normalisation path of the library against float64, element by element, at its chunk, group and offset edges:
GroupNorm on both of its paths (one kernel with a per-image barrier, statistics + apply) at shapes on either side of
the boundary between them, the one-kernel path against the two-kernel path bit for bit, group_norm_stats and the
fused-input-GroupNorm convolution, CUDA-graph replays of the stateful paths, every layer_norm_kernel instantiation, and
the LayerNorm folded into the GEMMs on both sides (consumer, producer, both in one launch, and the statistics written
through a guarded window).  References, bounds (derived in norm_ref's docstrings), the geometry port and the generators
live in tests/norm_ref.py; each test prints its worst err / bound."""
import ctypes
import os
import subprocess
import sys
import textwrap

import pytest
import torch

import norm_ref as nr

pytestmark = pytest.mark.gpu
bf16 = torch.bfloat16
TESTS = os.path.dirname(os.path.abspath(__file__))


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


def _gn_counters_zero(ops):
    ws = [w for key, w in ops._ws_cache.items() if key[-1] == "gn"]
    assert ws
    for w in ws:
        assert int(w[:nr.GN_WS_COUNTER_FLOATS].view(torch.int32).abs().sum()) == 0


# ---------------------------------------------------------------------------------------------------------------------
# GroupNorm, per element, on both paths
# ---------------------------------------------------------------------------------------------------------------------
GN_SHAPES = [
    (2, 64 * 64, 640), (2, 32 * 32, 1280), (2, 32 * 32, 2560),
    (4, 32 * 32, 1280),          # chunks * N == SMs (148)
    (2, 1000, 1280),             # ragged: the last chunk has 6 pixels
    (1, 136, 128),               # last chunk of 8 pixels for 16 thread rows
    (2, 1024, 960),              # 240 of 256 threads active
    (128, 8 * 8, 64),            # groups of 2 channels split the 8-channel vectors
    (8, 32 * 32, 1280),          # one image past the SM count
    (129, 8 * 8, 64),            # N > 128
    (2, 128 * 128, 320), (2, 64 * 64, 1920),
    (1, 1024 * 1024, 128),       # SR3 / VAE size, 296 chunks
]
GN_VARIANTS = [(1e-5, True, None), (1e-6, False, None), (1e-5, False, 1.0), (1e-6, True, 0.6)]   # eps, silu, SFT cs


def _gn_case(shape, eps, cs, seed):
    N, HW, C = shape
    x = nr.gn_inputs(N, HW, C, eps=eps, seed=seed).cuda()
    w, b, gam, bet, raw = (t.cuda() for t in nr.gn_params(C, seed=seed, sft_shape=shape if cs is not None else (1,)))
    sft = dict(sft_gamma=gam, sft_beta=bet, raw=raw, control_scale=cs) if cs is not None else {}
    return x, w, b, sft


@pytest.mark.parametrize("variant", GN_VARIANTS, ids=lambda v: f"eps{v[0]:g}-silu{int(v[1])}-cs{v[2]}")
@pytest.mark.parametrize("shape", GN_SHAPES, ids=lambda s: "x".join(map(str, s)))
def test_group_norm_per_element(ops, lib, num_sms, shape, variant):
    eps, silu, cs = variant
    N, HW, C = shape
    geo = nr.gn_geometry(N, HW, C, 32, num_sms)
    assert lib.b200sr_group_norm_launches(N, HW, C, 32) == geo["launches"]
    x, w, b, sft = _gn_case(shape, eps, cs, seed=HW + C)
    y = ops.group_norm(x, w, b, groups=32, eps=eps, silu=silu, **sft)
    torch.cuda.synchronize()
    _gn_counters_zero(ops)
    ref, bound = nr.group_norm(x, w, b, groups=32, eps=eps, silu=silu, num_sms=num_sms, **sft)
    path = "one kernel" if geo["launches"] == 1 else "two kernels"
    what = f"group_norm {shape} ({path}, last chunk {geo['last_chunk']}) eps={eps:g} silu={silu} cs={cs}"
    _report(what, nr.assert_within(y, ref, bound, what))
    if cs is None and not silu:
        # var = 0: the reference of a constant group is exactly its bias, so the check above holds the output to the bias
        # within the bound.  That bound keeps an absolute term for x * sc + (b - mean * sc): at eps = 1e-6 (rstd = 1000)
        # the fp32 rounding of mean * sc alone exceeds one bf16 ulp of a small bias.
        const = (nr.gn_regimes(N, 32) == nr.REGIMES.index("const")).cuda().repeat_interleave(C // 32, 1)
        rc = ref.permute(0, 2, 1)[const]
        assert rc.numel() and torch.equal(rc, b.double().expand(N, C)[const][:, None].expand_as(rc))


_CHILD = textwrap.dedent("""
    import sys
    sys.path[:0] = [{root!r}, {pkg!r}, {tests!r}]
    import torch
    import norm_ref as nr
    from b200sr import _lib, ops
    out = {{}}
    for shape, eps, silu, cs in {cases!r}:
        N, HW, C = shape
        assert _lib.load().b200sr_group_norm_launches(N, HW, C, 32) == 2
        x = nr.gn_inputs(N, HW, C, eps=eps, seed=HW + C).cuda()
        w, b, gam, bet, raw = (t.cuda() for t in nr.gn_params(C, seed=HW + C, sft_shape=shape))
        sft = dict(sft_gamma=gam, sft_beta=bet, raw=raw, control_scale=cs) if cs is not None else {{}}
        out[str((shape, eps, silu, cs))] = ops.group_norm(x, w, b, groups=32, eps=eps, silu=silu, **sft).cpu()
    torch.save(out, {path!r})
""")


def test_one_kernel_equals_two_kernels_bit_for_bit(ops, num_sms, tmp_path):
    """The one-kernel path folds the partials in the fixed order of the two-kernel path (DESIGN.md): the same inputs
    through both give the same bits.  B200SR_GN_FUSED is read once per process, so the two-kernel run is a child."""
    cases = [(s, eps, silu, cs) for s in GN_SHAPES if nr.gn_geometry(*s, 32, num_sms)["launches"] == 1
             for eps, silu, cs in ((1e-5, True, None), (1e-6, False, 0.6))]
    assert cases
    root = os.path.dirname(TESTS)
    pkg = os.path.join(root, "remote-sensing-vision-language-diffusion-model_b200")
    path = str(tmp_path / "two_kernel.pt")
    env = dict(os.environ, B200SR_GN_FUSED="0")
    code = _CHILD.format(root=root, pkg=pkg, tests=TESTS, cases=cases, path=path)
    flags = ["-s"] if sys.flags.no_user_site else []
    r = subprocess.run([sys.executable, *flags, "-c", code], env=env, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-4000:]
    two = torch.load(path)
    for shape, eps, silu, cs in cases:
        N, HW, C = shape
        x, w, b, sft = _gn_case(shape, eps, cs, seed=HW + C)
        one = ops.group_norm(x, w, b, groups=32, eps=eps, silu=silu, **sft).cpu()
        other = two[str((shape, eps, silu, cs))]
        assert torch.equal(one.view(torch.int16), other.view(torch.int16)), f"{shape} eps={eps} silu={silu} cs={cs}"
    print(f"\n[bitwise] one kernel == two kernels on {len(cases)} cases")


# ---------------------------------------------------------------------------------------------------------------------
# group_norm_stats and the fused-input convolution
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("shape,eps", [((2, 1000, 1280), 1e-5), ((1, 136, 128), 1e-6), ((129, 64, 64), 1e-5),
                                       ((1, 1024 * 1024, 128), 1e-6), ((2, 1024, 960), 1e-6)])
def test_group_norm_stats_per_group(ops, num_sms, shape, eps):
    N, HW, C = shape
    x = nr.gn_inputs(N, HW, C, eps=eps, seed=C).cuda()
    st = ops.group_norm_stats(x, 32, eps)
    ref, bound = nr.gn_stats_bounds(x, 32, eps, num_sms)
    what = f"group_norm_stats {shape} eps={eps:g}"
    wm = nr.assert_within(st[..., 0], ref[..., 0], bound[..., 0], what + " mean")
    wr = nr.assert_within(st[..., 1], ref[..., 1], bound[..., 1], what + " rstd")
    _report(what + " mean", wm)
    _report(what + " rstd", wr)


@pytest.mark.parametrize("n,h,w,cin,cout,silu", [(1, 16, 8, 64, 64, True), (3, 48, 40, 128, 256, True),
                                                 (2, 32, 32, 320, 64, False), (1, 256, 256, 64, 64, True)])
def test_conv3x3_fused_input_group_norm_per_element(ops, num_sms, n, h, w, cin, cout, silu):
    """Border pixels of groups with large offsets: the padding must stay 0, not silu(b - mean * a)."""
    x = nr.gn_inputs(n, h * w, cin, seed=cin + h).view(n, h, w, cin).cuda()
    assert ops.conv3x3_gn_fusable(x)
    g = torch.Generator().manual_seed(cout)
    wt = (torch.randn(cout, cin, 3, 3, generator=g) * (1.0 / (9 * cin)) ** 0.5).cuda()
    b = (0.1 * torch.randn(cout, generator=g)).cuda()
    gw, gb = (t.cuda() for t in nr.gn_params(cin, seed=cout))
    st = ops.group_norm_stats(x, 32, 1e-5)
    y = ops.conv3x3(x, ops.pack_conv3x3(wt), b, gn=(st, gw, gb, 32, silu))
    ref, bound = nr.conv3x3_fused_gn(x, wt, b, gw, gb, groups=32, eps=1e-5, silu=silu, num_sms=num_sms)
    what = f"conv3x3 fused GN {n}x{h}x{w} {cin}->{cout} silu={silu}"
    _report(what, nr.assert_within(y, ref, bound, what))


# ---------------------------------------------------------------------------------------------------------------------
# CUDA-graph replay: GroupNorm on both paths and a producer -> consumer LayerNorm fold
# ---------------------------------------------------------------------------------------------------------------------
def test_graph_replay_group_norm_and_fold(ops, num_sms):
    shapes = [(2, 32 * 32, 1280), (8, 32 * 32, 1280)]
    assert sorted(nr.gn_geometry(*s, 32, num_sms)["launches"] for s in shapes) == [1, 2] or num_sms != 148
    M, K, N = 1000, 640, 1920
    xs = [torch.empty(s, dtype=bf16, device="cuda") for s in shapes]
    params = [tuple(t.cuda() for t in nr.gn_params(s[2], seed=i)) for i, s in enumerate(shapes)]
    a_s, r_s = torch.empty(M, K, dtype=bf16, device="cuda"), torch.empty(M, K, dtype=bf16, device="cuda")
    _, w0, _ = nr.fold_producer_inputs(M, K, seed=0)
    w0 = w0.cuda()
    wp, colsum, shift = (t.cuda() for t in nr.fold_weights(N, K, seed=3))

    def load(i):
        for x, s in zip(xs, shapes):
            x.copy_(nr.gn_inputs(*s, seed=100 * i + s[0]))
        a, _, res = nr.fold_producer_inputs(M, K, seed=10 + i)
        a_s.copy_(a)
        r_s.copy_(res)

    def run():
        outs = [ops.group_norm(x, w, b, eps=1e-6, silu=True) for x, (w, b) in zip(xs, params)]
        h, st = ops.gemm(a_s, w0, None, residual=r_s, want_stats=True)
        return outs + [h, st.buf, ops.gemm(h, wp, None, ln=(st, colsum, shift, 1e-5))]

    load(0)
    run()
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        got = run()
    for i in range(3):
        load(i)
        graph.replay()
        torch.cuda.synchronize()
        _gn_counters_zero(ops)
        eager = run()
        torch.cuda.synchronize()
        for g_, e_ in zip(got, eager):
            assert torch.equal(g_, e_), f"replay {i}"
        _gn_counters_zero(ops)
        for x, (w, b), y in zip(xs, params, got[:2]):
            ref, bound = nr.group_norm(x, w, b, eps=1e-6, silu=True, num_sms=num_sms)
            _report(f"graph replay {i} group_norm {tuple(x.shape)}", nr.assert_within(y, ref, bound, f"replay {i}"))
        ref, bound = nr.ln_fold(got[2], wp, got[3], colsum, shift)
        _report(f"graph replay {i} LayerNorm fold", nr.assert_within(got[4], ref, bound, f"replay {i} fold"))


# ---------------------------------------------------------------------------------------------------------------------
# layer_norm: every template, partial lanes
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("M", [1, 77, 333])
@pytest.mark.parametrize("C", [8, 248, 264, 768, 1280, 2560, 2568, 5120])
def test_layer_norm_per_element(ops, M, C):
    x = nr.ln_rows(M, C, seed=M + C).cuda()
    w, b = (t.cuda() for t in nr.gn_params(C, seed=C))
    y = ops.layer_norm(x, w, b, 1e-5)
    ref, bound = nr.layer_norm(x, w, b, 1e-5)
    what = f"layer_norm M={M} C={C} (layer_norm_kernel<{nr.ln_template(C)}>)"
    _report(what, nr.assert_within(y, ref, bound, what))


# ---------------------------------------------------------------------------------------------------------------------
# LayerNorm folded into the GEMMs
# ---------------------------------------------------------------------------------------------------------------------
def _producer(ops, M, K, seed):
    a, w0, res = (t.cuda() for t in nr.fold_producer_inputs(M, K, seed=seed))
    return ops.gemm(a, w0, None, residual=res, want_stats=True)


@pytest.mark.parametrize("M,K,N,kind", [(2048, 1280, 3840, "plain"), (2048, 1280, 10240, "geglu"),
                                        (8192, 640, 1920, "plain"), (8192, 640, 5120, "geglu"), (300, 320, 200, "plain"),
                                        (768, 320, 640, "groups")])
def test_ln_fold_consumer_per_element(ops, M, K, N, kind):
    x, st = _producer(ops, M, K, seed=M + N)
    groups = 3 if kind == "groups" else 1
    rpg = 256 if kind == "groups" else 0
    wp, colsum, shift = (t.cuda() for t in nr.fold_weights(N, K, groups=groups, seed=N, geglu=kind == "geglu"))
    y = ops.gemm(x, wp, None, geglu=kind == "geglu", w_rows_per_group=rpg, ln=(st, colsum, shift, 1e-5))
    ref, bound = nr.ln_fold(x, wp, st.buf, colsum, shift, 1e-5, geglu=kind == "geglu", w_rows_per_group=rpg)
    what = f"LayerNorm fold consumer {kind} {M}x{K}->{N} parts={st.parts}"
    _report(what, nr.assert_within(y, ref, bound, what))


@pytest.mark.parametrize("M,K,N", [(2048, 1280, 1280), (8192, 640, 640), (300, 320, 200)])
def test_ln_fold_producer_partials(ops, M, K, N):
    a, w0, res = (t.cuda() for t in nr.fold_producer_inputs(M, K, seed=N))
    w0 = w0[:N].contiguous()
    res = res[:, :N].contiguous()
    y, st = ops.gemm(a, w0, None, residual=res, want_stats=True)
    bn = ops.gemm_n_tile(M, N, K)
    ref, bound = nr.ln_partials(y, bn)
    what = f"LayerNorm fold producer {M}x{K}->{N} BN={bn}"
    _report(what, nr.assert_within(st.buf.reshape(-1, 2), ref.reshape(-1, 2), bound.reshape(-1, 2), what))


def test_ln_fold_consume_residual_and_produce_in_one_launch(ops):
    M, K, N = 2048, 640, 640
    x, st = _producer(ops, M, K, seed=5)
    wp, colsum, shift = (t.cuda() for t in nr.fold_weights(N, K, seed=6))
    _, _, res2 = nr.fold_producer_inputs(M, N, seed=7)
    res2 = res2.cuda()
    y, st2 = ops.gemm(x, wp, None, residual=res2, ln=(st, colsum, shift, 1e-5), want_stats=True)
    ref, bound = nr.ln_fold(x, wp, st.buf, colsum, shift, 1e-5, residual=res2)
    _report("fold consume + residual + produce: output", nr.assert_within(y, ref, bound, "consume+produce output"))
    ref, bound = nr.ln_partials(y, ops.gemm_n_tile(M, N, K))
    _report("fold consume + residual + produce: partials",
            nr.assert_within(st2.buf.reshape(-1, 2), ref.reshape(-1, 2), bound.reshape(-1, 2), "consume+produce stats"))


@pytest.mark.parametrize("M,N,K", [(300, 200, 320), (1000, 640, 128)])
def test_ln_stats_written_inside_their_window_only(ops, lib, M, N, K):
    """The statistics buffer handed through the C ABI as a window of a NaN-filled guard buffer: every partial inside it
    is written (and right), nothing outside it -- rows >= M of the last M tile included."""
    g = torch.Generator().manual_seed(M)
    a = torch.randn(M, K, generator=g).to(bf16).cuda()
    w0 = (torch.randn(N, K, generator=g) * K ** -0.5 + 0.05).to(bf16).cuda()
    bn = ops.gemm_n_tile(M, N, K)
    parts = -(-N // bn)
    pad = 4096
    guard = torch.full((2 * pad + parts * M * 2,), float("nan"), device="cuda")
    window = guard[pad:pad + parts * M * 2]
    out = torch.empty(M, N, dtype=bf16, device="cuda")
    e = ops._epilogue(out, N, None, None, 0, None, 0, False, False, 1.0)
    e.ln_stats_out = window.data_ptr()
    rc = lib.b200sr_gemm_bf16(a.data_ptr(), K, w0.data_ptr(), M, N, K, ctypes.byref(e), 0, ops._stream())
    assert rc == 0
    torch.cuda.synchronize()
    assert bool(guard[:pad].isnan().all()) and bool(guard[pad + parts * M * 2:].isnan().all())
    assert bool(window.isfinite().all())
    assert torch.equal(out, ops.gemm(a, w0))
    ref, bound = nr.ln_partials(out, bn)
    what = f"statistics window {M}x{K}->{N} BN={bn}"
    _report(what, nr.assert_within(window.view(-1, 2), ref.reshape(-1, 2), bound.reshape(-1, 2), what))
