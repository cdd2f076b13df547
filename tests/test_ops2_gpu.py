"""GPU parity of the round-2 operator additions against plain torch fp32 references: the chunked single-head attention
helper, copy_batch, weighted strips."""
import pytest
import torch

pytestmark = pytest.mark.gpu
bf16 = torch.bfloat16


def rel_l2(a, b):
    a, b = a.float(), b.float()
    return ((a - b).norm() / (b.norm() + 1e-12)).item()


@pytest.mark.parametrize("t,chunk", [(1024, 1 << 30), (4096, 4 * 4096 * 1024)])
def test_single_head_attention_chunked(t, chunk, monkeypatch):
    from b200sr import ops

    monkeypatch.setattr(ops, "SCORE_CHUNK_BYTES", chunk)      # second case: 4 query chunks
    g = torch.Generator(device="cuda").manual_seed(t)
    c = 512
    q = (torch.randn(t, c, generator=g, device="cuda") * 0.5).to(bf16)
    k = (torch.randn(t, c, generator=g, device="cuda") * 0.5).to(bf16)
    v = (torch.randn(t, c, generator=g, device="cuda") * 0.5).to(bf16)
    bias = torch.randn(c, generator=g, device="cuda")
    o = ops.single_head_attention(q, k, v.t().contiguous(), c ** -0.5, out_bias=bias)
    ref = torch.softmax(q.float() @ k.float().t() * c ** -0.5, -1) @ v.float() + bias
    assert rel_l2(o, ref) < 1e-2


def test_copy_batch_and_strips():
    from b200sr import ops

    g = torch.Generator(device="cuda").manual_seed(1)
    srcs = [torch.randn(n, generator=g, device="cuda") for n in (6, 1000, 4096, 3, 65536, 7, 128, 12)]
    dsts = [torch.zeros_like(s) for s in srcs]
    ops.copy_batch(list(zip(dsts, srcs)))
    assert all(torch.equal(d, s) for d, s in zip(dsts, srcs))
    h = torch.randn(2, 8, 16, generator=g, device="cuda").to(bf16)
    d = torch.zeros_like(h)
    ops.copy_batch([(d, h)])
    assert torch.equal(d, h)
    tile = torch.randn(1, 4, 32, 32, generator=g, device="cuda")
    w = torch.rand(32, 32, generator=g, device="cuda")
    acc1, acc2 = torch.zeros(1, 4, 64, 64, device="cuda"), torch.zeros(1, 4, 64, 64, device="cuda")
    ops.tile_accumulate(tile, w, acc1, None, 8, 24)
    # the same contribution shipped as two strips and added on the "owner": identical bits
    for (y0, x0, sh, sw) in ((0, 0, 32, 10), (0, 10, 32, 22)):
        ops.strip_add(ops.tile_weighted_strip(tile, w, y0, x0, sh, sw), acc2, 8 + y0, 24 + x0)
    assert torch.equal(acc1, acc2)
    assert torch.equal(acc1[:, :, 8:40, 24:56], tile * w)


@pytest.mark.parametrize("n,h,w,cin,cout,extras", [
    (2, 32, 32, 1280, 1280, "rowvec"), (2, 128, 128, 320, 320, "residual"), (1, 64, 64, 640, 320, ""),
    (1, 16, 8, 64, 64, ""), (1, 256, 256, 64, 64, "residual"), (3, 48, 40, 128, 256, "rowvec"), (1, 1024, 64, 128, 64, ""),
])
def test_conv3x3_with_fused_input_groupnorm(n, h, w, cin, cout, extras):
    """GroupNorm + SiLU applied to the staged input tiles inside the halo convolution == GroupNorm kernel followed by the
    convolution, bit for bit (same arithmetic, same bf16 rounding point), and == a torch fp32 reference within bf16."""
    import torch.nn.functional as F
    from b200sr import ops

    g = torch.Generator(device="cuda").manual_seed(n * 1000 + h + cin)
    x = (torch.randn(n, h, w, cin, generator=g, device="cuda") * 1.5 + 0.3).to(bf16)
    wt = torch.randn(cout, cin, 3, 3, generator=g, device="cuda") * (1.0 / (9 * cin)) ** 0.5
    b = torch.randn(cout, generator=g, device="cuda") * 0.1
    gw = 1 + 0.1 * torch.randn(cin, generator=g, device="cuda")
    gb = 0.1 * torch.randn(cin, generator=g, device="cuda")
    kw = {}
    if extras == "rowvec":
        kw["rowvec"] = torch.randn(n, cout, generator=g, device="cuda")
    if extras == "residual":
        kw["residual"] = torch.randn(n, h, w, cout, generator=g, device="cuda").to(bf16)
    assert ops.conv3x3_gn_fusable(x)
    wp = ops.pack_conv3x3(wt)
    two = ops.conv3x3(ops.group_norm(x, gw, gb, groups=32, eps=1e-5, silu=True), wp, b, **kw)
    stats = ops.group_norm_stats(x, 32, 1e-5)
    fused = ops.conv3x3(x, wp, b, gn=(stats, gw, gb, 32, True), **kw)
    assert torch.equal(fused, two)
    xf = x.float().permute(0, 3, 1, 2)
    y = F.silu(F.group_norm(xf, 32, gw, gb, 1e-5)).to(bf16).float()
    ref = F.conv2d(y, wt.to(bf16).float(), b, padding=1).permute(0, 2, 3, 1)
    if "rowvec" in kw:
        ref = ref + kw["rowvec"][:, None, None, :]
    if "residual" in kw:
        ref = ref + kw["residual"].float()
    assert rel_l2(fused, ref) < 5e-3
    mean = xf.reshape(n, 32, -1).mean(-1)
    assert torch.allclose(stats[..., 0], mean, atol=2e-3)


def _row_stats_ref(y):
    y = y.float().reshape(-1, y.shape[-1])
    return y.mean(1), y.var(1, unbiased=False)


@pytest.mark.parametrize("m,k,n", [(2048, 1280, 1280), (8192, 640, 640), (300, 320, 200)])
def test_gemm_row_statistics_of_the_output(m, k, n):
    """want_stats: the per-N-tile partial (sum, sum of squares) of the output rows fold to the rows' mean / variance."""
    from b200sr import ops

    g = torch.Generator(device="cuda").manual_seed(m + n)
    a = torch.randn(m, k, generator=g, device="cuda").to(bf16)
    w = (torch.randn(n, k, generator=g, device="cuda") * k ** -0.5).to(bf16)
    b = torch.randn(n, generator=g, device="cuda")
    res = (torch.randn(m, n, generator=g, device="cuda") * 3 + 1.5).to(bf16)
    plain = ops.gemm(a, w, b, residual=res)
    y, st = ops.gemm(a, w, b, residual=res, want_stats=True)
    assert torch.equal(y, plain)                                   # same arithmetic with or without the statistics
    assert st.parts == -(-n // ops.gemm_n_tile(m, n, k)) and st.buf.shape == (st.parts, m, 2) and st.dim == n
    tot = st.buf.sum(0)
    mean, var = _row_stats_ref(y)
    # the kernel sums the fp32 values before their rounding to bf16: |mean error| ~ 2^-9 |x| / sqrt(n)
    assert torch.allclose(tot[:, 0] / n, mean, atol=2e-3, rtol=1e-3)
    assert torch.allclose(tot[:, 1] / n - (tot[:, 0] / n) ** 2, var, atol=2e-2, rtol=2e-3)


@pytest.mark.parametrize("m,c,n,kind", [(2048, 1280, 3840, "plain"), (8192, 640, 1920, "plain"), (2048, 1280, 10240, "geglu"),
                                        (8192, 640, 5120, "geglu"), (300, 320, 200, "plain")])
def test_layer_norm_folded_into_gemm(m, c, n, kind):
    """gemm(ln=...) on the raw rows == gemm(layer_norm(rows)): compared against the fp32 composition, and required to be
    at least as close to it as the two-kernel bf16 path (which rounds the normalised rows to bf16 in between)."""
    from b200sr import ops

    g = torch.Generator(device="cuda").manual_seed(m + n)
    # the residual stream: written by a producing GEMM (bias + residual), rows with a non-zero mean
    a = torch.randn(m, c, generator=g, device="cuda").to(bf16)
    w0 = (torch.randn(c, c, generator=g, device="cuda") * c ** -0.5).to(bf16)
    res = (torch.randn(m, c, generator=g, device="cuda") * 2 + 0.7).to(bf16)
    x, st = ops.gemm(a, w0, None, residual=res, want_stats=True)
    gamma = 1 + 0.3 * torch.randn(c, generator=g, device="cuda")
    beta = 0.2 * torch.randn(c, generator=g, device="cuda")
    w = torch.randn(n, c, generator=g, device="cuda") * c ** -0.5
    b = 0.1 * torch.randn(n, generator=g, device="cuda")
    ln32 = torch.nn.functional.layer_norm(x.float(), (c,), gamma, beta, 1e-5)
    if kind == "geglu":
        ref = ln32 @ w.t() + b
        ref = ref[:, :n // 2] * torch.nn.functional.gelu(ref[:, n // 2:])
        wp, colsum, shift = ops.pack_geglu_ln(w, b, gamma, beta)
        y = ops.gemm(x, wp, None, geglu=True, ln=(st, colsum, shift, 1e-5))
        w2, b2 = ops.pack_geglu(w, b)
        two = ops.gemm(ops.layer_norm(x, gamma, beta, 1e-5), w2, b2, geglu=True)
    else:
        ref = ln32 @ w.t() + b
        wp, colsum, shift = ops.pack_linear_ln(w, gamma, beta, b)
        y = ops.gemm(x, wp, None, ln=(st, colsum, shift, 1e-5))
        two = ops.gemm(ops.layer_norm(x, gamma, beta, 1e-5), ops.pack_linear(w), b)
    e_fold, e_two = rel_l2(y, ref), rel_l2(two, ref)
    assert e_fold < 6e-3 and e_fold <= 1.1 * e_two, (e_fold, e_two)


@pytest.mark.parametrize("b,t,c,heads", [(2, 1024, 1280, 20), (4, 1024, 1280, 20), (2, 4096, 640, 10)])
def test_layer_norm_folded_into_bound_cross_attention(b, t, c, heads):
    """The folded-key product with per-batch-element keys and the per-head softmax epilogue, LayerNorm folded in."""
    from b200sr import ops

    g = torch.Generator(device="cuda").manual_seed(b * t + c)
    a = torch.randn(b * t, c, generator=g, device="cuda").to(bf16)
    w0 = (torch.randn(c, c, generator=g, device="cuda") * c ** -0.5).to(bf16)
    res = (torch.randn(b * t, c, generator=g, device="cuda") * 2 - 0.4).to(bf16)
    x, st = ops.gemm(a, w0, None, residual=res, want_stats=True)
    gamma = 1 + 0.3 * torch.randn(c, generator=g, device="cuda")
    beta = 0.2 * torch.randn(c, generator=g, device="cuda")
    groups, seg, tk = 2, 80, 77                                        # [uncond; cond] captions shared by b / 2 latents each
    kp = torch.zeros(groups, heads, seg, c, device="cuda")
    kp[:, :, :tk] = torch.randn(groups, heads, tk, c, generator=g, device="cuda") * (3.0 * c ** -0.5)
    kp = kp.reshape(groups, heads * seg, c)
    kg = (kp * gamma).to(bf16).contiguous()
    colsum, shift = kg.float().sum(-1).contiguous(), (kp @ beta).contiguous()
    rpg = t * (b // groups)
    p = ops.gemm(x.view(b, t, c), kg, softmax_valid=tk, w_rows_per_group=rpg, ln=(st, colsum, shift, 1e-5))
    ln32 = torch.nn.functional.layer_norm(x.float(), (c,), gamma, beta, 1e-5).view(groups, rpg, c)
    logits = torch.einsum("gmc,gnc->gmn", ln32, kp).view(groups, rpg, heads, seg)[..., :tk]
    ref = torch.zeros(groups, rpg, heads, seg, device="cuda")
    ref[..., :tk] = torch.softmax(logits * 0.6931471805599453, dim=-1)                 # the epilogue works in base 2
    two = ops.gemm(ops.layer_norm(x, gamma, beta, 1e-5).view(b, t, c), kp.to(bf16).contiguous(), softmax_valid=tk,
                   w_rows_per_group=rpg)
    e_fold, e_two = rel_l2(p.view(-1), ref.view(-1)), rel_l2(two.view(-1), ref.view(-1))
    assert torch.equal(p.view(groups, rpg, heads, seg)[..., tk:], torch.zeros_like(ref[..., tk:]).to(bf16))
    assert e_fold < 1e-2 and e_fold <= 1.1 * e_two, (e_fold, e_two)


@pytest.mark.parametrize("m,n,k", [(16384, 16384, 512), (5000, 4104, 512), (4096, 8192, 64), (9000, 2056, 1280)])
def test_fp32_output_of_a_many_tile_gemm(m, n, k):
    """fp32 output with several tiles per CTA (attention scores of the SR3 / first-stage single-head attention) leaves
    through the TMA-store epilogue: rows / columns beyond M / N are clipped by the tensor map, alpha and bias apply."""
    from b200sr import ops

    g = torch.Generator(device="cuda").manual_seed(m + n + k)
    a = (torch.randn(m, k, generator=g, device="cuda") * 0.5).to(bf16)
    w = (torch.randn(n, k, generator=g, device="cuda") * 0.5).to(bf16)
    b = torch.randn(n, generator=g, device="cuda")
    guard = torch.full((m + 2, n + 8), 7.0, device="cuda")                 # the output is a window of a wider buffer
    out = guard[1:m + 1, :n]
    ops.gemm(a, w, b, alpha=0.25, out=out, out_fp32=True)
    ref = torch.empty(m, n, device="cuda")
    for r0 in range(0, m, 4096):                                            # fp32 reference in row chunks (memory)
        ref[r0:r0 + 4096] = (a[r0:r0 + 4096].float() @ w.float().t() + b) * 0.25
    assert rel_l2(out, ref) < 2e-6
    assert (out - ref).abs().max().item() < 1e-3
    assert torch.all(guard[0] == 7.0) and torch.all(guard[m + 1] == 7.0) and torch.all(guard[:, n:] == 7.0)


@pytest.mark.parametrize("m,n,valid", [(4096, 4096, None), (1000, 16384, 16001), (256, 1024, 77), (16384, 16384, None),
                                       (300, 2056, 2050)])
def test_two_pass_row_softmax_gemm(m, n, valid):
    """softmax(scale * q k^T) over whole rows from two passes of the GEMM (statistics, then probabilities) against torch on
    the fp32 product; masked columns are exactly 0 and every row sums to 1."""
    from b200sr import ops

    g = torch.Generator(device="cuda").manual_seed(m + n)
    k_dim = 512
    q = (torch.randn(m, k_dim, generator=g, device="cuda") * 0.7).to(bf16)
    k = (torch.randn(n, k_dim, generator=g, device="cuda") * 0.7).to(bf16)
    scale = k_dim ** -0.5
    p = ops.gemm_row_softmax(q, k, scale, valid)
    v = n if valid is None else valid
    assert p.dtype == bf16 and p.shape == (m, n)
    assert torch.equal(p[:, v:], torch.zeros_like(p[:, v:]))
    worst = 0.0
    for r0 in range(0, m, 2048):
        ref = torch.softmax((q[r0:r0 + 2048].float() @ k.float().t())[:, :v] * scale, dim=-1)
        worst = max(worst, rel_l2(p[r0:r0 + 2048, :v], ref))
        assert torch.allclose(p[r0:r0 + 2048].float().sum(-1), torch.ones(ref.shape[0], device="cuda"), atol=2e-2)
    assert worst < 4e-3, worst


def test_single_head_attention_with_bias():
    from b200sr import ops

    g = torch.Generator(device="cuda").manual_seed(11)
    t, c = 4096, 512
    q, k, v = ((torch.randn(t, c, generator=g, device="cuda") * 0.5).to(bf16) for _ in range(3))
    bias = torch.randn(c, generator=g, device="cuda")
    v_t = v.t().contiguous()
    a = ops.single_head_attention(q, k, v_t, c ** -0.5, bias)
    ref = torch.softmax(q.float() @ k.float().t() * c ** -0.5, dim=-1) @ v.float() + bias
    assert rel_l2(a, ref) < 6e-3
