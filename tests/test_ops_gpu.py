"""Per-kernel parity: every C-ABI op against a plain fp32 torch statement of the same op.

Tolerances: operands are rounded to bf16 once on both sides, accumulation is fp32, outputs are
rounded to bf16 -> relative L2 error <= 1e-2 (BASELINE.json tolerance for the whole step) and in
practice ~3e-3 per op.
"""
import math

import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu
bf16 = torch.bfloat16


def rel_l2(a, b):
    a, b = a.float(), b.float()
    return ((a - b).norm() / (b.norm() + 1e-12)).item()


@pytest.fixture(scope="module")
def ops():
    from b200sr import ops as _ops

    return _ops


def _rand(*shape, scale=1.0, seed=0):
    g = torch.Generator(device="cuda").manual_seed(seed)
    return torch.randn(*shape, generator=g, device="cuda") * scale


@pytest.mark.parametrize(
    "M,N,K,bn",
    [(128, 128, 64, 0), (256, 320, 320, 0), (2048, 1280, 1280, 0), (2, 1280, 320, 0), (154, 640, 2048, 0),
     (333, 72, 200, 0), (8192, 640, 640, 0), (512, 256, 512, 32), (512, 256, 512, 64), (512, 512, 512, 256),
     (1024, 1280, 5120, 0)],
)
def test_gemm_bias(ops, M, N, K, bn):
    a = _rand(M, K, seed=1).to(bf16)
    w = (_rand(N, K, seed=2) / math.sqrt(K)).to(bf16)
    b = _rand(N, seed=3)
    out = ops.gemm(a, w, b, force_bn=bn)
    ref = a.float() @ w.float().t() + b
    assert out.shape == (M, N)
    assert rel_l2(out, ref) < 5e-3


def test_gemm_residual_alpha_rowvec_fp32(ops):
    M, N, K = 1024, 640, 640
    a = _rand(M, K, seed=1).to(bf16)
    w = (_rand(N, K, seed=2) / math.sqrt(K)).to(bf16)
    b = _rand(N, seed=3)
    res = _rand(M, N, seed=4).to(bf16)
    rv = _rand(2, N, seed=5)
    out = ops.gemm(a, w, b, residual=res, alpha=0.5, rowvec=rv, rows_per_group=512)
    ref = 0.5 * (a.float() @ w.float().t() + b) + rv.repeat_interleave(512, 0) + res.float()
    assert rel_l2(out, ref) < 5e-3
    out32 = ops.gemm(a, w, b, out_fp32=True)
    assert out32.dtype == torch.float32
    assert rel_l2(out32, a.float() @ w.float().t() + b) < 2e-3


def test_gemm_out_slice(ops):
    M, N, K = 256, 320, 640
    a = _rand(M, K, seed=1).to(bf16)
    w = (_rand(N, K, seed=2) / math.sqrt(K)).to(bf16)
    res = _rand(M, N, seed=4).to(bf16)
    buf = torch.zeros(M, 960, dtype=bf16, device="cuda")
    ops.gemm(a, w, None, residual=res, out=buf[:, 640:])
    ref = a.float() @ w.float().t() + res.float()
    assert rel_l2(buf[:, 640:], ref) < 5e-3
    assert buf[:, :640].abs().max().item() == 0


@pytest.mark.parametrize("M,C", [(2048, 1280), (512, 640), (130, 320)])
def test_gemm_geglu(ops, M, C):
    inner = 4 * C
    x = _rand(M, C, seed=1).to(bf16)
    w = (_rand(2 * inner, C, seed=2) / math.sqrt(C))
    b = _rand(2 * inner, seed=3) * 0.1
    wp, bp = ops.pack_geglu(w, b)
    out = ops.gemm(x, wp, bp, geglu=True)
    y = x.float() @ w.to(bf16).float().t() + b
    val, gate = y.chunk(2, dim=-1)
    ref = val * F.gelu(gate)
    assert out.shape == (M, inner)
    assert rel_l2(out, ref) < 6e-3


@pytest.mark.parametrize(
    "N,H,W,Cin,Cout,stride",
    [(2, 32, 32, 64, 64, 1), (2, 16, 16, 128, 320, 1), (1, 128, 128, 320, 320, 1), (2, 64, 64, 640, 640, 1),
     (2, 32, 32, 1280, 1280, 1), (2, 8, 8, 128, 64, 1), (3, 4, 4, 64, 128, 1), (2, 24, 40, 64, 96, 1),
     # halo-tile path (stride 1, W % 8 == 0, H >= 16): partial tiles in H, odd image counts (cluster round-up),
     # 1 / 3 / 5 channel chunks (halo ring of depth 1 / 2 wrapping), Cout not a multiple of the N tile
     (3, 40, 8, 64, 72, 1), (1, 16, 24, 192, 128, 1), (5, 48, 16, 320, 256, 1), (1, 17, 8, 128, 64, 1),
     (1, 16, 8, 64, 512, 1),  # a single M block (no CTA pair) with a wide N tile
    
     (2, 32, 32, 64, 64, 2), (2, 128, 128, 320, 320, 2), (2, 16, 16, 128, 128, 2), (1, 8, 8, 64, 64, 2)],
)
def test_conv3x3(ops, N, H, W, Cin, Cout, stride):
    x = _rand(N, Cin, H, W, seed=1).to(bf16)
    w = (_rand(Cout, Cin, 3, 3, seed=2) / math.sqrt(9 * Cin))
    b = _rand(Cout, seed=3)
    emb = _rand(N, Cout, seed=4)
    ref = F.conv2d(x.float(), w.to(bf16).float(), b, stride=stride, padding=1) + emb[:, :, None, None]
    res = _rand(*ref.shape, seed=5).to(bf16)
    ref = ref + res.float()
    out = ops.conv3x3(x.permute(0, 2, 3, 1).contiguous(), ops.pack_conv3x3(w), b, stride=stride, rowvec=emb,
                      residual=res.permute(0, 2, 3, 1).contiguous())
    assert rel_l2(out.permute(0, 3, 1, 2), ref) < 5e-3


@pytest.mark.parametrize("N,H,W,C,eps,silu", [(2, 128, 128, 320, 1e-5, True), (2, 32, 32, 1280, 1e-6, False),
                                              (2, 32, 32, 2560, 1e-5, True), (1, 16, 16, 64, 1e-5, True),
                                              (3, 8, 8, 960, 1e-5, True), (2, 64, 64, 1920, 1e-5, False)])
def test_group_norm(ops, N, H, W, C, eps, silu):
    x = (_rand(N, C, H, W, seed=1) * 2 + 0.7).to(bf16)
    g = _rand(C, seed=2) * 0.3 + 1.0
    b = _rand(C, seed=3) * 0.3
    ref = F.group_norm(x.float(), 32, g, b, eps)
    if silu:
        ref = F.silu(ref)
    out = ops.group_norm(x.permute(0, 2, 3, 1).contiguous(), g, b, eps=eps, silu=silu)
    assert rel_l2(out.permute(0, 3, 1, 2), ref) < 5e-3


def test_group_norm_sft(ops):
    N, H, W, C = 2, 32, 32, 640
    x = _rand(N, H, W, C, seed=1).to(bf16)
    gamma = (_rand(N, H, W, C, seed=2) * 0.2).to(bf16)
    beta = (_rand(N, H, W, C, seed=3) * 0.2).to(bf16)
    raw = _rand(N, H, W, C, seed=4).to(bf16)
    g = _rand(C, seed=5) * 0.3 + 1.0
    b = _rand(C, seed=6) * 0.3
    xn = F.group_norm(x.float().permute(0, 3, 1, 2), 32, g, b, 1e-5).permute(0, 2, 3, 1)
    for s in (1.0, 0.6):
        ref = (xn * (1 + gamma.float()) + beta.float()) * s + raw.float() * (1 - s)
        out = ops.group_norm(x, g, b, sft_gamma=gamma, sft_beta=beta, raw=raw, control_scale=s)
        assert rel_l2(out, ref) < 5e-3


@pytest.mark.parametrize("M,C", [(2048, 1280), (8192, 640), (77, 320), (5, 2560)])
def test_layer_norm(ops, M, C):
    x = (_rand(M, C, seed=1) * 1.5 + 0.3).to(bf16)
    g = _rand(C, seed=2) * 0.3 + 1.0
    b = _rand(C, seed=3) * 0.3
    out = ops.layer_norm(x, g, b, 1e-5)
    assert rel_l2(out, F.layer_norm(x.float(), (C,), g, b, 1e-5)) < 5e-3


@pytest.mark.parametrize("B,H,Nq,Nk", [(2, 20, 1024, 1024), (2, 10, 4096, 4096), (2, 10, 4096, 77), (2, 20, 1024, 77),
                                       (1, 2, 256, 256), (2, 5, 64, 64), (1, 3, 200, 333), (2, 4, 128, 640),
                                       # tail-split plans: all tiles in the partial wave, ragged last key block / 5 key
                                       # blocks over 3 ranges / one more tile than a full wave of 296
                                       (1, 4, 256, 1000), (1, 2, 300, 640), (1, 33, 1152, 512)])
def test_attention(ops, B, H, Nq, Nk):
    C = H * 64
    q = _rand(B, Nq, C, seed=1).to(bf16)
    k = _rand(B, Nk, C, seed=2).to(bf16)
    v = _rand(B, Nk, C, seed=3).to(bf16)
    out = ops.attention(q, k, v, H)
    qf, kf, vf = (t.float().view(B, -1, H, 64).transpose(1, 2) for t in (q, k, v))
    ref = F.scaled_dot_product_attention(qf, kf, vf).transpose(1, 2).reshape(B, Nq, C)
    assert rel_l2(out, ref) < 8e-3


def test_attention_fused_qkv_and_peaky(ops):
    B, H, N = 2, 10, 1024
    C = H * 64
    qkv = (_rand(B, N, 3 * C, seed=1) * 3.0).to(bf16)  # large logits -> exercises the lazy rescale
    out = ops.attention(qkv, qkv, qkv, H, q_col=0, k_col=C, v_col=2 * C)
    q, k, v = qkv.float().split(C, dim=-1)
    qf, kf, vf = (t.reshape(B, N, H, 64).transpose(1, 2) for t in (q, k, v))
    ref = F.scaled_dot_product_attention(qf, kf, vf).transpose(1, 2).reshape(B, N, C)
    assert rel_l2(out, ref) < 8e-3


@pytest.mark.parametrize("B,T,C,H,Tk", [(2, 1024, 1280, 20, 77), (2, 4096, 640, 10, 77), (1, 256, 128, 2, 33)])
def test_gemm_grouped_weights_and_head_softmax_epilogue(ops, B, T, C, H, Tk):
    """Folded cross-attention building blocks: per-batch-element weights (w_rows_per_group) and the per-head
    softmax epilogue over 80-column segments (first Tk columns valid, base 2, pad -> 0)."""
    x = _rand(B, T, C, seed=1).to(bf16)
    kf = (_rand(B, H * 80, C, seed=2) * 0.08).to(bf16)
    p = ops.gemm(x, kf, softmax_valid=Tk, w_rows_per_group=T)
    logits = torch.einsum("btc,bnc->btn", x.float(), kf.float()).view(B, T, H, 80)
    logits[..., Tk:] = float("-inf")
    ref = torch.softmax(logits * math.log(2.0), dim=-1).reshape(B, T, H * 80)
    assert p.shape == ref.shape and rel_l2(p, ref) < 8e-3
    assert float(p.view(B, T, H, 80)[..., Tk:].abs().max()) == 0.0
    vf = (_rand(B, C, H * 80, seed=3) * 0.1).to(bf16)
    bias = _rand(C, seed=4) * 0.1
    res = _rand(B, T, C, seed=5).to(bf16)
    out = ops.gemm(p, vf, bias, residual=res, alpha=0.7, w_rows_per_group=T)
    ref2 = 0.7 * (torch.einsum("btn,bcn->btc", p.float(), vf.float()) + bias) + res.float()
    assert rel_l2(out, ref2) < 8e-3


def test_gemm_dynamic_w_operand_inside_a_graph(ops):
    """An activation used as the B operand (SR3's single-head attention computes Q K^T and P V as GEMMs) must not be
    prefetched ahead of the kernel's programmatic dependency: inside a CUDA graph the producer is still running."""
    x = _rand(4096, 512, seed=1).to(bf16)
    wq = (_rand(512, 512, seed=2) * 0.05).to(bf16)
    wk = (_rand(512, 512, seed=3) * 0.05).to(bf16)
    xs = torch.empty_like(x)

    def chain():
        q, k = ops.gemm(xs, wq), ops.gemm(xs, wk)
        return ops.gemm(q, k, out_fp32=True, w_dynamic=True)

    xs.copy_(x)
    chain()
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        s_g = chain()
    for scale in (1.0, -0.5, 2.0):  # new producer outputs every replay: a stale prefetch of k would show
        xs.copy_(x * scale)
        g.replay()
        torch.cuda.synchronize()
        q = (xs.float() @ wq.float().t()).to(bf16).float()
        k = (xs.float() @ wk.float().t()).to(bf16).float()
        assert rel_l2(s_g, q @ k.t()) < 8e-3
        assert torch.equal(s_g, chain())


def test_attention_split_is_deterministic_and_leaves_counters_zero(ops):
    """The last partial wave of tiles is split over the key range and merged by the last CTA to arrive:
    repeated calls must agree bit for bit and the arrival counters must be back at zero."""
    from b200sr import ops as _ops
    B, H, N = 2, 20, 1024  # 320 tiles = 296 + 24 -> the 24 tail tiles are split over the key range
    C = H * 64
    qkv = _rand(B, N, 3 * C, seed=7).to(bf16)
    outs = [ops.attention(qkv, qkv, qkv, H, q_col=0, k_col=C, v_col=2 * C) for _ in range(4)]
    torch.cuda.synchronize()
    for o in outs[1:]:
        assert torch.equal(o, outs[0])
    ws = [w for key, w in _ops._ws_cache.items() if key[-1] == "attn"]
    assert ws, "the split plan should have asked for a workspace"
    for w in ws:
        assert int(w[:512].view(torch.int32).abs().sum()) == 0


def test_layout_strided_upsample_concat_misc(ops):
    x = _rand(2, 4, 16, 24, seed=1)
    y = ops.nchw_to_nhwc_bf16(x, 0.5)
    assert torch.equal(y, (x * 0.5).to(bf16).permute(0, 2, 3, 1).contiguous())
    z = _rand(2, 16, 24, 320, seed=2).to(bf16)
    from b200sr import _lib
    for c in (4, 320):   # the first 4 of 320 channels: the stride of the <= 4-channel convolutions' padded output
        y = torch.empty(2, c, 16, 24, device="cuda")
        assert _lib.load().b200sr_nhwc_bf16_to_nchw_f32_strided(z.data_ptr(), y.data_ptr(), 2, c, 320, 16 * 24,
                                                                ops._stream()) == 0
        assert torch.equal(y, z[..., :c].float().permute(0, 3, 1, 2).contiguous())
    up = ops.upsample2x(z)
    ref = F.interpolate(z.float().permute(0, 3, 1, 2), scale_factor=2, mode="nearest").permute(0, 2, 3, 1).to(bf16)
    assert torch.equal(up, ref.contiguous())
    a = _rand(2, 8, 8, 640, seed=3).to(bf16)
    b = _rand(2, 8, 8, 320, seed=4).to(bf16)
    c = _rand(2, 8, 8, 320, seed=5).to(bf16)
    cat = ops.concat_add(a, b, c)
    assert torch.equal(cat, torch.cat([a, (b.float() + c.float()).to(bf16)], dim=-1))
    assert torch.equal(ops.concat_add(a, b), torch.cat([a, b], dim=-1))
    assert rel_l2(ops.axpy(b, c, 0.5), b.float() + 0.5 * c.float()) < 4e-3
    assert rel_l2(ops.silu(b), F.silu(b.float())) < 4e-3
    t = torch.tensor([999.0, 3.0], device="cuda")
    emb = ops.sinusoid_embedding(t, 320)
    half = 160
    freqs = torch.exp(-math.log(10000) * torch.arange(half, device="cuda", dtype=torch.float32) / half)
    args = t[:, None] * freqs[None]
    ref = torch.cat([torch.cos(args), torch.sin(args)], -1)
    assert (emb.float() - ref).abs().max().item() < 1e-2
    emb2 = ops.sinusoid_embedding(torch.tensor([0.7], device="cuda"), 64, sin_first=True)
    step = torch.arange(32, device="cuda", dtype=torch.float32) / 32
    enc = 0.7 * torch.exp(-math.log(1e4) * step)
    assert (emb2.float()[0] - torch.cat([torch.sin(enc), torch.cos(enc)])).abs().max().item() < 1e-2


def test_sampler_kernels(ops):
    B, C, H, W = 1, 4, 32, 32
    x = _rand(B, C, H, W, seed=1) * 10
    noise = _rand(B, C, H, W, seed=2)
    sigma, gamma, sigma_next, sigma_q, cfg, s_noise = 14.6146, 0.1, 12.0, 14.3, 5.5, 1.003
    sigma_hat = sigma * (1 + gamma)
    sc = torch.tensor([sigma, sigma_hat, sigma_next, sigma_q, cfg, s_noise], device="cuda")
    x_hat, net_in = ops.sampler_pre(x, noise, sc, 2)
    ref_hat = x + noise * s_noise * (sigma_hat**2 - sigma**2) ** 0.5
    assert torch.allclose(x_hat, ref_hat, rtol=1e-5, atol=1e-5)
    ref_in = (ref_hat / (sigma_q**2 + 1) ** 0.5).to(bf16).permute(0, 2, 3, 1)
    assert rel_l2(net_in[0], ref_in[0]) < 1e-3 and torch.equal(net_in[0], net_in[1])
    eps = _rand(2 * B, C, H, W, seed=3)
    x_next, den = ops.sampler_post(eps, x_hat, sc)
    du, dc = eps[:B] * -sigma_q + ref_hat, eps[B:] * -sigma_q + ref_hat
    rden = du + cfg * (dc - du)
    rnext = ref_hat + (ref_hat - rden) / sigma_hat * (sigma_next - sigma_hat)
    assert torch.allclose(den, rden, rtol=1e-4, atol=1e-4) and torch.allclose(x_next, rnext, rtol=1e-4, atol=1e-4)
    assert torch.allclose(ops.euler_from_denoised(den, x_hat, sc), x_next, rtol=1e-5, atol=1e-5)
    # similarity
    a = _rand(2, 32, 32, 1280, seed=4).to(bf16)
    b = (a.float() + 0.1 * _rand(2, 32, 32, 1280, seed=5)).to(bf16)
    thr = torch.tensor([0.3], device="cuda")
    r = ops.rel_l1_similarity(a, b, thr)
    ref = ((a.float() - b.float()).abs().mean() / (a.float().abs().mean() + 1e-6)).item()
    assert abs(r[0].item() - ref) < 1e-5 * max(1, ref) and r[1].item() == float(ref < 0.3)
    r2 = ops.rel_l1_similarity(a, b, torch.tensor([0.01], device="cuda"))
    assert abs(r2[0].item() - ref) < 1e-5 and r2[1].item() == 0.0
    # tile blend
    acc = torch.zeros(1, 4, 48, 48, device="cuda")
    cnt = torch.zeros_like(acc)
    wgt = torch.rand(32, 32, device="cuda") + 0.1
    tiles = [(0, 0), (0, 16), (16, 0), (16, 16)]
    racc, rcnt = torch.zeros_like(acc), torch.zeros_like(acc)
    for i, (h0, w0) in enumerate(tiles):
        t = _rand(1, 4, 32, 32, seed=10 + i)
        ops.tile_accumulate(t, wgt, acc, cnt, h0, w0)
        racc[:, :, h0:h0 + 32, w0:w0 + 32] += t * wgt
        rcnt[:, :, h0:h0 + 32, w0:w0 + 32] += wgt
    assert torch.allclose(ops.tile_normalize(acc, cnt), racc / rcnt, rtol=1e-5, atol=1e-6)
    # sr3 update
    x3, e3, n3 = _rand(1, 3, 16, 16, seed=20), _rand(1, 3, 16, 16, seed=21), _rand(1, 3, 16, 16, seed=22)
    s5 = torch.tensor([1.2, 0.66, 0.4, 0.58, -3.0], device="cuda")
    x0 = (1.2 * x3 - 0.66 * e3).clamp(-1, 1)
    ref = 0.4 * x0 + 0.58 * x3 + n3 * math.exp(-1.5)
    assert torch.allclose(ops.sr3_update(x3, e3, n3, s5), ref, rtol=1e-5, atol=1e-5)
