"""TEST DOUBLE for ``b200sr.ops`` — test infrastructure only, never imported by the package.

Plain torch (CPU-capable) stand-ins with the same signatures, dtypes and layouts as the CUDA
ops: bf16 storage, fp32 arithmetic inside each op, result rounded to bf16.  Used by the
``-m "not gpu"`` suite to check the *host wiring* of the drop-in modules (which op is called with
which tensor, residual/concat order, state_dict keys) against the oracle without a GPU, and as a
CPU emulation of the bf16 pipeline's rounding.  The product path never routes through this file:
``b200sr.ops`` has no fallback and raises on non-CUDA tensors.
"""
from __future__ import annotations

import math

import torch
import torch.nn.functional as F

bf16 = torch.bfloat16


def require_cuda(t, what):
    """The double runs anywhere."""


def gemm(a, w, bias=None, *, residual=None, rowvec=None, rows_per_group=0, geglu=False, alpha=1.0, act=0, out=None,
         out_fp32=False, force_bn=0, softmax_valid=0, w_rows_per_group=0, w_dynamic=False, ln=None, want_stats=False):
    a2 = a.float().reshape(-1, a.shape[-1])
    n_groups = (a2.shape[0] + w_rows_per_group - 1) // w_rows_per_group if w_rows_per_group else 1
    if w_rows_per_group:
        y = torch.cat([a2[g * w_rows_per_group:(g + 1) * w_rows_per_group] @ w[g].float().t() for g in range(n_groups)], 0)
    else:
        y = a2 @ w.float().t()
    if ln is not None:
        # the library's arithmetic: statistics from the producer's partial sums, applied around the raw product
        st, colsum, shift, eps = ln
        assert st.buf.shape[1] == a2.shape[0] and st.dim == a2.shape[1]
        tot = st.buf.sum(0)
        mean = tot[:, 0] / st.dim
        rstd = torch.rsqrt((tot[:, 1] / st.dim - mean * mean).clamp_min(0) + eps)
        gidx = torch.arange(a2.shape[0]) // w_rows_per_group if w_rows_per_group else torch.zeros(a2.shape[0], dtype=torch.long)
        cs, sh = colsum.reshape(n_groups, -1)[gidx], shift.reshape(n_groups, -1)[gidx]
        y = rstd[:, None] * (y - mean[:, None] * cs) + sh
    if softmax_valid:
        seg = y.view(y.shape[0], -1, 80).clone()
        seg[:, :, softmax_valid:] = float("-inf")
        y = torch.softmax(seg * math.log(2.0), dim=-1).reshape(y.shape[0], -1)
    if bias is not None:
        y = y + bias
    if geglu:
        n = w.shape[0]
        y = y.view(y.shape[0], n // 32, 2, 16)
        y = (y[:, :, 0] * F.gelu(y[:, :, 1])).reshape(y.shape[0], n // 2)
    else:
        y = y * alpha
        if rowvec is not None:
            g = torch.arange(y.shape[0]) // rows_per_group if rows_per_group else torch.zeros(y.shape[0], dtype=torch.long)
            y = y + rowvec[g]
        if residual is not None:
            y = y + residual.float().reshape(-1, residual.shape[-1])
        if act == 1:
            y = F.silu(y)
        elif act == 2:
            y = F.gelu(y)
        elif act == 3:
            y = y * torch.sigmoid(1.702 * y)
    y = y.reshape(*a.shape[:-1], y.shape[-1])
    y = y if out_fp32 else y.to(bf16)
    stats = None
    if want_stats:
        # two column tiles, like a GEMM whose N tile is half the row
        y2 = y.float().reshape(-1, y.shape[-1])
        half = (y2.shape[1] // 2 + 7) // 8 * 8
        parts = [y2[:, :half], y2[:, half:]]
        stats = RowStats(torch.stack([torch.stack([p.sum(1), (p * p).sum(1)], -1) for p in parts]), 2, y2.shape[1])
    if out is not None:
        out.copy_(y.reshape(out.shape))
        y = out
    return (y, stats) if want_stats else y


def gemm_row_softmax(a, w, scale, valid_cols=None, w_dynamic=True):
    s = a.float().reshape(-1, a.shape[-1]) @ w.float().t()
    return _softmax_rows(s, scale, valid_cols=valid_cols)


class RowStats:
    def __init__(self, buf, parts, dim):
        self.buf, self.parts, self.dim = buf, parts, dim


def conv3x3_gn_fusable(x, stride=1, cout=None):
    ok = stride == 1 and x.dim() == 4 and x.shape[2] % 8 == 0 and x.shape[1] >= 16 and x.shape[3] % 64 == 0
    return ok and (cout is None or cout <= 256)


def group_norm_stats(x, groups=32, eps=1e-5):
    n, c = x.shape[0], x.shape[-1]
    xf = x.float().reshape(n, -1, groups, c // groups)
    mean = xf.mean(dim=(1, 3))
    var = xf.var(dim=(1, 3), unbiased=False)
    return torch.stack([mean, torch.rsqrt(var + eps)], dim=-1)


def conv3x3(x, w, bias=None, *, stride=1, rowvec=None, residual=None, alpha=1.0, act=0, out=None, force_bn=0, pad_lo=1,
            gn=None):
    if gn is not None:
        stats, gw, gb, groups, gsilu = gn
        c = x.shape[-1]
        mean = stats[..., 0].repeat_interleave(c // groups, dim=1)[:, None, None, :]
        rstd = stats[..., 1].repeat_interleave(c // groups, dim=1)[:, None, None, :]
        a = rstd * gw
        y = x.float() * a + (gb - mean * a)
        x = (F.silu(y) if gsilu else y).to(bf16)
    n, h, wd, cin = x.shape
    cout = w.shape[0]
    w4 = w.float().view(cout, 3, 3, cin).permute(0, 3, 1, 2)
    xin = x.float().permute(0, 3, 1, 2)
    if pad_lo == 0:
        assert stride == 2
        y = F.conv2d(F.pad(xin, (0, 1, 0, 1)), w4, bias, stride=2, padding=0) * 1.0
    else:
        y = F.conv2d(xin, w4, bias, stride=stride, padding=1) * 1.0
    if alpha != 1.0:
        y = y * alpha
    if rowvec is not None:
        y = y + rowvec[:, :, None, None]
    y = y.permute(0, 2, 3, 1)
    if residual is not None:
        y = y + residual.float()
    if act == 1:
        y = F.silu(y)
    y = y.to(bf16).contiguous()
    if out is not None:
        out.copy_(y)
        return out
    return y


def group_norm(x, weight, bias, *, groups=32, eps=1e-5, silu=False, sft_gamma=None, sft_beta=None, raw=None,
               control_scale=1.0):
    shape = x.shape
    n, c = shape[0], shape[-1]
    xf = x.float().reshape(n, -1, c).permute(0, 2, 1)
    y = F.group_norm(xf, groups, weight, bias, eps)
    if silu:
        y = F.silu(y)
    y = y.permute(0, 2, 1).reshape(shape)
    if sft_gamma is not None:
        y = y * (1 + sft_gamma.float()) + sft_beta.float()
        if raw is not None and control_scale != 1.0:
            y = y * control_scale + raw.float() * (1 - control_scale)
    return y.to(bf16).contiguous()


def layer_norm(x, weight, bias, eps=1e-5):
    return F.layer_norm(x.float(), (x.shape[-1],), weight, bias, eps).to(bf16)


def attention(q, k, v, heads, *, q_col=0, k_col=0, v_col=0, scale=None, causal=False):
    b, nq, _ = q.shape
    c = heads * 64
    qf = q.float()[..., q_col:q_col + c].reshape(b, nq, heads, 64).transpose(1, 2)
    kf = k.float()[..., k_col:k_col + c].reshape(b, -1, heads, 64).transpose(1, 2)
    vf = v.float()[..., v_col:v_col + c].reshape(b, -1, heads, 64).transpose(1, 2)
    sc = qf @ kf.transpose(-1, -2) * (scale if scale is not None else 0.125)
    if causal:
        sc = sc + torch.full((nq, sc.shape[-1]), float("-inf")).triu(1)
    att = torch.softmax(sc, dim=-1)
    return (att @ vf).transpose(1, 2).reshape(b, nq, c).to(bf16)


def single_head_attention(q, k, v_t, scale, out_bias=None, valid_keys=None):
    s = q.float() @ k.float().t()
    p = _softmax_rows(s, scale, valid_cols=valid_keys).float()
    o = p @ v_t.float().t()
    if out_bias is not None:
        o = o + out_bias
    return o.to(bf16)


def _softmax_rows(x, scale=1.0, valid_cols=None):
    v = x.shape[-1] if valid_cols is None else valid_cols
    y = torch.zeros_like(x, dtype=torch.float32)
    y[..., :v] = torch.softmax(x.float()[..., :v] * scale, dim=-1)
    return y.to(bf16)


def nchw_to_nhwc_bf16(x, scale=1.0):
    return (x * scale).to(bf16).permute(0, 2, 3, 1).contiguous()


def cast_bf16(x):
    return x.to(bf16).contiguous()


def conv3x3_to_nchw_f32(x, w8, b8, cout):
    return conv3x3(x, w8, b8).float().permute(0, 3, 1, 2)[:, :cout].contiguous()


def upsample2x(x):
    return x.repeat_interleave(2, dim=1).repeat_interleave(2, dim=2).contiguous()


def concat_add(a, b, c=None):
    if c is not None:
        b = (b.float() + c.float()).to(bf16)
    return (torch.cat([a, b], dim=-1) if a is not None else b).contiguous()


def axpy(a, b, alpha=1.0):
    return (a.float() + alpha * b.float()).to(bf16)


def pad_channels(x, cpad):
    y = torch.zeros(*x.shape[:-1], cpad, dtype=bf16)
    y[..., : x.shape[-1]] = x
    return y


def silu(x):
    return F.silu(x.float()).to(bf16)


def pointwise_small(x, w, bias, *, out_nchw_f32=False, scale=1.0):
    y = F.linear(x.float(), w.float(), bias) * scale
    return y.permute(0, 3, 1, 2).contiguous() if out_nchw_f32 else y.to(bf16)


def diag_gaussian(moments, noise, scale=1.0):
    mean, logvar = moments.chunk(2, dim=1)
    if noise is None:
        return mean * scale
    return (mean + torch.exp(0.5 * logvar.clamp(-30.0, 20.0)) * noise) * scale


def embed_tokens(ids, tok, pos):
    return (tok[ids] + pos[None, : ids.shape[1]]).to(bf16)


def sinusoid_embedding(t, dim, max_period=10000.0, sin_first=False):
    t = t.reshape(-1).float()
    half = dim // 2
    freqs = torch.exp(-math.log(max_period) * torch.arange(half, dtype=torch.float32) / half)
    args = t[:, None] * freqs[None]
    parts = [torch.sin(args), torch.cos(args)] if sin_first else [torch.cos(args), torch.sin(args)]
    return torch.cat(parts, dim=-1).to(bf16)


def sampler_pre(x, noise, scalars, cfg_copies=2):
    sigma, sigma_hat, _, sigma_q, _, s_noise = [float(v) for v in scalars]
    x_hat = x if noise is None else x + noise * s_noise * max(sigma_hat**2 - sigma**2, 0.0) ** 0.5
    net = (x_hat / (sigma_q**2 + 1) ** 0.5).to(bf16).permute(0, 2, 3, 1)
    return x_hat, torch.cat([net] * cfg_copies, 0).contiguous()


def sampler_post(eps, x_hat, scalars, use_cfg=True, want_denoised=True):
    _, sigma_hat, sigma_next, sigma_q, cfg, _ = [float(v) for v in scalars]
    if use_cfg:
        eu, ec = eps.chunk(2)
        du, dc = eu * -sigma_q + x_hat, ec * -sigma_q + x_hat
        den = du + cfg * (dc - du)
    else:
        den = eps * -sigma_q + x_hat
    return x_hat + (x_hat - den) / sigma_hat * (sigma_next - sigma_hat), den


def euler_from_denoised(denoised, x_hat, scalars):
    _, sigma_hat, sigma_next = [float(v) for v in scalars[:3]]
    return x_hat + (x_hat - denoised) / sigma_hat * (sigma_next - sigma_hat)


def tile_accumulate(tile, weight, acc, cnt, h0, w0):
    th, tw = tile.shape[-2:]
    acc[:, :, h0:h0 + th, w0:w0 + tw] += tile * weight
    if cnt is not None:
        cnt[:, :, h0:h0 + th, w0:w0 + tw] += weight


def tile_weighted_strip(tile, weight, y0, x0, sh, sw, out=None):
    r = (tile * weight)[:, :, y0:y0 + sh, x0:x0 + sw].contiguous()
    if out is not None:
        out.copy_(r)
        return out
    return r


def strip_add(strip, acc, h0, w0):
    sh, sw = strip.shape[-2:]
    acc[:, :, h0:h0 + sh, w0:w0 + sw] += strip


def copy_batch(pairs):
    for dst, src in pairs:
        dst.view(-1).view(torch.uint8).copy_(src.view(-1).view(torch.uint8))


def tile_normalize(acc, cnt):
    return acc / cnt


def rel_l1_similarity(prev, cur, threshold):
    d = ((prev.float() - cur.float()).abs().mean() / (prev.float().abs().mean() + 1e-6))
    return torch.stack([d, (d < threshold[0]).float()])


def sr3_update(x, eps, noise, scalars):
    cr, crm1, c1, c2, lv = [float(v) for v in scalars]
    x0 = (cr * x - crm1 * eps).clamp(-1, 1)
    out = c1 * x0 + c2 * x
    return out if noise is None else out + noise * math.exp(0.5 * lv)


def wavelet_level(img, radius, high=None, first=False):
    k = torch.tensor([[0.0625, 0.125, 0.0625], [0.125, 0.25, 0.125], [0.0625, 0.125, 0.0625]])[None, None]
    c = img.shape[1]
    low = F.conv2d(F.pad(img, (radius,) * 4, mode="replicate"), k.repeat(c, 1, 1, 1), groups=c, dilation=radius)
    if high is not None:
        if first:
            high.zero_()
        high += img - low
    return low


def add_f32(a, b):
    return a + b


def image_to_u8(x, oh, ow):
    y = F.interpolate(x[None], size=(oh, ow), mode="bicubic")[0]
    return (y.permute(1, 2, 0) * 127.5 + 127.5).clamp(0, 255).to(torch.uint8)


ALL = [n for n, f in list(globals().items()) if callable(f) and not n.startswith("_") and n not in ("F", "torch", "math")]


def install(monkeypatch, ops_module):
    for name in ALL:
        if hasattr(ops_module, name):
            monkeypatch.setattr(ops_module, name, globals()[name])
