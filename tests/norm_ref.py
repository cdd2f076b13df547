"""float64 references, per-element error bounds, launch geometry and designed inputs for the library's normalisations.

Test infrastructure only (CPU-capable; the GPU tests run the same code on the device in float64).  Every reference is
computed on the values the kernel reads: bf16 activations are exact in float64, and the fp32 weight, bias, SFT, colsum,
shift and row-statistics operands are used as they are.  The error model and its constants are softmax_ref's
(``U_BF16``, ``U_F32``, ``ACC_ULP``, ``EX2``, ``FTZ``, ``SAFETY``); what is particular to the normalisations:

* A sum of n fp32 terms, in any order, is off by at most ``(n - 1) ACC_ULP * sum |terms|`` (one ulp of a partial sum no
  larger than the sum of magnitudes per add).  ``n`` is the longest chain of adds that builds the value: for GroupNorm the
  ``ceil(ppc / P)`` pixels a thread walks, then the ``P * cpg`` per-thread sums the CTA folds per group (the fold across
  chunks is fp64 and charged one ulp); bf16 x bf16 products are exact in fp32, so x^2 costs nothing.
* Sums are exact when they can be: if every term is a multiple of q (the lowest set bit of the group's values) and the
  sum of magnitudes that one fp32 accumulation absorbs stays below ``2^24 q``, every partial sum is representable.  For
  LayerNorm that is the whole row; for GroupNorm it is one chunk (the fold across chunks is fp64: ``2^53 q``).  Constant
  groups and rows use this.
* The variance from sums, ``E[x^2] - mean^2``, carries the absolute error ``dvar`` of both sums (the cancellation grows
  with ``(mean / std)^2``); relative to ``var + eps`` it is ``t = dvar / (var + eps)``, and ``rstd`` is then off by at most
  ``rho(t) = 1 / sqrt(1 - t) - 1`` (>= t / 2, and >= the change for a var that moved up by t instead), plus the fp32
  roundings of the cast, ``+ eps``, the square root and the reciprocal (or ``rsqrtf``, 2 ulps).
* The affine step ``x * sc + sh`` with ``sc = rstd * w``, ``sh = b - mean * sc`` costs three fp32 roundings of values no
  larger than ``rstd |w| (|x| + |mean|) + |b|``; the mean's own error enters multiplied by ``rstd |w|``.
* ``silu_f`` = ``x * rcp.approx(1 + ex2.approx(-x log2 e))``: relative ``EX2 + 2^-22 + 2 U_F32 + U_F32 |x|`` (the last
  from the rounded exponent argument), its slope is at most 1.1, and results below 2^-126 flush to zero (absolute
  ``FTZ (1 + |x|)``).
* The bf16 output rounding: ``U_BF16 |y|``.

The bounds are worst cases of that arithmetic, not fits to observed errors: the observed ``err / bound`` of a healthy
kernel is well below 1, and a defect confined to one (image, group) or one row shows as ``err / bound`` far above 1 even
where a whole-tensor relative L2 cannot see it.
"""
from __future__ import annotations

import math

import torch

from softmax_ref import ACC_ULP, EX2, FTZ, SAFETY, U_BF16, U_F32, assert_within, mma_terms, rel_l2  # noqa: F401

f64 = torch.float64
bf16 = torch.bfloat16

GN_WS_COUNTER_FLOATS = 256     # norm.cu: arrival (and, one-kernel path, departure) counters at the start of the workspace
GELU_ERF = 3e-7                # |erf error| of gelu_erf_f's polynomial (common.cuh)


# ------------------------------------------------------------------------------------------------------------------------
# launch geometry (ports of norm.cu)
# ------------------------------------------------------------------------------------------------------------------------
def gn_geometry(N: int, HW: int, C: int, groups: int = 32, num_sms: int = 148) -> dict:
    """norm.cu's gn_geometry + gn_fused_eligible: thread rows P, threads, pixels per chunk, chunks, the path
    (``launches`` 1 = gn_fused_kernel, 2 = gn_stats_kernel + gn_apply_kernel; equals b200sr_group_norm_launches), the
    pixels of the last chunk, and which fold the statistics kernel's last CTA runs ("rows" or "warp")."""
    C8 = C // 8
    P = max(1, 256 // C8)
    threads = (C8 * P + 31) // 32 * 32
    ctas_per_sm = 2 if N * HW * C * 2 >= (16 << 20) else 1
    want = max(1, (ctas_per_sm * num_sms + N - 1) // N)
    ppc = min(max(-(-HW // want), P * 8), HW)
    chunks = -(-HW // ppc)
    smem = ppc * C * 2 + 2 * P * C * 4 + 2 * groups * 4
    fold_fits = groups <= threads and 2 * threads * 8 <= 2 * P * C * 4
    fused = chunks * N <= num_sms and N <= 128 and smem <= 100 * 1024 and fold_fits
    return dict(P=P, threads=threads, active=C8 * P, ppc=ppc, chunks=chunks, last_chunk=HW - (chunks - 1) * ppc,
                smem=smem, launches=1 if fused else 2,
                stats_fold="rows" if threads % groups == 0 and 2 * threads * 8 <= 2 * P * C * 4 else "warp")


def ln_template(C: int) -> int:
    """layer_norm_kernel<VEC_PER_LANE> that norm.cu's layer_norm launches for C channels."""
    vpl = (C // 8 + 31) // 32
    return next(t for t in (1, 3, 5, 10, 20) if vpl <= t)


# ------------------------------------------------------------------------------------------------------------------------
# shared pieces of the error model
# ------------------------------------------------------------------------------------------------------------------------
def _rho(t: torch.Tensor) -> torch.Tensor:
    """Relative error bound of 1 / sqrt(v) when v is off by at most t * v."""
    return torch.where(t < 1, 1.0 / torch.sqrt((1.0 - t).clamp_min(1e-300)) - 1.0, torch.full_like(t, math.inf))


def _lowbit(x: torch.Tensor) -> torch.Tensor:
    """Value of the lowest set bit of each bf16-valued float64 element (inf for 0)."""
    m, e = torch.frexp(x)
    im = (m.abs() * 256).to(torch.int64)
    q = (im & -im).to(f64) * torch.exp2((e - 8).to(f64))
    return torch.where(x == 0, torch.full_like(x, math.inf), q)


def _sums_exact(x: torch.Tensor, dims) -> torch.Tensor:
    """True where fp32 sums of x and of x^2 over ``dims`` are exact in every order (see the module docstring)."""
    q = _lowbit(x).amin(dims)
    return (x.abs().sum(dims) < 2.0 ** 24 * q) & ((x * x).sum(dims) < 2.0 ** 24 * q * q)


def _gn_sums_exact(xg: torch.Tensor, ppc: int) -> torch.Tensor:
    """[N, groups]: True where GroupNorm's sums of x and x^2 are exact: xg [N, HW, groups, cpg] is summed in fp32 within
    each chunk of ``ppc`` pixels (per thread, then per CTA) and the chunk partials in fp64."""
    N, HW, G, _ = xg.shape
    q = _lowbit(xg).amin((1, 3))
    chunk = torch.arange(HW, device=xg.device) // ppc
    n_chunks = int(chunk[-1]) + 1
    per_chunk = lambda t: torch.zeros(N, n_chunks, G, dtype=f64, device=xg.device).index_add_(1, chunk, t.sum(3))  # noqa: E731
    ca, cq = per_chunk(xg.abs()), per_chunk(xg * xg)
    return ((ca.amax(1) < 2.0 ** 24 * q) & (cq.amax(1) < 2.0 ** 24 * q * q)
            & (ca.sum(1) < 2.0 ** 53 * q) & (cq.sum(1) < 2.0 ** 53 * q * q))


def _silu(v: torch.Tensor) -> torch.Tensor:
    return v * torch.sigmoid(v)


def _silu_err(v: torch.Tensor, e_v: torch.Tensor) -> torch.Tensor:
    """Error of silu_f(v_computed) against silu(v) when v_computed is off by at most e_v."""
    z = _silu(v)
    return 1.1 * e_v + (EX2 + 2.0 ** -22 + 2 * U_F32 + U_F32 * v.abs()) * z.abs() + FTZ * (1.0 + v.abs())


# ------------------------------------------------------------------------------------------------------------------------
# GroupNorm: statistics, the whole op, the fused-input convolution
# ------------------------------------------------------------------------------------------------------------------------
def gn_stats(x: torch.Tensor, groups: int, eps: float, num_sms: int = 148) -> dict:
    """float64 (mean, rstd) per (image, group) of channels-last x [N, ..., C] and the kernel's error on them.

    Returned fields, all [N, groups]: ``mean``, ``rstd``, ``err_mean`` (absolute error of the fp32 mean the kernel
    uses), ``rel_rstd`` (relative error of its fp32 rstd).  Chain length ``n = ceil(ppc / P) + P cpg + 1``:
    ``err_s = n ACC_ULP sum|x|`` and ``n ACC_ULP sum x^2`` (0 where the sums are exact, ``_gn_sums_exact``);
    ``err_mean = err_s1 / cnt + U_F32 |mean|`` (the fp32 cast);
    ``dvar = err_s2 / cnt + 2 |mean| err_s1 / cnt + (err_s1 / cnt)^2 + 2^-50 (E[x^2] + mean^2)`` (the fp64 arithmetic);
    ``rel_rstd = rho(dvar / (var + eps)) + 4 U_F32`` (cast, + eps, sqrtf, division)."""
    N, C = x.shape[0], x.shape[-1]
    HW = x.numel() // (N * C)
    cpg = C // groups
    geo = gn_geometry(N, HW, C, groups, num_sms)
    xg = x.reshape(N, HW, groups, cpg).to(f64)
    cnt = HW * cpg
    s1, s1a, s2 = xg.sum((1, 3)), xg.abs().sum((1, 3)), (xg * xg).sum((1, 3))
    mean = s1 / cnt
    var = ((xg - mean[:, None, :, None]) ** 2).sum((1, 3)) / cnt
    rstd = 1.0 / torch.sqrt(var + eps)
    n_acc = -(-geo["ppc"] // geo["P"]) + geo["P"] * cpg + 1
    exact = _gn_sums_exact(xg, geo["ppc"])
    e1 = torch.where(exact, torch.zeros_like(s1), n_acc * ACC_ULP * s1a) / cnt
    e2 = torch.where(exact, torch.zeros_like(s2), n_acc * ACC_ULP * s2) / cnt
    dvar = e2 + 2 * mean.abs() * e1 + e1 * e1 + 2.0 ** -50 * (s2 / cnt + mean * mean)
    return dict(mean=mean, rstd=rstd, var=var, err_mean=e1 + U_F32 * mean.abs(),
                rel_rstd=_rho(dvar / (var + eps)) + 4 * U_F32, geo=geo)


def _gn_pre(x, weight, bias, groups, st):
    """Per element: the float64 normalised + affine value v and the bound e_v of the kernel's fp32 value before any
    activation, both [N, HW, C]."""
    N, C = x.shape[0], x.shape[-1]
    cpg = C // groups
    x64 = x.reshape(N, -1, C).to(f64)
    ch = lambda t: t.repeat_interleave(cpg, dim=1)[:, None, :]   # noqa: E731  [N, G] -> [N, 1, C]
    w = weight.to(f64) if weight is not None else torch.ones(C, dtype=f64, device=x.device)
    b = bias.to(f64) if bias is not None else torch.zeros(C, dtype=f64, device=x.device)
    mean, rstd = ch(st["mean"]), ch(st["rstd"])
    xm = x64 - mean
    A = rstd * w.abs()
    v = xm * rstd * w + b
    e_v = A * (xm.abs() * ch(st["rel_rstd"]) + ch(st["err_mean"])) + 3 * U_F32 * (A * (x64.abs() + mean.abs()) + b.abs())
    return v, e_v


def group_norm(x, weight, bias, *, groups=32, eps=1e-5, silu=False, sft_gamma=None, sft_beta=None, raw=None,
               control_scale=1.0, num_sms=148):
    """ops.group_norm in float64: (ref, bound), shaped like x.  Bound: e_v from the statistics and the affine step
    (see gn_stats / the module docstring), through silu_f (``_silu_err``), through the SFT ``z (1 + gamma) + beta``
    (``e |1 + gamma| + 3 U_F32 (|z (1 + gamma)| + |beta|)``) and the lerp ``m cs + raw (1 - cs)`` with the fp32 value of
    cs (``e |cs| + 3 U_F32 (|m cs| + |raw (1 - cs)|)``); then ``SAFETY (e + U_BF16 |ref|)``."""
    st = gn_stats(x, groups, eps, num_sms)
    y, e = _gn_pre(x, weight, bias, groups, st)
    if silu:
        e = _silu_err(y, e)
        y = _silu(y)
    if sft_gamma is not None:
        g1 = 1.0 + sft_gamma.reshape(y.shape).to(f64)
        be = sft_beta.reshape(y.shape).to(f64)
        e = e * g1.abs() + 3 * U_F32 * ((y * g1).abs() + be.abs())
        y = y * g1 + be
        cs = float(torch.tensor(control_scale, dtype=torch.float32))
        if raw is not None and cs != 1.0:
            r = raw.reshape(y.shape).to(f64)
            e = e * abs(cs) + 3 * U_F32 * ((y * cs).abs() + (r * (1.0 - cs)).abs())
            y = y * cs + r * (1.0 - cs)
    return y.reshape(x.shape), (SAFETY * (e + U_BF16 * y.abs())).reshape(x.shape)


def gn_stats_bounds(x, groups, eps, num_sms=148):
    """group_norm_stats in float64: (ref [N, groups, 2] of (mean, rstd), bound [N, groups, 2])."""
    st = gn_stats(x, groups, eps, num_sms)
    ref = torch.stack([st["mean"], st["rstd"]], -1)
    bound = torch.stack([SAFETY * st["err_mean"], SAFETY * st["rstd"] * st["rel_rstd"]], -1)
    return ref, bound


def conv3x3_fused_gn(x, w, b, gn_weight, gn_bias, *, groups=32, eps=1e-5, silu=True, num_sms=148):
    """conv3x3(x, w, b, gn=(group_norm_stats(x), ...)) in float64: the input normalised (+SiLU) in float64, rounded to
    bf16 as the kernel does, padded with ZEROS (a padding pixel is not normalised), convolved in float64.

    x [N, H, W, Cin] bf16, w [Cout, Cin, 3, 3] (its bf16 values are what the kernel multiplies).  Bound per output:
    ``SAFETY ((e_y + U_BF16 |y|) * |w| + (9 Cin / 16 + 2) ACC_ULP |y| * |w| + U_BF16 |out|)`` with ``*`` the convolution
    and e_y the bound of the normalised input before its rounding (a rounding may flip by one bf16 ulp)."""
    import torch.nn.functional as F

    n, h, wd, cin = x.shape
    st = gn_stats(x, groups, eps, num_sms)
    y, e = _gn_pre(x, gn_weight, gn_bias, groups, st)
    if silu:
        e = _silu_err(y, e)
        y = _silu(y)
    yr = y.to(bf16).to(f64)
    to_nchw = lambda t: t.reshape(n, h, wd, cin).permute(0, 3, 1, 2)   # noqa: E731
    w64 = w.to(bf16).to(f64)
    out = F.conv2d(to_nchw(yr), w64, None if b is None else b.to(f64), padding=1)
    mag = F.conv2d(to_nchw(y.abs()), w64.abs(), padding=1)
    err = F.conv2d(to_nchw(e + U_BF16 * y.abs()), w64.abs(), padding=1)
    bound = SAFETY * (err + mma_terms(9 * cin) * ACC_ULP * mag + U_BF16 * out.abs())
    return out.permute(0, 2, 3, 1), bound.permute(0, 2, 3, 1)


# ------------------------------------------------------------------------------------------------------------------------
# LayerNorm: the kernel and the fold around the GEMMs
# ------------------------------------------------------------------------------------------------------------------------
def layer_norm(x, weight, bias, eps=1e-5):
    """ops.layer_norm in float64: (ref, bound) [M, C].

    layer_norm_kernel: per lane ``8 ceil(C / 256)`` fp32 adds, a 5-level warp tree, ``/ C``: chain ``L = 8 ceil(C / 256)
    + 6``, ``err_mean = L ACC_ULP sum|x| / C + U_F32 |mean|`` (0 + U_F32 |mean| where exact).  Two-pass variance from
    ``d = x - mean_f``: ``sum d^2 = C var + C err_mean^2``; each ``d^2`` is off by 3 U_F32 and the sum by L ulps, so
    ``dvar = (L + 3) ACC_ULP var + err_mean^2 + 2 U_F32 (var + eps)``; ``rel_rstd = rho(dvar / (var + eps)) + 2 ACC_ULP``
    (rsqrtf).  Output ``(x - mean) rstd w + b``: ``rstd |w| (|x - mean| rel_rstd + err_mean) + 4 U_F32 (rstd |w|
    |x - mean| + |b|)``, then the bf16 rounding."""
    C = x.shape[-1]
    x64 = x.reshape(-1, C).to(f64)
    w, b = weight.to(f64), bias.to(f64)
    mean = x64.mean(1, keepdim=True)
    xm = x64 - mean
    var = (xm * xm).mean(1, keepdim=True)
    rstd = 1.0 / torch.sqrt(var + eps)
    L = 8 * -(-C // 256) + 6
    exact = _sums_exact(x64, (1,))[:, None]
    err_mean = torch.where(exact, torch.zeros_like(mean), L * ACC_ULP * x64.abs().mean(1, keepdim=True)) \
        + U_F32 * mean.abs()
    dvar = (L + 3) * ACC_ULP * var + err_mean ** 2 + 2 * U_F32 * (var + eps)
    rel = _rho(dvar / (var + eps)) + 2 * ACC_ULP
    A = rstd * w.abs()
    y = xm * rstd * w + b
    e = A * (xm.abs() * rel + err_mean) + 4 * U_F32 * (A * xm.abs() + b.abs())
    return y.reshape(x.shape), (SAFETY * (e + U_BF16 * y.abs())).reshape(x.shape)


def _fold_stats(buf: torch.Tensor, K: int, eps: float):
    """(mean, rstd, err_mean, rel_rstd) [M] of the consumer's fp32 fold of ``parts`` (sum, sum of squares) partials:
    chains of ``parts`` adds, ``* (1 / K)`` with 1 / K rounded to fp32, ``s2 / K - mean^2`` (3 roundings), ``+ eps``,
    rsqrtf (2 ulps).  The partials are an input: the reference takes their float64 sum as the truth."""
    b = buf.to(f64)
    parts = b.shape[0]
    s1, s2 = b[..., 0].sum(0), b[..., 1].sum(0)
    s1a, s2a = b[..., 0].abs().sum(0), b[..., 1].abs().sum(0)
    mean = s1 / K
    var = (s2 / K - mean * mean).clamp_min(0.0)
    rstd = 1.0 / torch.sqrt(var + eps)
    err_mean = (parts + 2) * ACC_ULP * s1a / K
    err_var = (parts + 4) * ACC_ULP * (s2a / K + mean * mean) + 2.0 * mean.abs() * err_mean + err_mean ** 2
    rel_rstd = _rho(err_var / (var + eps)) + 2 * ACC_ULP + U_F32
    return mean, rstd, err_mean, rel_rstd


def _gelu(g):
    return 0.5 * g * (1.0 + torch.erf(g / math.sqrt(2.0)))


def ln_fold(a, w, buf, colsum, shift, eps=1e-5, *, geglu=False, w_rows_per_group=0, residual=None, alpha=1.0):
    """gemm(a, w, ln=(RowStats(buf), colsum, shift, eps), ...) in float64: (ref, bound), [M, N] (plain) or [M, N / 2]
    (GEGLU, rows of w interleaved as ops.geglu_interleave_index packs them).

    v = rstd (a w^T - mean colsum) + shift, with (mean, rstd) from the float64 sum of the partials (``_fold_stats``).
    Bound of v: ``rstd (K / 16 + 2) ACC_ULP |a| |w|^T`` (the MMA) + ``rel_rstd |rstd (acc - mean colsum)|`` +
    ``rstd |colsum| err_mean`` + ``4 U_F32 (rstd |acc| + rstd |mean colsum| + |shift|)`` (nm = -mean rstd, the two
    ``fma.rn.f32x2`` of ln_apply2).  Plain: ``alpha v + residual`` (2 roundings); GEGLU: ``val * gelu_erf_f(gate)`` with
    gelu's slope <= 1.13 and its own error ``0.5 |gate| (3e-7 + 128 U_F32)`` (polynomial; six fma, four squarings and
    the approximate reciprocal of p^-16) + 2 U_F32 of the result.  Then ``SAFETY (e + U_BF16 |ref|)``."""
    M, K = a.reshape(-1, a.shape[-1]).shape
    a2 = a.reshape(M, K).to(f64)
    w3 = w.to(f64) if w.dim() == 3 else w.to(f64)[None]
    N = w3.shape[1]
    colsum = colsum.to(f64).reshape(-1, N)
    shift = shift.to(f64).reshape(-1, N)
    mean, rstd, err_mean, rel_rstd = _fold_stats(buf, K, eps)
    rpg = w_rows_per_group if w_rows_per_group else M
    v = torch.empty(M, N, dtype=f64, device=a2.device)
    e = torch.empty_like(v)
    for g0 in range(0, M, rpg):
        g = g0 // rpg if w_rows_per_group else 0
        r = slice(g0, min(M, g0 + rpg))
        aa, wg = a2[r], w3[g]
        acc = aa @ wg.T
        mag = mma_terms(K) * ACC_ULP * (aa.abs() @ wg.abs().T)
        rs, mu = rstd[r, None], mean[r, None]
        cen = acc - mu * colsum[g]
        v[r] = rs * cen + shift[g]
        e[r] = (rs * mag + rel_rstd[r, None] * (rs * cen).abs() + rs * colsum[g].abs() * err_mean[r, None]
                + 4 * U_F32 * (rs * acc.abs() + (rs * mu * colsum[g]).abs() + shift[g].abs()))
    if geglu:
        vv, ee = v.view(M, N // 32, 2, 16), e.view(M, N // 32, 2, 16)
        val, gate, e_val, e_gate = vv[:, :, 0], vv[:, :, 1], ee[:, :, 0], ee[:, :, 1]
        gl = _gelu(gate)
        y = (val * gl).reshape(M, N // 2)
        e = (gl.abs() * e_val + val.abs() * (1.13 * e_gate + 0.5 * gate.abs() * (GELU_ERF + 128 * U_F32))
             + 2 * U_F32 * (val * gl).abs()).reshape(M, N // 2)
    else:
        y = alpha * v
        e = abs(alpha) * e
        if residual is not None:
            r64 = residual.reshape(M, N).to(f64)
            e = e + 2 * U_F32 * (y.abs() + r64.abs())
            y = y + r64
    return y, SAFETY * (e + U_BF16 * y.abs())


def ln_partials(y: torch.Tensor, bn: int):
    """The producer's per-row, per-N-tile (sum, sum of squares) against the bf16 output y [M, N] it stored: (ref, bound),
    [parts, M, 2].  The kernel sums the fp32 values before their rounding to bf16 (|v - y| <= U_BF16 |y|, so
    |v^2 - y^2| <= 2 U_BF16 y^2), two interleaved chains of ``bn / 2`` columns per lane (``stats_acc2``) and one add:
    ``SAFETY ((U_BF16 + (bn / 2 + 2) ACC_ULP) sum|y|, (2 U_BF16 + (bn / 2 + 2) ACC_ULP) sum y^2)``."""
    M, N = y.shape
    parts = -(-N // bn)
    y64 = torch.zeros(M, parts * bn, dtype=f64, device=y.device)
    y64[:, :N] = y.to(f64)
    t = y64.view(M, parts, bn)
    ref = torch.stack([t.sum(-1), (t * t).sum(-1)], -1).transpose(0, 1)
    chain = (bn / 2 + 2) * ACC_ULP
    bound = torch.stack([(U_BF16 + chain) * t.abs().sum(-1), (2 * U_BF16 + chain) * (t * t).sum(-1)], -1).transpose(0, 1)
    return ref.contiguous(), SAFETY * bound.contiguous()


def exact_partials(x: torch.Tensor, parts: int) -> torch.Tensor:
    """[parts, M, 2] fp32 (sum, sum of squares) of x [M, K] over ``parts`` column ranges, summed in float64 and rounded
    once: statistics a consumer can be fed independently of any producer."""
    M, K = x.shape
    x64 = x.to(f64)
    edges = [K * i // parts for i in range(parts + 1)]
    out = torch.empty(parts, M, 2, dtype=f64, device=x.device)
    for i in range(parts):
        s = x64[:, edges[i]:edges[i + 1]]
        out[i, :, 0], out[i, :, 1] = s.sum(1), (s * s).sum(1)
    return out.float()


# ------------------------------------------------------------------------------------------------------------------------
# designed inputs (deterministic, seeded; CPU generator so the same values arise on every machine)
# ------------------------------------------------------------------------------------------------------------------------
REGIMES = ("r0", "r1", "r8", "r32", "r64", "tiny", "const", "big", "outlier")
CONSTS = (-3.0, 0.75, 5.0, -1.5, 2.0)
OUTLIER = 60.0


def gn_regimes(N: int, groups: int) -> torch.Tensor:
    """[N, groups] regime index: neighbouring groups and the same group of neighbouring images differ."""
    n, g = torch.arange(N)[:, None], torch.arange(groups)[None, :]
    return (g + 4 * n) % len(REGIMES)


def _regime_moments(kind: torch.Tensor, eps: float, gen: torch.Generator):
    """(mean, std) per entry of ``kind``: offset ratios r in {0, 1, 8, 32, 64} at a random std in [0.5, 2) and sign;
    ``tiny``: std in [0.7, 1.4) sqrt(eps), mean 0; ``const``: std 0; ``big``: mean +-1e4, std 1e3; ``outlier``: mean 0.5,
    std 1 (plus one planted pixel)."""
    shape = kind.shape
    std = 2.0 ** (2 * torch.rand(shape, generator=gen, dtype=f64) - 1)
    sign = torch.where(torch.rand(shape, generator=gen) < 0.5, -1.0, 1.0).to(f64)
    ratio = torch.tensor([0.0, 1.0, 8.0, 32.0, 64.0, 0.0, 0.0, 0.0, 0.0], dtype=f64)[kind]
    mean = sign * ratio * std
    tiny = kind == REGIMES.index("tiny")
    std = torch.where(tiny, math.sqrt(eps) * (0.7 + 0.7 * torch.rand(shape, generator=gen, dtype=f64)), std)
    const = kind == REGIMES.index("const")
    cval = torch.tensor(CONSTS, dtype=f64)[torch.arange(kind.numel()).reshape(shape) % len(CONSTS)]
    mean = torch.where(const, cval, mean)
    std = torch.where(const, torch.zeros_like(std), std)
    big = kind == REGIMES.index("big")
    mean, std = torch.where(big, sign * 1e4, mean), torch.where(big, torch.full_like(std, 1e3), std)
    out = kind == REGIMES.index("outlier")
    mean, std = torch.where(out, torch.full_like(mean, 0.5), mean), torch.where(out, torch.ones_like(std), std)
    return mean, std


def gn_inputs(N: int, HW: int, C: int, groups: int = 32, eps: float = 1e-5, seed: int = 0) -> torch.Tensor:
    """x [N, HW, C] bf16 (CPU) with a different regime per (image, group) (``gn_regimes``); ``outlier`` groups carry
    OUTLIER at their first channel of the image's LAST pixel, which lies in the last (possibly ragged) chunk."""
    cpg = C // groups
    g = torch.Generator().manual_seed(seed)
    kind = gn_regimes(N, groups)
    mean, std = _regime_moments(kind, eps, g)
    z = torch.randn(N, HW, groups, cpg, generator=g, dtype=f64)
    x = mean[:, None, :, None] + std[:, None, :, None] * z
    n_i, g_i = (kind == REGIMES.index("outlier")).nonzero(as_tuple=True)
    x[n_i, HW - 1, g_i, 0] = OUTLIER
    return x.reshape(N, HW, C).to(bf16)


def gn_params(C: int, seed: int = 0, sft_shape=None):
    """(weight, bias) fp32 [C]; with ``sft_shape``, also (gamma, beta, raw) bf16 of that shape."""
    g = torch.Generator().manual_seed(seed + 1)
    w = 1.0 + 0.25 * torch.randn(C, generator=g)
    b = 0.5 * torch.randn(C, generator=g)
    if sft_shape is None:
        return w, b
    gam, bet, raw = (0.5 * torch.randn(*sft_shape, generator=g)).to(bf16), (0.5 * torch.randn(*sft_shape, generator=g)).to(bf16), \
        torch.randn(*sft_shape, generator=g).to(bf16)
    return w, b, gam, bet, raw


def ln_rows(M: int, C: int, eps: float = 1e-5, seed: int = 0) -> torch.Tensor:
    """x [M, C] bf16 (CPU), row m in regime REGIMES[m % 9] (an ``outlier`` row has OUTLIER in its last column)."""
    g = torch.Generator().manual_seed(seed)
    kind = torch.arange(M) % len(REGIMES)
    mean, std = _regime_moments(kind, eps, g)
    x = mean[:, None] + std[:, None] * torch.randn(M, C, generator=g, dtype=f64)
    x[kind == REGIMES.index("outlier"), C - 1] = OUTLIER
    return x.to(bf16)


FOLD_OFFSETS = (0.0, 1.0, 8.0, 32.0, 64.0)


def fold_producer_inputs(M: int, K: int, seed: int = 0):
    """(a [M, K], w0 [K, K], residual [M, K]) bf16 (CPU) for a producing GEMM ``a w0^T + residual`` whose output row m
    has a mean of +-FOLD_OFFSETS[m % 5] (std about 1)."""
    g = torch.Generator().manual_seed(seed)
    a = torch.randn(M, K, generator=g, dtype=f64).to(bf16)
    w0 = (torch.randn(K, K, generator=g, dtype=f64) * (0.5 / math.sqrt(K))).to(bf16)
    off = torch.tensor(FOLD_OFFSETS, dtype=f64)[torch.arange(M) % len(FOLD_OFFSETS)]
    off = off * torch.where(torch.rand(M, generator=g) < 0.5, -1.0, 1.0).to(f64)
    res = (off[:, None] + 0.8 * torch.randn(M, K, generator=g, dtype=f64)).to(bf16)
    return a, w0, res


def fold_weights(N: int, K: int, groups: int = 1, seed: int = 0, geglu: bool = False):
    """(w' = W gamma bf16 [groups, N, K] (or [N, K]), colsum fp32 [groups, N], shift fp32 [groups, N]) as
    ops.pack_linear_ln packs them (GEGLU: rows interleaved as ops.pack_geglu_ln does)."""
    g = torch.Generator().manual_seed(seed + 7)
    W = torch.randn(groups, N, K, generator=g) * K ** -0.5
    gamma = 1 + 0.3 * torch.randn(K, generator=g)
    beta = 0.2 * torch.randn(K, generator=g)
    bias = 0.1 * torch.randn(N, generator=g)
    if geglu:
        j = torch.arange(N // 2)
        val_pos = (j // 16) * 32 + (j % 16)
        idx = torch.empty(N, dtype=torch.long)
        idx[val_pos], idx[val_pos + 16] = j, j + N // 2
        W, bias = W[:, idx], bias[idx]
    wp = (W * gamma).to(bf16)
    colsum = wp.float().sum(-1)
    shift = W @ beta + bias
    if groups == 1:
        return wp[0].contiguous(), colsum.contiguous(), shift.contiguous()
    return wp.contiguous(), colsum.contiguous(), shift.contiguous()
