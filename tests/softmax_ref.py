"""float64 references, per-element error bounds and designed inputs for the library's softmax paths.

Test infrastructure only (CPU-capable; the GPU tests run the same code on the device in float64).  Every reference is
computed on the values the kernel actually reads: bf16 operands are taken as they are (exactly representable in float64),
fp32 operands likewise, so the only difference between a kernel and its reference is the kernel's own arithmetic.

Error model, shared by every bound below.  Symbols:

* ``U_BF16 = 2^-8``: unit roundoff of bf16 (8 significant bits, round to nearest).  Every bf16 value the kernels write
  (probabilities, P before P.V, attention outputs) is off by at most ``U_BF16`` of itself.
* ``ACC_ULP = 2^-23``: one unit in the last place of an fp32 accumulator, relative to the sum of the magnitudes it has
  absorbed.  A ``tcgen05.mma`` bf16 instruction reduces 16 exact products and adds them to the fp32 accumulator; we charge
  two ulps per instruction (the reduction and the add, without assuming round-to-nearest), so a K-term dot product is off
  by at most ``(K / 16 + 2) * ACC_ULP * sum |a_i b_i|``.
* ``EX2 = 2^-22``: relative error of ``ex2.approx.f32`` (the PTX ISA states 2 ulps across the range); ``__expf`` is that
  instruction applied to ``x * log2(e)``.
* ``FTZ = 2^-126``: ``ex2.approx.ftz`` returns 0 below the smallest normal float, so a probability under ``2^-126`` may
  come out as 0: an absolute floor.
* A logit error of at most ``delta`` (log2 units) on every logit of a row changes each probability by a factor within
  ``2^(+-2 delta)`` (numerator and normaliser move at most ``delta`` each): relative ``2^(2 delta) - 1``.  The fp32
  roundings of a logit's own arithmetic (``x * scale``, ``x - max``, ``* log2 e``; at most three, each ``2^-24`` of a value
  no larger than ``2 max|t|``) are charged as ``2^-21 * max|t|``.
* ``SAFETY = 2``: one factor for all bounds, covering the second-order products the first-order sums above drop.

The bounds are worst cases of that arithmetic, not fits to observed errors: the observed ``err / bound`` of a healthy
kernel is well below 1, and a defect that confines itself to one row or one tile shows as ``err / bound`` far above 1
even where a whole-tensor relative L2 cannot see it.
"""
from __future__ import annotations

import math

import torch

f64 = torch.float64
bf16 = torch.bfloat16

U_BF16 = 2.0 ** -8
U_F32 = 2.0 ** -24
ACC_ULP = 2.0 ** -23
EX2 = 2.0 ** -22
FTZ = 2.0 ** -126
SAFETY = 2.0
LOG2E = 1.0 / math.log(2.0)
SOFTMAX_SEG = 80          # columns per head segment of the per-head softmax epilogue (gemm_conv.cu)
ATT_BLOCK = 128           # keys per block of attention_d64_kernel; also its query tile
RESCALE_LOG2 = 8.0        # attention_d64_kernel rescales O only when a row maximum grew by more than this


def mma_terms(k: int) -> float:
    """Accumulator ulps charged to a K-term tensor-core dot product (two per 16-wide MMA instruction, plus two)."""
    return k / 16.0 + 2.0


def _chunk_rows(n_cols: int, budget: int = 1 << 23) -> int:
    return max(1, budget // max(1, n_cols))


def _softmax2(t: torch.Tensor) -> torch.Tensor:
    """Base-2 softmax over the last dim of float64 log2 logits (-inf = excluded; a row of all -inf gives zeros)."""
    m = t.amax(-1, keepdim=True)
    m = torch.where(torch.isfinite(m), m, torch.zeros_like(m))
    e = torch.exp2(t - m)
    return e / e.sum(-1, keepdim=True).clamp_min(1e-300)


def _prob_bound(p: torch.Tensor, delta: torch.Tensor, n_sum: float) -> torch.Tensor:
    """|p - p64| <= SAFETY * ((U_BF16 + 2 EX2 + n_sum ulps of the normaliser + (2^(2 delta) - 1)) * p64 + FTZ).

    ``delta``: per-row logit error (log2 units), broadcast against p.  ``n_sum``: fp32 roundings (2^-24 each, ex2 rescale
    factors 2^-22 each -- charged as EX2) along the longest chain that forms the row's normaliser."""
    rel = U_BF16 + 2 * EX2 + n_sum * EX2 + torch.expm1(2.0 * delta * math.log(2.0))
    return SAFETY * (rel * p + FTZ)


# ------------------------------------------------------------------------------------------------------------------------
# attention (ops.attention: attention_d64_kernel)
# ------------------------------------------------------------------------------------------------------------------------
def _heads(x: torch.Tensor, col: int, heads: int) -> torch.Tensor:
    b, n, _ = x.shape
    return x[..., col:col + heads * 64].to(f64).reshape(b, n, heads, 64).transpose(1, 2)


def attention(q, k, v, heads: int, scale: float = 0.125, causal: bool = False, cols=(0, 0, 0)):
    """softmax(q k^T * scale) v per head on the bf16 inputs, float64: returns (ref, bound), both [B, Nq, heads * 64].

    Bound per output element o (row r, column d), with S = sum_k p_k |v_k| and p the float64 probabilities:

        |o - o64| <= SAFETY * ((U_BF16 + 2^-20 + eps_acc + (2^(2 delta_r) - 1)) * S + U_BF16 * |o64| + 2^-118 sum_k |v_k|)

    * ``U_BF16 * S``: P is rounded to bf16 before P.V while the sum l takes the unrounded exponentials; scaling P by a
      stale maximum (up to 2^8 above it) does not change a relative rounding.
    * ``U_BF16 * |o64|``: the output is rounded to bf16.
    * ``delta_r = scale log2(e) (64/16 + 2) ACC_ULP max_k sum_d |q_d k_d| + 2^-21 max_k |t_k|``: the fp32 logit of the
      K = 64 tensor-core dot product, times the fp32 ``scale * log2 e``, minus the running maximum (``fmaf``).
    * ``2^-20``: ex2.approx on every exponential, on the rescale factor and on each merge weight (O and l share them, so
      they act as relative errors of the weights).
    * ``eps_acc = (Nk / 16 + 64) ACC_ULP``: O accumulates Nk / 16 MMA instructions in fp32; l is a 64-term per-thread
      chain plus one add per key block and per rescale; the merge adds at most 4 partials.
    * ``2^-118 sum |v|``: exponentials below 2^-126 relative to a maximum that may be 2^8 stale are flushed to zero.
    """
    qh, kh, vh = _heads(q, cols[0], heads), _heads(k, cols[1], heads), _heads(v, cols[2], heads)
    B, H, Nq, _ = qh.shape
    Nk = kh.shape[2]
    c = scale * LOG2E
    eps_acc = (Nk / 16.0 + 64.0) * ACC_ULP
    ref = torch.empty(B, H, Nq, 64, dtype=f64, device=qh.device)
    bound = torch.empty_like(ref)
    rows = _chunk_rows(Nk)
    for b in range(B):
        for h in range(H):
            kk, vv = kh[b, h], vh[b, h]
            vabs = vv.abs()
            floor = 2.0 ** -118 * vabs.sum(0)
            for r0 in range(0, Nq, rows):
                qq = qh[b, h, r0:r0 + rows]
                t = (qq @ kk.T) * c
                mag = (qq.abs() @ kk.abs().T) * c
                if causal:
                    qi = torch.arange(r0, r0 + qq.shape[0], device=t.device)[:, None]
                    masked = torch.arange(Nk, device=t.device)[None, :] > qi
                    t = t.masked_fill(masked, -math.inf)
                    mag = mag.masked_fill(masked, 0.0)
                p = _softmax2(t)
                o = p @ vv
                s = p @ vabs
                tfin = torch.where(torch.isfinite(t), t.abs(), torch.zeros_like(t))
                delta = mma_terms(64) * ACC_ULP * mag.amax(1, keepdim=True) + 2.0 ** -21 * tfin.amax(1, keepdim=True)
                rel = U_BF16 + 2.0 ** -20 + eps_acc + torch.expm1(2.0 * delta * math.log(2.0))
                ref[b, h, r0:r0 + rows] = o
                bound[b, h, r0:r0 + rows] = SAFETY * (rel * s + U_BF16 * o.abs() + floor)
    return (ref.transpose(1, 2).reshape(B, Nq, H * 64), bound.transpose(1, 2).reshape(B, Nq, H * 64))


def attention_logits(q, k, heads: int, b: int, h: int, scale: float = 0.125, cols=(0, 0)) -> torch.Tensor:
    """float64 log2 logits [Nq, Nk] of one (batch, head): what the lazy-rescale emulator looks at."""
    qq = q[b, :, cols[0] + 64 * h:cols[0] + 64 * h + 64].to(f64)
    kk = k[b, :, cols[1] + 64 * h:cols[1] + 64 * h + 64].to(f64)
    return (qq @ kk.T) * (scale * LOG2E)


# ------------------------------------------------------------------------------------------------------------------------
# whole-row softmax: ops.gemm_row_softmax, ops.single_head_attention
# ------------------------------------------------------------------------------------------------------------------------
def gemm_row_softmax(a: torch.Tensor, w: torch.Tensor, scale: float, valid_cols=None):
    """softmax(scale * a @ w^T) over the first ``valid_cols`` columns of each row (others exactly 0): (ref, bound).

    Pass 1 keeps a running (max, sum of ex2) per row and N tile over 32-column chunks (16-term sums, one ex2 rescale
    factor per chunk whose maximum grew), the fold adds one term per tile, pass 2 writes ``ex2(t - M) / L``: the
    normaliser's chain is at most ``N / 32 + 32`` roundings, each charged as EX2.  Logit error: the K-term tensor-core dot
    product times ``alpha = scale log2 e`` plus 2^-21 max|t|."""
    a2 = a.reshape(-1, a.shape[-1]).to(f64)
    w2 = w.to(f64)
    M, K = a2.shape
    N = w2.shape[0]
    valid = N if valid_cols is None else int(valid_cols)
    alpha = scale * LOG2E
    ref = torch.zeros(M, N, dtype=f64, device=a2.device)
    bound = torch.zeros_like(ref)
    n_sum = N / 32.0 + 32.0
    wv = w2[:valid]
    rows = _chunk_rows(valid)
    for r0 in range(0, M, rows):
        aa = a2[r0:r0 + rows]
        t = (aa @ wv.T) * alpha
        mag = (aa.abs() @ wv.abs().T) * alpha
        p = _softmax2(t)
        delta = mma_terms(K) * ACC_ULP * mag.amax(1, keepdim=True) + 2.0 ** -21 * t.abs().amax(1, keepdim=True)
        ref[r0:r0 + rows, :valid] = p
        bound[r0:r0 + rows, :valid] = _prob_bound(p, delta, n_sum)
    return ref, bound


def single_head_attention(q, k, v_t, scale: float, valid_keys=None, out_bias=None):
    """softmax(q k^T * scale) v (+ bias) for one wide head: P from gemm_row_softmax (bf16, bounded by its own bound bp),
    then a bf16 GEMM with fp32 accumulation over Tk keys and a bf16 output:

        |o - o64| <= bp @ |v| + SAFETY * ((Tk / 16 + 2) ACC_ULP * (p + bp) @ |v| + (U_BF16 + U_F32) * |o64|)"""
    p, bp = gemm_row_softmax(q, k, scale, valid_keys)
    v = v_t.to(f64).T
    vabs = v.abs()
    o = p @ v
    if out_bias is not None:
        o = o + out_bias.to(f64)
    tk = v.shape[0]
    bound = bp @ vabs + SAFETY * (mma_terms(tk) * ACC_ULP * ((p + bp) @ vabs) + (U_BF16 + U_F32) * o.abs())
    return o, bound


# ------------------------------------------------------------------------------------------------------------------------
# per-head segment softmax epilogue: ops.gemm(..., softmax_valid=...), optionally with the LayerNorm fold
# ------------------------------------------------------------------------------------------------------------------------
def head_softmax(a: torch.Tensor, w: torch.Tensor, valid: int, *, w_rows_per_group: int = 0, ln=None):
    """Base-2 softmax (no scale) of ``a @ w^T`` over each 80-column head segment, of which the first ``valid`` columns
    take part and the rest are exactly 0: (ref, bound), [M, N].

    ``w_rows_per_group`` > 0: w is [G, N, K] and rows [g * w_rows_per_group, ...) of a use w[g].

    ``ln = (stats [parts, M, 2], colsum [G, N], shift [G, N], eps)``: the LayerNorm fold, stated as the library states it
    (tests/test_ops2_gpu.py): logit = rstd * (a w^T - mean * colsum) + shift with (mean, rstd) from the summed (sum, sum of
    squares) partials the producing GEMM handed over.  Those statistics are an input here, taken as given; the bound
    covers the fold's own fp32 arithmetic: the partial sums (``parts + 2`` ulps of their magnitudes), ``E[x^2] - mean^2``
    (absolute ``(parts + 4) ACC_ULP (E|x^2| + mean^2)``, relative to ``var + eps`` halved by the square root, plus 2 ulps
    of ``rsqrtf``), and four roundings of the affine step.

    Probability bound: per segment, ``delta`` = the largest logit error over its valid columns + 2^-22 of the logit range
    (``v - max`` in fp32); the segment sum is a chain of 80 adds, a division and a product."""
    M, K = a.reshape(-1, a.shape[-1]).shape
    a2 = a.reshape(M, K).to(f64)
    w3 = w.to(f64) if w.dim() == 3 else w.to(f64)[None]
    N = w3.shape[1]
    rpg = w_rows_per_group if w_rows_per_group else M
    heads = N // SOFTMAX_SEG
    ref = torch.zeros(M, N, dtype=f64, device=a2.device)
    bound = torch.zeros_like(ref)
    if ln is not None:
        st, colsum, shift, eps = ln
        buf = st.buf.to(f64)
        parts = buf.shape[0]
        s1, s2 = buf[..., 0].sum(0), buf[..., 1].sum(0)
        s1a, s2a = buf[..., 0].abs().sum(0), buf[..., 1].abs().sum(0)
        mean = s1 / K
        var = (s2 / K - mean * mean).clamp_min(0.0)
        rstd = 1.0 / torch.sqrt(var + eps)
        err_mean = (parts + 2) * ACC_ULP * s1a / K
        err_var = (parts + 4) * ACC_ULP * (s2a / K + mean * mean) + 2.0 * mean.abs() * err_mean
        rel_rstd = 0.5 * err_var / (var + eps) + 2 * ACC_ULP
        colsum = colsum.to(f64).reshape(-1, N)
        shift = shift.to(f64).reshape(-1, N)
    for g0 in range(0, M, rpg):
        g = g0 // rpg if w_rows_per_group else 0
        wg = w3[g]
        rows = _chunk_rows(N)
        for r0 in range(g0, min(M, g0 + rpg), rows):
            r1 = min(M, g0 + rpg, r0 + rows)
            aa = a2[r0:r1]
            acc = aa @ wg.T
            mag = mma_terms(K) * ACC_ULP * (aa.abs() @ wg.abs().T)
            if ln is None:
                t = acc
            else:
                rs, mu = rstd[r0:r1, None], mean[r0:r1, None]
                cen = acc - mu * colsum[g]
                t = rs * cen + shift[g]
                mag = (rs * mag + rel_rstd[r0:r1, None] * (rs * cen).abs() + rs * colsum[g].abs() * err_mean[r0:r1, None]
                       + 4 * ACC_ULP * (rs * acc.abs() + (rs * mu * colsum[g]).abs() + shift[g].abs()))
            t = t.reshape(-1, heads, SOFTMAX_SEG)[..., :valid]
            mag = mag.reshape(-1, heads, SOFTMAX_SEG)[..., :valid]
            p = _softmax2(t)
            rng = t.amax(-1, keepdim=True) - t.amin(-1, keepdim=True)
            delta = mag.amax(-1, keepdim=True) + 2.0 ** -22 * rng
            pb = _prob_bound(p, delta, (SOFTMAX_SEG + 4) * U_F32 / EX2)
            ref[r0:r1].view(-1, heads, SOFTMAX_SEG)[..., :valid] = p
            bound[r0:r1].view(-1, heads, SOFTMAX_SEG)[..., :valid] = pb
    return ref, bound


# ------------------------------------------------------------------------------------------------------------------------
# the checker
# ------------------------------------------------------------------------------------------------------------------------
def assert_within(out: torch.Tensor, ref: torch.Tensor, bound: torch.Tensor, what: str) -> float:
    """Fail on the first element with |out - ref| > bound (a bound of 0 demands equality; NaN always fails).  Reports the
    (row, column) of the last dimension, the values, the error, the bound and the worst err / bound over the tensor.
    Returns that worst ratio."""
    o = out.detach().to(f64).reshape(-1, out.shape[-1])
    r = ref.detach().to(f64).reshape(o.shape)
    bd = bound.detach().to(f64).reshape(o.shape)
    err = (o - r).abs()
    ok = err <= bd
    ratio = torch.where(bd > 0, err / bd, torch.where(err > 0, torch.full_like(err, math.inf), torch.zeros_like(err)))
    ratio = torch.where(torch.isnan(err), torch.full_like(err, math.inf), ratio)
    worst = float(ratio.max()) if ratio.numel() else 0.0
    if not bool(ok.all()):
        flat = int((~ok).reshape(-1).nonzero()[0])
        row, col = divmod(flat, o.shape[1])
        raise AssertionError(
            f"{what}: element (row {row}, col {col}) = {float(o[row, col])!r}, reference {float(r[row, col])!r}, "
            f"|err| {float(err[row, col]):.3e} > bound {float(bd[row, col]):.3e}; "
            f"{int((~ok).sum())} of {ok.numel()} elements over; worst err/bound {worst:.3g}")
    return worst


def rel_l2(a: torch.Tensor, b: torch.Tensor) -> float:
    """The whole-tensor metric the older tests use (kept to show what it cannot see)."""
    a, b = a.to(f64), b.to(f64)
    return float((a - b).norm() / (b.norm() + 1e-300))


# ------------------------------------------------------------------------------------------------------------------------
# attention work plan and the lazy-rescale emulator
# ------------------------------------------------------------------------------------------------------------------------
ATT_WS_COUNTERS = 512
ATT_PART_FLOATS = 66 * 128


def attention_plan(B: int, H: int, Nq: int, Nk: int, num_sms: int = 148) -> dict:
    """Python statement of attention.cu's attention_plan: tiles of the last partial wave of 2 * num_sms are split over
    their key blocks.  ``workspace_bytes`` must equal b200sr_attention_d64_workspace_bytes on a device with num_sms SMs."""
    n_qtiles = -(-Nq // ATT_BLOCK)
    tiles = B * H * n_qtiles
    nblk = -(-Nk // ATT_BLOCK)
    slots = 2 * num_sms
    split, bps, full, tail = 1, nblk, tiles, 0
    full_c = (tiles // slots) * slots
    tail_c = tiles - full_c
    if 0 < tail_c <= ATT_WS_COUNTERS:
        s = 1
        while s * 2 <= nblk and tail_c * s * 2 <= slots and s * 2 <= 4:
            s *= 2
        if s > 1:
            bps = -(-nblk // s)
            split = -(-nblk // bps)
            full, tail = full_c, tail_c
    ws = 0 if tail == 0 else ATT_WS_COUNTERS * 4 + tail * split * ATT_PART_FLOATS * 4
    return dict(n_qtiles=n_qtiles, tiles=tiles, nblk=nblk, full=full, tail=tail, split=split, blocks_per_split=bps,
                workspace_bytes=ws)


def split_tiles(B: int, H: int, Nq: int, plan: dict) -> torch.Tensor:
    """[B, H, Nq] bool: the query rows whose tile is one of the split tail tiles (tile = (b * H + h) * n_qtiles + qtile)."""
    nqt = plan["n_qtiles"]
    tile = (torch.arange(B)[:, None, None] * H + torch.arange(H)[None, :, None]) * nqt + \
        (torch.arange(Nq)[None, None, :] // ATT_BLOCK)
    return tile >= plan["full"]


def block_maxima(t: torch.Tensor) -> torch.Tensor:
    """[rows, Nk] log2 logits (-inf = masked) -> [rows, nblk] maximum of each 128-key block."""
    rows, nk = t.shape
    nblk = -(-nk // ATT_BLOCK)
    pad = torch.full((rows, nblk * ATT_BLOCK - nk), -math.inf, dtype=t.dtype, device=t.device)
    return torch.cat([t, pad], 1).reshape(rows, nblk, ATT_BLOCK).amax(-1)


def emulate_lazy_rescale(bmax: torch.Tensor, blocks_per_split=None):
    """The kernel's rescale decisions from block maxima [rows, nblk] (log2 units): within each key range (the whole row,
    or ranges of ``blocks_per_split`` blocks for a split tile) m_used is set by the range's first block and replaced by
    a later block's maximum when that exceeds m_used + 8 (O and l rescaled then).  Returns per row (number of
    rescales, number of them in a non-first block of a split range)."""
    rows, nblk = bmax.shape
    bps = nblk if blocks_per_split is None else int(blocks_per_split)
    count = torch.zeros(rows, dtype=torch.long, device=bmax.device)
    m_used = torch.full((rows,), -math.inf, dtype=bmax.dtype, device=bmax.device)
    for j in range(nblk):
        mx = bmax[:, j]
        if j % bps == 0:
            m_used = mx.clone()
            continue
        grow = mx > m_used + RESCALE_LOG2
        count += grow.long()
        m_used = torch.where(grow, mx, m_used)
    in_split = count if blocks_per_split is not None else torch.zeros_like(count)
    return count, in_split


def attention_coverage(q, k, heads: int, scale: float = 0.125, cols=(0, 0), num_sms: int = 148) -> dict:
    """Run the emulator over every (batch, head) of an attention input with the plan the kernel uses: rows that rescale,
    rescales inside split ranges, rows within 0.05 of the threshold on either side, rows whose maximum sits in the last
    key block."""
    B, Nq = q.shape[0], q.shape[1]
    Nk = k.shape[1]
    plan = attention_plan(B, heads, Nq, Nk, num_sms)
    in_tail = split_tiles(B, heads, Nq, plan)
    out = dict(rows=0, rows_rescaled=0, rescales=0, rescales_in_split=0, split_rows=0, near_below=0, near_above=0,
               max_in_last_block=0, plan=plan)
    for b in range(B):
        for h in range(heads):
            bm = block_maxima(attention_logits(q, k, heads, b, h, scale, cols))
            tail = in_tail[b, h].to(bm.device)
            for rows_mask, bps in ((~tail, None), (tail, plan["blocks_per_split"])):
                if not bool(rows_mask.any()):
                    continue
                sel = bm[rows_mask]
                cnt, ins = emulate_lazy_rescale(sel, bps if bps is not None and plan["tail"] else None)
                out["rows_rescaled"] += int((cnt > 0).sum())
                out["rescales"] += int(cnt.sum())
                out["rescales_in_split"] += int(ins.sum())
                if bps is not None:
                    out["split_rows"] += int(rows_mask.sum())
            growth = bm[:, 1:] - bm[:, :1]
            out["near_below"] += int(((growth > RESCALE_LOG2 - 0.05) & (growth <= RESCALE_LOG2)).any(1).sum())
            out["near_above"] += int(((growth > RESCALE_LOG2) & (growth < RESCALE_LOG2 + 0.05)).any(1).sum())
            out["max_in_last_block"] += int((bm[:, -1] >= bm.amax(1)).sum()) if bm.shape[1] > 1 else 0
            out["rows"] += bm.shape[0]
    return out


# ------------------------------------------------------------------------------------------------------------------------
# designed inputs (deterministic, seeded; CPU generator so the same values arise on every machine)
# ------------------------------------------------------------------------------------------------------------------------
ROW_KINDS = ("ladder", "threshold", "decreasing", "spike", "random", "uniform")
THRESHOLD_OFFSETS = (-0.05, -0.02, -0.01, 0.01, 0.02, 0.05)
SPIKES = (5.0, 12.0, 40.0)


def _split_bf16(x: torch.Tensor):
    """x (float64) as hi + lo, both bf16: 16 significant bits of x through two bf16 operands."""
    hi = x.to(bf16)
    lo = (x - hi.to(f64)).to(bf16)
    return hi, lo


def attention_offsets(Nq: int, nblk: int, b: int = 0, h: int = 0, seed: int = 0):
    """Per (row, key block) log2 offsets of the growth ladder and the row kind of each row.

    ladder: +g per block, g in [0, 24) across rows (3x the rescale threshold); threshold: +8 +- {0.01 .. 0.05} per block
    (no noise on these rows); decreasing: -g per block (maximum in block 0); spike: 0 everywhere but the last block, which
    is +5 (stale maximum, no rescale), +12 or +40; random: uniform [0, 16) per block; uniform: all logits equal."""
    g = torch.Generator().manual_seed(seed * 7919 + b * 131 + h)
    r = torch.arange(Nq)
    kind = (r + 5 * h + 3 * b) % len(ROW_KINDS)
    j = torch.arange(nblk, dtype=f64)[None, :]
    u = torch.rand(Nq, 1, generator=g, dtype=f64)
    off = torch.zeros(Nq, nblk, dtype=f64)
    ladder = 24.0 * u * j
    thr = (RESCALE_LOG2 + torch.tensor(THRESHOLD_OFFSETS, dtype=f64)[r % len(THRESHOLD_OFFSETS)])[:, None] * j
    dec = -(1.0 + 23.0 * u) * j
    spike = torch.zeros(Nq, nblk, dtype=f64)
    spike[:, -1] = torch.tensor(SPIKES, dtype=f64)[(r // len(ROW_KINDS)) % len(SPIKES)]
    rnd = 16.0 * torch.rand(Nq, nblk, generator=g, dtype=f64)
    for i, val in enumerate((ladder, thr, dec, spike, rnd)):
        off = torch.where((kind == i)[:, None], val.expand(Nq, nblk), off)
    return off, kind


def attention_inputs(B: int, H: int, Nq: int, Nk: int, seed: int = 0, scale: float = 0.125):
    """q [B, Nq, H*64], k, v [B, Nk, H*64] bf16 (CPU) whose log2 logits are ``offset[row, block] + noise``.

    Head dims 2j and 2j + 1 carry block j's code: k = 1 on the keys of block j, q = the row's offset / (scale log2 e) as a
    bf16 hi + lo pair (16 significant bits, so rows sit within 0.05 of the threshold as designed).  The remaining
    64 - 2 nblk dims carry noise with a logit standard deviation of 1 (log2 units); threshold and uniform rows have none,
    uniform rows have q = 0.  Keys beyond Nk do not exist: for Nk = 128 n + 1 the one key of the last block carries that
    block's offset, so spike rows put their maximum on it."""
    nblk = -(-Nk // ATT_BLOCK)
    nd = 64 - 2 * nblk
    assert nd >= 8, "at most 28 key blocks (two code dims per block)"
    c = scale * LOG2E
    g = torch.Generator().manual_seed(seed)
    q = torch.zeros(B, Nq, H, 64, dtype=f64)
    k = torch.zeros(B, Nk, H, 64, dtype=f64)
    kb = torch.arange(Nk) // ATT_BLOCK
    for b in range(B):
        for h in range(H):
            off, kind = attention_offsets(Nq, nblk, b, h, seed)
            hi, lo = _split_bf16(off / c)
            q[b, :, h, 0:2 * nblk:2] = hi.to(f64)
            q[b, :, h, 1:2 * nblk:2] = lo.to(f64)
            noisy = ((kind != ROW_KINDS.index("threshold")) & (kind != ROW_KINDS.index("uniform"))).to(f64)[:, None]
            q[b, :, h, 2 * nblk:] = torch.randn(Nq, nd, generator=g, dtype=f64) / (c * math.sqrt(nd)) * noisy
            q[b, kind == ROW_KINDS.index("uniform"), h, :] = 0.0
            k[b, torch.arange(Nk), h, 2 * kb] = 1.0
            k[b, torch.arange(Nk), h, 2 * kb + 1] = 1.0
            k[b, :, h, 2 * nblk:] = torch.randn(Nk, nd, generator=g, dtype=f64)
    v = torch.randn(B, Nk, H * 64, generator=g, dtype=f64)
    return q.reshape(B, Nq, H * 64).to(bf16), k.reshape(B, Nk, H * 64).to(bf16), v.to(bf16)


def causal_inputs(B: int, H: int, N: int, seed: int = 0, scale: float = 0.125):
    """Causal self-attention inside one key block (N <= 128): logit of key j for row r = g_r * j / 8 (+ noise), g_r in
    [-24, 24) -- a ladder over the keys the row may see, so the maximum of a rising row is its last visible key."""
    c = scale * LOG2E
    g = torch.Generator().manual_seed(seed)
    q = torch.randn(B, N, H, 64, generator=g, dtype=f64) / (c * 8.0)
    k = torch.randn(B, N, H, 64, generator=g, dtype=f64)
    gr = 48.0 * torch.rand(B, N, H, generator=g, dtype=f64) - 24.0
    q[..., 0] = gr / c
    k[..., 0] = (torch.arange(N, dtype=f64) / 8.0)[None, :, None]
    v = torch.randn(B, N, H * 64, generator=g, dtype=f64)
    return q.reshape(B, N, H * 64).to(bf16), k.reshape(B, N, H * 64).to(bf16), v.to(bf16)


def head_softmax_inputs(M: int, K: int, heads: int, log2_range: float, seed: int = 0, groups: int = 1):
    """a [M, K] bf16 and w [groups, heads * 80, K] bf16 whose logits (base 2, no scale) spread over about ``log2_range``
    within a segment: a ~ N(0, 1), w ~ N(0, (log2_range / 5)^2 / K) -- 80 normal samples span about 5 standard deviations.
    Pad rows of w (columns >= valid of a segment) are random too: the epilogue must ignore them, however large."""
    g = torch.Generator().manual_seed(seed)
    a = torch.randn(M, K, generator=g, dtype=f64).to(bf16)
    w = (torch.randn(groups, heads * SOFTMAX_SEG, K, generator=g, dtype=f64) * (log2_range / 5.0 / math.sqrt(K))).to(bf16)
    return a, w


def row_softmax_inputs(M: int, N: int, K: int, tile: int, far: float = 140.0, seed: int = 0, scale: float = 0.125):
    """a [M, K], w [N, K] bf16 for gemm_row_softmax whose N tiles sit at different log2 offsets per row (noise of
    standard deviation 1 on top): row kinds cycle through alternating tiles 0 / -far, a random offset in [-far, 0) per
    tile, one tile at +far above the rest, and no offset.  Two dims per tile carry the code (hi + lo pair as in
    attention_inputs), the rest noise."""
    n_tiles = -(-N // tile)
    nd = K - 2 * n_tiles
    assert nd >= 8
    alpha = scale * LOG2E
    g = torch.Generator().manual_seed(seed)
    r = torch.arange(M)
    kind = r % 4
    ti = torch.arange(n_tiles, dtype=f64)[None, :]
    off = torch.zeros(M, n_tiles, dtype=f64)
    off = torch.where((kind == 0)[:, None], -far * (ti % 2).expand(M, n_tiles), off)
    off = torch.where((kind == 1)[:, None], -far * torch.rand(M, n_tiles, generator=g, dtype=f64), off)
    hot = torch.randint(0, n_tiles, (M,), generator=g)
    off = torch.where((kind == 2)[:, None] & (torch.arange(n_tiles)[None, :] == hot[:, None]), torch.full_like(off, far), off)
    hi, lo = _split_bf16(off / alpha)
    a = torch.zeros(M, K, dtype=f64)
    w = torch.zeros(N, K, dtype=f64)
    a[:, 0:2 * n_tiles:2] = hi.to(f64)
    a[:, 1:2 * n_tiles:2] = lo.to(f64)
    a[:, 2 * n_tiles:] = torch.randn(M, nd, generator=g, dtype=f64) / (alpha * math.sqrt(nd))
    nt = torch.arange(N) // tile
    w[torch.arange(N), 2 * nt] = 1.0
    w[torch.arange(N), 2 * nt + 1] = 1.0
    w[:, 2 * n_tiles:] = torch.randn(N, nd, generator=g, dtype=f64)
    return a.to(bf16), w.to(bf16)
