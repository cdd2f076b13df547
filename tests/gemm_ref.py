"""float64 references, per-element error bounds, launch geometry and designed inputs for the GEMM and the 3x3 convolution
(gemm_conv.cu: the plain, general, GEGLU and fp32 epilogue families; the three convolution modes).

Test infrastructure only (CPU-capable; the GPU tests run the same code on the device in float64).  Every reference is
computed on the values the kernel reads: bf16 operands as they are (exact in float64), the fp32 bias, rowvec and alpha
as they are.  The error model and its constants are softmax_ref's (``U_BF16``, ``U_F32``, ``ACC_ULP``, ``EX2``, ``FTZ``,
``mma_terms``, ``SAFETY``) and norm_ref's (``GELU_ERF``, the activation slopes); what is particular to this kernel:

* The accumulator.  One ``tcgen05.mma`` reduces 16 exact bf16 products and adds them to the fp32 accumulator in TMEM;
  the K loop runs over 64-wide chunks, the last one zero-filled by the TMA, so a GEMM issues ``K_pad / 16`` MMAs with
  ``K_pad = ceil(K / 64) 64``, a convolution ``9 Cin / 16`` (Cin is a multiple of 64).  The accumulator is off by at
  most ``mma_terms(K_pad) ACC_ULP (|A| |W|^T)``; the magnitude product is the same float64 contraction on absolute
  values (for the convolution: the convolution of |x| with |w|, zero padding included).
* The epilogue, in the kernel's order: ``v = acc + bias``; ``v *= alpha`` (only when alpha != 1); ``v += rowvec``;
  ``v += residual``; the activation.  Each fp32 step costs ``U_F32`` of the running magnitude ``|v| + e``; alpha also
  scales the incoming error by ``|alpha|``.  Adding a zero bias is exact and is not charged.
* SiLU (``silu_f``) and quick GELU (``quick_gelu_f``) are ``x * rcp.approx(1 + ex2.approx(-k x log2 e))`` with k = 1 and
  1.702: their slope, ``sigma(u) + u sigma'(u)`` in ``u = k x``, is at most 1.1 for both; their own relative error is
  ``EX2`` (ex2.approx) + ``2^-22`` (rcp.approx) + ``2 U_F32`` (``1 + e`` and the product) + ``2 k U_F32 |x|`` (the
  fp32 constant ``-k log2 e`` and the product ``x * constant`` are each rounded: an absolute error of ``2 U_F32 |k x
  log2 e|`` in the exponent, which is a relative error of ``2 k U_F32 |x|`` of the exponential); results below 2^-126
  flush to zero (absolute ``FTZ (1 + |x|)``).
* Exact GELU (``gelu_erf_f``, act = 2): slope at most 1.13 (``Phi(x) + x phi(x)`` peaks at x = sqrt 2); own error
  ``0.5 |x| (GELU_ERF + 128 U_F32)`` (the polynomial's 3e-7 and the roundings of six fma, four squarings and the
  approximate reciprocal of ``p^16``) + ``2 U_F32 |gelu(x)|``.
* GEGLU: ``val * gelu_erf_f(gate)`` on the packed 16-column groups (columns 32j..32j+15 value, 32j+16..32j+31 gate):
  ``|dval| |gelu(gate)| + |val| (1.13 |dgate| + 0.5 |gate| (GELU_ERF + 128 U_F32)) + 2 U_F32 |val gelu(gate)|``.
* The output: bf16 rounds once, ``U_BF16 (|ref| + e)``; fp32 output is the last fp32 step and adds nothing.
* ``SAFETY`` covers the second-order products the first-order sums drop.

The bounds are worst cases of that arithmetic, not fits to observed errors: a healthy kernel stays well below 1, and a
defect confined to one tile, one row block or one column chunk shows as ``err / bound`` far above 1 even where a
whole-tensor relative L2 cannot see it.
"""
from __future__ import annotations

import math

import torch
import torch.nn.functional as F

from norm_ref import GELU_ERF
from softmax_ref import EX2, FTZ, SAFETY, U_BF16, U_F32, ACC_ULP, assert_within, mma_terms, rel_l2  # noqa: F401

f64 = torch.float64
bf16 = torch.bfloat16

# gemm_conv.cu constants
BLOCK_M, BLOCK_K, KSUB, HALO_TAPS = 128, 64, 2, 3
A_STAGE_BYTES, A_HALO_BYTES = 128 * 64 * 2, 23 * 1024
MAX_STAGES, MAX_B_STAGES, MAX_A_HALO_STAGES = 8, 16, 4
BAR_REGION_BYTES, EPI_SLABS, SMEM_MAX = 512, 4, 227 * 1024
HALO_TILE_W, HALO_TILE_H = 8, 16


# ------------------------------------------------------------------------------------------------------------------------
# launch geometry (ports of gemm_conv.cu's host code)
# ------------------------------------------------------------------------------------------------------------------------
def pick_bn(m_blocks: int, N: int, k_iters: int, sms: int = 148, cluster: int = 2) -> int:
    """pick_bn: the N tile that minimises waves x per-tile cost."""
    best, best_cost = 128, 1e30
    slots = sms // cluster
    m_groups = (m_blocks + cluster - 1) // cluster
    for bn in range(32, 257, 32):
        if bn > ((N + 31) // 32) * 32 and bn != 32:
            continue
        n_blocks = (N + bn - 1) // bn
        waves = (m_groups * n_blocks + slots - 1) // slots
        tile_cost = max(4.0 * (bn / 2.0), 2.0 * (16384.0 + bn * 128.0 / cluster) / 128.0) * k_iters + 2500.0 + bn * 8.0
        cost = waves * tile_cost
        if cost < best_cost - 1e-9:
            best_cost, best = cost, bn
    return best


def gemm_n_tile(M: int, N: int, K: int, sms: int = 148) -> int:
    """b200sr_gemm_n_tile."""
    mb = -(-M // BLOCK_M)
    return pick_bn(mb, N, -(-K // BLOCK_K), sms, 2 if mb >= 2 else 1)


def conv_box(NB: int, H: int, W: int, stride: int = 1, halo_enabled: bool = True) -> dict:
    """b200sr_conv3x3_bf16's tile box: mode (1 direct, 2 stride 2, 3 halo), (bw, bh, bn) pixels x rows x images of one
    128-row tile, the tile counts and the real M blocks."""
    OH, OW = H // stride, W // stride
    bw = 1
    while bw * 2 <= 128 and OW % (bw * 2) == 0:
        bw *= 2
    bh = 1
    while bw * bh * 2 <= 128 and bh < OH:
        bh *= 2
    bn = 128 // (bw * bh)
    halo = halo_enabled and stride == 1 and W % HALO_TILE_W == 0 and H >= HALO_TILE_H
    if halo:
        bw, bh, bn = HALO_TILE_W, HALO_TILE_H, 1
    tw, th, tn = OW // bw, -(-OH // bh), -(-NB // bn)
    return dict(mode=3 if halo else (1 if stride == 1 else 2), bw=bw, bh=bh, bn=bn, OH=OH, OW=OW, tiles_w=tw, tiles_h=th,
                tiles_n=tn, m_blocks=tw * th * tn)


def plan(M: int, N: int, K: int, m_blocks: int, *, mode: int = 0, Cin: int = 0, force_bn: int = 0, geglu: bool = False,
         out_fp32: bool = False, residual: bool = False, rowvec: bool = False, ldc: int = 0, ldr: int = 0,
         out_align: int = 256, res_align: int = 256, sms: int = 148, wide_enabled: bool = True,
         epi_tma_enabled: bool = True, resident_enabled: bool = True) -> dict:
    """finish + launch_t: cluster, phantom M blocks, BN (picked or forced, the halo cap), N blocks, the wide_io and
    epi_tma conditions, the ring (stages; mode 3: a_stages, w_resident) and the persistent grid.  ``ldc`` / ``ldr`` in
    elements (0 = dense), ``*_align`` the byte alignment of the out / residual base."""
    cluster = 2 if m_blocks >= 2 else 1
    num_m = -(-m_blocks // cluster) * cluster
    k_iters = 9 * (Cin // BLOCK_K) if mode else -(-K // BLOCK_K)
    BN = force_bn if force_bn > 0 else pick_bn(m_blocks, N, k_iters, sms, cluster)
    if mode == 3 and cluster == 1 and BN > 192 and force_bn <= 0:
        BN = 192
    n_blocks = -(-N // BN)
    n_out = N // 2 if geglu else N
    ldc = ldc or n_out
    ldr = ldr or N
    esz = 4 if out_fp32 else 2
    wide = (wide_enabled and not out_fp32 and n_out % 16 == 0 and (ldc * esz) % 32 == 0 and out_align % 32 == 0
            and (not residual or ((ldr * 2) % 32 == 0 and res_align % 32 == 0)))
    work = (num_m // cluster) * n_blocks
    slots = sms // cluster
    epi_tma = (epi_tma_enabled and mode == 0 and out_fp32 and not geglu and not residual and not rowvec and ldc % 4 == 0
               and work >= 2 * slots)
    xform = EPI_SLABS * 4 * 4096 + 1024 if epi_tma else 0
    budget = SMEM_MAX - 1024 - BAR_REGION_BYTES - 4096 - xform
    b_sub = (BN // cluster) * BLOCK_K * 2
    a_stages, w_resident = 0, False
    if mode == 3:
        kc = Cin // BLOCK_K
        b_stage = HALO_TAPS * b_sub
        a_stages = 2 if kc >= 2 else 1
        stages = min((budget - a_stages * A_HALO_BYTES) // b_stage, MAX_B_STAGES)
        assert stages >= 2
        if resident_enabled and n_blocks == 1 and 3 * kc <= stages and 3 * kc <= MAX_B_STAGES:
            w_resident, stages = True, 3 * kc
            while a_stages < MAX_A_HALO_STAGES and (budget - (a_stages + 1) * A_HALO_BYTES) // b_stage >= stages:
                a_stages += 1
    else:
        s_iters = -(-k_iters // KSUB)
        stages = max(2, min(budget // (KSUB * (A_STAGE_BYTES + b_sub)), MAX_STAGES, s_iters + 1))
    grid = min(work, slots) * cluster
    return dict(cluster=cluster, num_m_blocks=num_m, phantom=num_m - m_blocks, BN=BN, num_n_blocks=n_blocks,
                k_iters=k_iters, wide_io=wide, epi_tma=epi_tma, stages=stages, a_stages=a_stages, w_resident=w_resident,
                work=work, grid=grid)


def schedule(p: dict) -> list:
    """The persistent schedule: per CTA pair, its tiles in order as (m_group, n_blk)."""
    m_groups = p["num_m_blocks"] // p["cluster"]
    stride = p["grid"] // p["cluster"]
    return [[(w % m_groups, w // m_groups) for w in range(c, p["work"], stride)] for c in range(stride)]


def n_block_changes(p: dict) -> list:
    """(pair, tile index, previous n_blk, n_blk) of every tile whose CTA pair changes N block from its previous tile:
    where the epilogue stages a new bias slice."""
    out = []
    for c, tiles in enumerate(schedule(p)):
        for i in range(1, len(tiles)):
            if tiles[i][1] != tiles[i - 1][1]:
                out.append((c, i, tiles[i - 1][1], tiles[i][1]))
    return out


def gemm_plan(M, N, K, **kw) -> dict:
    return plan(M, N, K, -(-M // BLOCK_M), **kw)


def conv_plan(NB, H, W, Cin, Cout, stride=1, halo_enabled=True, **kw) -> dict:
    box = conv_box(NB, H, W, stride, halo_enabled)
    p = plan(NB * box["OH"] * box["OW"], Cout, 9 * Cin, box["m_blocks"], mode=box["mode"], Cin=Cin, **kw)
    p.update(box)
    return p


# ------------------------------------------------------------------------------------------------------------------------
# error propagation through the epilogue
# ------------------------------------------------------------------------------------------------------------------------
def _sigmoid_act(v, e, k):
    z = v * torch.sigmoid(k * v)
    return z, 1.1 * e + (EX2 + 2.0 ** -22 + 2 * U_F32 + 2 * k * U_F32 * v.abs()) * z.abs() + FTZ * (1.0 + v.abs())


def _gelu(v):
    return 0.5 * v * (1.0 + torch.erf(v / math.sqrt(2.0)))


def _gelu_act(v, e):
    z = _gelu(v)
    return z, 1.13 * e + 0.5 * v.abs() * (GELU_ERF + 128 * U_F32) + 2 * U_F32 * z.abs()


def f32(x: float) -> float:
    """The fp32 value the kernel holds for a Python float (alpha crosses the ABI as a C float)."""
    return float(torch.tensor(x, dtype=torch.float32))


def epilogue(acc, e, *, bias=None, alpha=1.0, rv=None, res=None, act=0, geglu=False, out_fp32=False):
    """(ref, bound) from the float64 accumulator ``acc`` [M, N] and its bound ``e``: the epilogue in the kernel's order
    with the costs of the module docstring.  ``rv`` / ``res``: float64 [M, N] (rowvec already expanded per row)."""
    v = acc
    if bias is not None:
        v = v + bias.to(f64)[None]
        e = e + U_F32 * (v.abs() + e)
    if geglu:
        M, N = v.shape
        vv, ee = v.view(M, N // 32, 2, 16), e.view(M, N // 32, 2, 16)
        val, gate, e_val, e_gate = vv[:, :, 0], vv[:, :, 1], ee[:, :, 0], ee[:, :, 1]
        gl = _gelu(gate)
        y = (val * gl).reshape(M, N // 2)
        e = (gl.abs() * e_val + val.abs() * (1.13 * e_gate + 0.5 * gate.abs() * (GELU_ERF + 128 * U_F32))
             + 2 * U_F32 * (val * gl).abs()).reshape(M, N // 2)
    else:
        a = f32(alpha)
        if a != 1.0:
            v = v * a
            e = abs(a) * e + U_F32 * (v.abs() + abs(a) * e)
        for t in (rv, res):
            if t is not None:
                v = v + t
                e = e + U_F32 * (v.abs() + e)
        if act == 1:
            v, e = _sigmoid_act(v, e, 1.0)
        elif act == 2:
            v, e = _gelu_act(v, e)
        elif act == 3:
            v, e = _sigmoid_act(v, e, 1.702)
        y = v
    if not out_fp32:
        e = e + U_BF16 * (y.abs() + e)
    return y, SAFETY * e


# ------------------------------------------------------------------------------------------------------------------------
# references
# ------------------------------------------------------------------------------------------------------------------------
def _chunk(n_cols: int) -> int:
    return max(1, (1 << 23) // max(1, n_cols))


def gemm(a, w, *, bias=None, alpha=1.0, rowvec=None, rows_per_group=0, residual=None, act=0, geglu=False,
         w_rows_per_group=0, out_fp32=False):
    """b200sr_gemm_bf16 in float64: (ref, bound) [M, N] (GEGLU: [M, N / 2]).  a [M, K] bf16 (any row stride), w [N, K]
    or [G, N, K] (group g serves rows [g w_rows_per_group, (g + 1) w_rows_per_group)), rowvec [groups, >= N] fp32
    (row m uses group m // rows_per_group), residual [M, >= N] bf16.  Row chunks of float64 matmuls on a's device."""
    M, K = a.shape
    w3 = w if w.dim() == 3 else w[None]
    N = w3.shape[1]
    kpad = -(-K // BLOCK_K) * BLOCK_K
    acc = torch.empty(M, N, dtype=f64, device=a.device)
    mag = torch.empty_like(acc)
    rpg = w_rows_per_group or M
    step = min(_chunk(N + K), rpg)
    for g0 in range(0, M, rpg):
        wg = w3[g0 // rpg if w_rows_per_group else 0].to(f64)
        wa = wg.abs()
        for r0 in range(g0, min(M, g0 + rpg), step):
            r1 = min(M, g0 + rpg, r0 + step)
            ar = a[r0:r1].to(f64)
            acc[r0:r1] = ar @ wg.T
            mag[r0:r1] = ar.abs() @ wa.T
    e = mma_terms(kpad) * ACC_ULP * mag
    del mag
    rv = None
    if rowvec is not None:
        grp = torch.arange(M, device=a.device) // rows_per_group if rows_per_group else torch.zeros(M, dtype=torch.long,
                                                                                                   device=a.device)
        rv = rowvec[:, :N].to(f64)[grp]
    res = residual[:, :N].to(f64) if residual is not None else None
    return epilogue(acc, e, bias=bias, alpha=alpha, rv=rv, res=res, act=act, geglu=geglu, out_fp32=out_fp32)


def unpack_conv(wp: torch.Tensor) -> torch.Tensor:
    """Packed [Cout, 9 Cin] (K = (kh 3 + kw) Cin + c) -> float64 [Cout, Cin, 3, 3]."""
    co = wp.shape[0]
    return wp.to(f64).view(co, 3, 3, -1).permute(0, 3, 1, 2)


def conv_cols(x: torch.Tensor, stride: int = 1, pad_lo: int = 1) -> torch.Tensor:
    """The implicit GEMM's A operand in float64: [NB OH OW, 9 Cin], row (n, oh, ow), column (kh 3 + kw) Cin + c, zero
    padding 1 on every side, or (0, 1, 0, 1) for pad_lo = 0."""
    n, h, wd, c = x.shape
    xp = x.to(f64).permute(0, 3, 1, 2)
    xp = F.pad(xp, (1, 1, 1, 1) if pad_lo else (0, 1, 0, 1))
    oh, ow = h // stride, wd // stride
    taps = [xp[:, :, kh:kh + stride * oh:stride, kw:kw + stride * ow:stride] for kh in range(3) for kw in range(3)]
    return torch.stack(taps, 1).permute(0, 3, 4, 1, 2).reshape(n * oh * ow, 9 * c)


def conv3x3(x, wp, *, stride=1, pad_lo=1, bias=None, rowvec=None, residual=None, alpha=1.0, act=0):
    """b200sr_conv3x3_bf16 in float64: (ref, bound) [NB, OH, OW, Cout].  x [NB, H, W, Cin] bf16, wp packed [Cout, 9 Cin]
    bf16, rowvec [NB, >= Cout] fp32 (one row per image), residual [NB, OH, OW, >= Cout] bf16.  The accumulator and its
    magnitude are float64 convolutions (of x and of |x|; padding as the kernel pads), image by image."""
    n, h, wd, cin = x.shape
    co = wp.shape[0]
    oh, ow = h // stride, wd // stride
    w4 = unpack_conv(wp)
    wa = w4.abs()
    acc = torch.empty(n, co, oh, ow, dtype=f64, device=x.device)
    mag = torch.empty_like(acc)
    for i in range(n):
        xi = x[i:i + 1].to(f64).permute(0, 3, 1, 2)
        if pad_lo or stride == 1:
            acc[i:i + 1] = F.conv2d(xi, w4, stride=stride, padding=1)
            mag[i:i + 1] = F.conv2d(xi.abs(), wa, stride=stride, padding=1)
        else:
            xi = F.pad(xi, (0, 1, 0, 1))
            acc[i:i + 1] = F.conv2d(xi, w4, stride=stride)
            mag[i:i + 1] = F.conv2d(xi.abs(), wa, stride=stride)
    acc = acc.permute(0, 2, 3, 1).reshape(-1, co)
    e = mma_terms(9 * cin) * ACC_ULP * mag.permute(0, 2, 3, 1).reshape(-1, co)
    del mag
    rv = rowvec[:, :co].to(f64).repeat_interleave(oh * ow, 0) if rowvec is not None else None
    res = residual[..., :co].reshape(-1, residual.shape[-1])[:, :co].to(f64) if residual is not None else None
    y, b = epilogue(acc, e, bias=bias, alpha=alpha, rv=rv, res=res, act=act)
    return y.view(n, oh, ow, co), b.view(n, oh, ow, co)


# ------------------------------------------------------------------------------------------------------------------------
# designed inputs (deterministic, seeded; CPU generator so the same values arise on every machine)
# ------------------------------------------------------------------------------------------------------------------------
def gemm_inputs(M: int, N: int, K: int, *, groups: int = 1, seed: int = 0):
    """(a [M, K] bf16, w [N, K] (or [groups, N, K]) bf16, bias [N], rowvec [M, N] source, residual [M, N]), CPU.

    Rows of a carry scales 2^(m % 5 - 2); the columns of the last (ragged) 64-wide K chunk are 4x larger, so that chunk
    holds a large share of every dot product.  Bias, rowvec and residual are of the product's size, and differ per
    column, group and row."""
    g = torch.Generator().manual_seed(seed)
    a = torch.randn(M, K, generator=g, dtype=f64)
    a *= torch.exp2((torch.arange(M) % 5 - 2).to(f64))[:, None]
    last = (-(-K // BLOCK_K) - 1) * BLOCK_K
    a[:, last:] *= 4.0
    w = torch.randn(groups, N, K, generator=g, dtype=f64) * (2.0 / K) ** 0.5
    bias = 2.0 * torch.randn(N, generator=g)
    rowvec = 2.0 * torch.randn(M, N, generator=g)
    res = 2.0 * torch.randn(M, N, generator=g, dtype=f64)
    w = w.to(bf16)
    return a.to(bf16), (w[0] if groups == 1 else w).contiguous(), bias, rowvec, res.to(bf16)


def conv_inputs(NB: int, H: int, W: int, Cin: int, Cout: int, *, stride: int = 1, seed: int = 0):
    """(x [NB, H, W, Cin] bf16, packed w [Cout, 9 Cin] bf16, bias [Cout], rowvec [NB, Cout], residual [NB, OH, OW, Cout]
    bf16), CPU.

    Each image has its own offset; its border rows and columns are set to +-(6 + noise) with the sign of the image, so a
    tap that reads a neighbour instead of the zero padding, or pads the wrong side, moves the result by many bounds."""
    g = torch.Generator().manual_seed(seed)
    x = 0.5 * torch.randn(NB, H, W, Cin, generator=g, dtype=f64) + torch.randn(NB, 1, 1, 1, generator=g, dtype=f64)
    sign = torch.where(torch.arange(NB) % 2 == 0, 1.0, -1.0).to(f64)[:, None, None, None]
    border = torch.zeros(1, H, W, 1, dtype=torch.bool)
    border[:, 0], border[:, -1], border[:, :, 0], border[:, :, -1] = True, True, True, True
    x = torch.where(border, sign * (6.0 + torch.randn(NB, H, W, Cin, generator=g, dtype=f64)), x)
    w = (torch.randn(Cout, 9 * Cin, generator=g, dtype=f64) * (1.0 / (9 * Cin)) ** 0.5).to(bf16)
    bias = 2.0 * torch.randn(Cout, generator=g)
    rowvec = 2.0 * torch.randn(NB, Cout, generator=g)
    OH, OW = H // stride, W // stride
    res = (2.0 * torch.randn(NB, OH, OW, Cout, generator=g, dtype=f64)).to(bf16)
    return x.to(bf16), w.contiguous(), bias, rowvec, res


# ------------------------------------------------------------------------------------------------------------------------
# guarded windows
# ------------------------------------------------------------------------------------------------------------------------
class Guarded:
    """A [rows, cols] window with row stride ``ld`` inside a sentinel-filled buffer: ``before`` / ``after`` whole rows
    around it and, in every row, the columns outside [col, col + cols).  ``col`` keeps the window's base 16-byte aligned
    (``col * element size % 16 == 0``) and 32-byte aligned when ``col * element size % 32 == 0``."""

    def __init__(self, rows, cols, ld, dtype, device, *, col=0, fill=float("nan"), before=2, after=2, values=None):
        assert col + cols <= ld
        self.rows, self.cols, self.ld, self.col, self.before, self.after = rows, cols, ld, col, before, after
        self.buf = torch.full(((before + rows + after) * ld + 64,), fill, dtype=dtype, device=device)
        base = self.buf.data_ptr()
        # the window's alignment is that of its offset (allocations are at least 64-byte aligned)
        assert base % 64 == 0
        self.view = self.buf[before * ld + col:].as_strided((rows, cols), (ld, 1))
        if values is not None:
            self.view.copy_(values)
        self.fill = fill

    def sentinels(self):
        """Every element of the buffer outside the window."""
        full = self.buf[:(self.before + self.rows + self.after) * self.ld].view(-1, self.ld)
        mask = torch.ones_like(full, dtype=torch.bool)
        mask[self.before:self.before + self.rows, self.col:self.col + self.cols] = False
        return torch.cat([full[mask], self.buf[(self.before + self.rows + self.after) * self.ld:]])

    def check(self, what: str, window_finite: bool = True):
        s = self.sentinels()
        ok = bool(s.isnan().all()) if math.isnan(self.fill) else bool((s == self.fill).all())
        assert ok, f"{what}: {int((~(s.isnan() if math.isnan(self.fill) else s == self.fill)).sum())} sentinels overwritten"
        if window_finite:
            assert bool(self.view.isfinite().all()), f"{what}: NaN / inf in the window"
