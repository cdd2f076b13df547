"""Operator layer: torch tensors in, libb200sr.so kernels underneath (through the C ABI).

Conventions
-----------
* activations are contiguous **bf16, channels last**: images ``[N, H, W, C]``, tokens ``[B, T, C]``;
* parameters handed to the kernels are *packed* once by the modules (``pack_linear`` /
  ``pack_conv3x3``): bf16, K-major, conv taps flattened as ``K = (kh*3 + kw) * Cin + c``;
* biases / norm affine parameters stay fp32;
* every call is enqueued on ``torch.cuda.current_stream()``; nothing synchronises.

There is no CPU path and no torch fallback here: tensors that are not CUDA tensors raise.
"""
from __future__ import annotations

import ctypes as C
import math
from typing import Optional

import numpy as np
import torch

from . import _lib
from ._lib import Epilogue, check

bf16 = torch.bfloat16


def launch_count() -> int:
    """Number of b200sr kernels enqueued by this process so far."""
    return _lib.LAUNCHES[0]


# Optional per-launch timing (bench.py roofline leg): when a list is installed, every gemm / conv3x3 / attention /
# group_norm / layer_norm launch is bracketed by CUDA events on the launching stream and appended as
# (kind, algorithmic work, start_event, end_event, description); work = FLOPs for the dense kernels and
# algorithmic bytes (each operand read once, the result written once, bf16) for the normalisation kernels.
_profile = None


def set_profile(records) -> None:
    global _profile
    _profile = records


class _Timed:
    def __init__(self, kind: str, flops: float, desc: str = ""):
        self.kind, self.flops, self.desc = kind, flops, desc

    def __enter__(self):
        if _profile is not None:
            self.t0 = torch.cuda.Event(enable_timing=True)
            self.t1 = torch.cuda.Event(enable_timing=True)
            self.t0.record()
        return self

    def __exit__(self, *exc):
        if _profile is not None:
            self.t1.record()
            _profile.append((self.kind, self.flops, self.t0, self.t1, self.desc))
        return False


def _stream() -> int:
    return torch.cuda.current_stream().cuda_stream


def _ptr(t: Optional[torch.Tensor]) -> Optional[int]:
    return None if t is None else t.data_ptr()


def _req(t: torch.Tensor, dtype, name: str) -> None:
    if not t.is_cuda:
        raise _lib.B200SRError(f"{name}: expected a CUDA tensor (b200sr has no CPU path)")
    if t.device.index != torch.cuda.current_device():
        # kernels are enqueued on the *current* device's current stream: one process drives one GPU, or the
        # caller selects the device (torch.cuda.device / set_device) around the call
        raise _lib.B200SRError(f"{name}: tensor lives on {t.device} but the current CUDA device is "
                               f"{torch.cuda.current_device()}; wrap the call in torch.cuda.device(tensor.device)")
    if t.dtype != dtype:
        raise _lib.B200SRError(f"{name}: expected {dtype}, got {t.dtype}")
    if not t.is_contiguous():
        raise _lib.B200SRError(f"{name}: expected a contiguous tensor")


def require_cuda(t: torch.Tensor, what: str) -> None:
    """The product path refuses host tensors up front (there is no CPU fallback)."""
    if not t.is_cuda:
        raise _lib.B200SRError(f"{what} runs on CUDA (sm_100a) only; there is no CPU fallback")


_ws_cache: dict = {}
_ws_retired: list = []  # outgrown scratch buffers: never freed, captured CUDA graphs may still hold their addresses
_ws_slot = [0]  # scratch buffers are per (device, slot): work issued concurrently on a second stream uses slot 1


class workspace_slot:
    """Context manager selecting the scratch-buffer slot for ops enqueued inside it (one per concurrent stream)."""

    def __init__(self, slot: int):
        self.slot = slot

    def __enter__(self):
        self.prev = _ws_slot[0]
        _ws_slot[0] = self.slot

    def __exit__(self, *exc):
        _ws_slot[0] = self.prev
        return False


def _workspace(device: torch.device, nbytes: int, kind: str = "gn") -> torch.Tensor:
    """Zero-initialised scratch per (device, stream slot, kernel family); the kernels keep their arrival
    counters at its start zeroed between launches, so it is reused by every call of that family.
    A buffer that has been handed out is never freed: a CUDA graph captured earlier (by this or another
    engine) has its address baked in and would otherwise write into recycled memory on replay.  An outgrown
    buffer is parked in ``_ws_retired``; sizes grow geometrically (floor 16 MB), so there are few of those."""
    key = (device.type, device.index, _ws_slot[0], kind)
    ws = _ws_cache.get(key)
    if ws is None or ws.numel() * 4 < nbytes:
        if torch.cuda.is_current_stream_capturing():
            raise _lib.B200SRError("workspace allocation during CUDA-graph capture; run one eager warm-up step first")
        if ws is not None:
            _ws_retired.append(ws)
        floats = max(nbytes // 4 + 1, 1 << 22, 0 if ws is None else 2 * ws.numel())
        ws = torch.zeros(floats, dtype=torch.float32, device=device)
        _ws_cache[key] = ws
    return ws


# ------------------------------------------------------------------------------------------------
# parameter packing (runs once per module, on whatever device the parameter lives on)
# ------------------------------------------------------------------------------------------------
def pack_linear(weight: torch.Tensor) -> torch.Tensor:
    """nn.Linear / 1x1-conv weight [N, K(,1,1)] fp32 -> bf16 [N, K] (K-major B operand)."""
    w = weight.detach().reshape(weight.shape[0], -1)
    return w.to(bf16).contiguous()


def pack_conv3x3(weight: torch.Tensor) -> torch.Tensor:
    """nn.Conv2d weight [Cout, Cin, 3, 3] fp32 -> bf16 [Cout, 9*Cin] with K = (kh*3+kw)*Cin + c."""
    co, ci, kh, kw = weight.shape
    assert kh == 3 and kw == 3
    return weight.detach().permute(0, 2, 3, 1).reshape(co, 9 * ci).to(bf16).contiguous()


def geglu_interleave_index(inner: int, device=None) -> torch.Tensor:
    """Row permutation for the GEGLU projection (attention.py:84-91): the reference computes
    ``x, gate = proj(x).chunk(2)``; the kernel epilogue wants value / gate rows of the same 16
    output features adjacent: packed rows 32k..32k+15 = value 16k..16k+15, 32k+16..32k+31 = gate."""
    assert inner % 16 == 0
    j = torch.arange(inner, device=device)
    val_pos = (j // 16) * 32 + (j % 16)
    idx = torch.empty(2 * inner, dtype=torch.long, device=device)
    idx[val_pos] = j
    idx[val_pos + 16] = j + inner
    return idx


def pack_geglu(weight: torch.Tensor, bias: torch.Tensor):
    inner = weight.shape[0] // 2
    idx = geglu_interleave_index(inner, weight.device)
    return weight.detach()[idx].to(bf16).contiguous(), bias.detach()[idx].float().contiguous()


def pack_linear_ln(weight: torch.Tensor, gamma: torch.Tensor, beta: torch.Tensor, bias: Optional[torch.Tensor] = None):
    """Operands of ``gemm(..., ln=...)`` for Linear(LayerNorm(x)): (W' = W * gamma as bf16 [N, K], colsum [1, N] of the
    ROUNDED W' so the mean term cancels exactly what the tensor cores accumulate, shift = W beta + bias [1, N])."""
    w32 = weight.detach().float()
    wp = (w32 * gamma.detach().float()[None, :]).to(bf16).contiguous()
    shift = w32 @ beta.detach().float()
    if bias is not None:
        shift = shift + bias.detach().float()
    return wp, wp.float().sum(1)[None].contiguous(), shift[None].contiguous()


def pack_geglu_ln(weight: torch.Tensor, bias: torch.Tensor, gamma: torch.Tensor, beta: torch.Tensor):
    """pack_linear_ln for the GEGLU projection: rows interleaved as pack_geglu does."""
    idx = geglu_interleave_index(weight.shape[0] // 2, weight.device)
    return pack_linear_ln(weight.detach()[idx], gamma, beta, bias.detach()[idx])


class RowStats:
    """Per-row partial (sum, sum of squares) of a bf16 [M, N] GEMM output, one pair per N tile of the GEMM that wrote it:
    buf [parts, M, 2] fp32.  Consumed by ``gemm(..., ln=(stats, colsum, shift, eps))``."""

    __slots__ = ("buf", "parts", "dim")

    def __init__(self, buf: torch.Tensor, parts: int, dim: int):
        self.buf, self.parts, self.dim = buf, parts, dim


_n_tile_cache: dict = {}


def gemm_n_tile(M: int, N: int, K: int) -> int:
    key = (M, N, K)
    t = _n_tile_cache.get(key)
    if t is None:
        t = _lib.load().b200sr_gemm_n_tile(M, N, K)
        if t <= 0:
            raise _lib.B200SRError(f"gemm_n_tile({M}, {N}, {K}) = {t}")
        _n_tile_cache[key] = t
    return t


# ------------------------------------------------------------------------------------------------
# dense contractions
# ------------------------------------------------------------------------------------------------
def _epilogue(out, ldc, bias, rowvec, rows_per_group, residual, ldr, out_fp32, geglu, alpha, act=0,
              softmax_valid=0, w_rows_per_group=0, w_group_stride=0, w_dynamic=False) -> Epilogue:
    e = Epilogue()
    e.bias = _ptr(bias)
    e.rowvec = _ptr(rowvec)
    e.rows_per_group = rows_per_group
    e.ld_rowvec = rowvec.stride(0) if rowvec is not None and rowvec.dim() == 2 else 0
    e.residual = _ptr(residual)
    e.ldr = ldr
    e.out = out.data_ptr()
    e.ldc = ldc
    e.out_fp32 = int(out_fp32)
    e.geglu = int(geglu)
    e.alpha = float(alpha)
    e.act = int(act)
    e.softmax_valid = int(softmax_valid)
    e.w_dynamic = int(w_dynamic)
    e.w_rows_per_group = int(w_rows_per_group)
    e.w_group_stride = int(w_group_stride)
    return e


def gemm(
    a: torch.Tensor,
    w: torch.Tensor,
    bias: Optional[torch.Tensor] = None,
    *,
    residual: Optional[torch.Tensor] = None,
    rowvec: Optional[torch.Tensor] = None,
    rows_per_group: int = 0,
    geglu: bool = False,
    alpha: float = 1.0,
    act: int = 0,
    out: Optional[torch.Tensor] = None,
    out_fp32: bool = False,
    force_bn: int = 0,
    softmax_valid: int = 0,
    w_rows_per_group: int = 0,
    w_dynamic: bool = False,
    ln=None,
    want_stats: bool = False,
):
    """``out = alpha * (a @ w.T + bias) + rowvec[group] + residual`` (or GEGLU).  a: [..., K] bf16
    (last-dim contiguous, uniform row stride), w: [N, K] packed bf16.  `out` may be a column
    slice of a wider row-major tensor (its row stride is honoured).
    `w_rows_per_group` > 0: w is [G, N, K] and rows [g * w_rows_per_group, ...) of a use w[g] (per-batch-element
    operands).  `softmax_valid` > 0: the epilogue is a row softmax (base 2, no scale) over each 80-column segment
    of which the first `softmax_valid` columns take part; output bf16 probabilities.
    `w_dynamic`: w was written by an earlier kernel on this stream (an activation used as the B operand): the
    kernel then must not prefetch it ahead of its programmatic dependency.
    `ln` = (RowStats of a, colsum, shift, eps): a holds RAW rows and the LayerNorm in front of the Linear is folded into
    the epilogue (operands from pack_linear_ln; colsum / shift are [G, N] with per-group weights).
    `want_stats`: also return the RowStats of the bf16 output -> (out, stats)."""
    _req(w, bf16, "gemm.w")
    if a.dtype != bf16 or not a.is_cuda:
        raise _lib.B200SRError("gemm.a: expected CUDA bf16")
    K = a.shape[-1]
    N = w.shape[-2]
    w_group_stride = 0
    if w_rows_per_group:
        assert w.dim() == 3 and w.is_contiguous() and w.shape[0] * w_rows_per_group >= a.numel() // K
        w_group_stride = N
    a2 = a.reshape(-1, K)
    if a2.stride(-1) != 1:
        a2 = a2.contiguous()
    M, lda = a2.shape[0], a2.stride(0)
    n_out = N // 2 if geglu else N
    if out is None:
        out = torch.empty(*a.shape[:-1], n_out, dtype=torch.float32 if out_fp32 else bf16, device=a.device)
    o2 = out.reshape(-1, n_out) if out.is_contiguous() else out
    assert o2.shape[-1] == n_out and o2.stride(-1) == 1
    ldc = o2.stride(-2) if o2.dim() >= 2 else n_out
    ldr = 0
    if residual is not None:
        r2 = residual if residual.dim() == 2 else residual.reshape(-1, residual.shape[-1])
        assert r2.dtype == bf16 and r2.stride(-1) == 1
        ldr = r2.stride(0)
    e = _epilogue(o2, ldc, bias, rowvec, rows_per_group, residual, ldr, out_fp32, geglu, alpha, act,
                  softmax_valid, w_rows_per_group, w_group_stride, w_dynamic)
    if ln is not None:
        st, colsum, shift, eps = ln
        groups = w.shape[0] if w_rows_per_group else 1
        if st.buf.shape[1] != M or st.dim != K:
            raise _lib.B200SRError(f"gemm.ln: statistics of a [{st.buf.shape[1]}, {st.dim}] matrix, a is [{M}, {K}]")
        for t, nme in ((colsum, "colsum"), (shift, "shift")):
            _req(t, torch.float32, f"gemm.ln.{nme}")
            if t.numel() != groups * N:
                raise _lib.B200SRError(f"gemm.ln.{nme}: expected [{groups}, {N}]")
        e.ln_stats, e.ln_parts, e.ln_colsum, e.ln_shift, e.ln_eps = st.buf.data_ptr(), st.parts, colsum.data_ptr(), \
            shift.data_ptr(), float(eps)
    stats = None
    if want_stats:
        if geglu or softmax_valid or out_fp32:
            raise _lib.B200SRError("gemm.want_stats: plain bf16 output only")
        parts = -(-N // (force_bn if force_bn > 0 else gemm_n_tile(M, N, K)))
        stats = RowStats(torch.empty(parts, M, 2, dtype=torch.float32, device=a.device), parts, N)
        e.ln_stats_out = stats.buf.data_ptr()
    with _Timed("gemm", 2.0 * M * N * K, f"M{M} N{N} K{K}{' geglu' if geglu else ''}{' ln' if ln is not None else ''}"):
        rc = _lib.load().b200sr_gemm_bf16(a2.data_ptr(), lda, w.data_ptr(), M, N, K, C.byref(e), force_bn, _stream())
    check(rc, f"gemm M={M} N={N} K={K}")
    return (out, stats) if want_stats else out


def conv3x3(
    x: torch.Tensor,
    w: torch.Tensor,
    bias: Optional[torch.Tensor] = None,
    *,
    stride: int = 1,
    rowvec: Optional[torch.Tensor] = None,
    residual: Optional[torch.Tensor] = None,
    alpha: float = 1.0,
    act: int = 0,
    out: Optional[torch.Tensor] = None,
    force_bn: int = 0,
    pad_lo: int = 1,
    gn=None,
) -> torch.Tensor:
    """3x3 conv, pad 1.  x: [N, H, W, Cin] bf16; w: packed [Cout, 9*Cin]; rowvec: fp32 [N, Cout]
    (added per image: ResBlock emb); residual: bf16 [N, OH, OW, Cout].  pad_lo = 0 (stride 2): pad (0, 1, 0, 1).
    gn = (stats, weight, bias, groups, silu): x is the RAW tensor and GroupNorm(+SiLU) is applied to the staged input
    tiles inside the kernel (stats from group_norm_stats; only where conv3x3_gn_fusable(x, stride))."""
    _req(x, bf16, "conv3x3.x")
    _req(w, bf16, "conv3x3.w")
    n, h, wd, cin = x.shape
    cout = w.shape[0]
    assert w.shape[1] == 9 * cin
    oh, ow = h // stride, wd // stride
    if out is None:
        out = torch.empty(n, oh, ow, cout, dtype=bf16, device=x.device)
    ldc = out.stride(2)
    ldr = residual.stride(2) if residual is not None else 0
    e = _epilogue(out, ldc, bias, rowvec, 0, residual, ldr, False, False, alpha, act)
    if gn is not None:
        stats, gw, gb, groups, gsilu = gn
        _req(stats, torch.float32, "conv3x3.gn.stats")
        e.a_gn_stats, e.a_gn_weight, e.a_gn_bias = stats.data_ptr(), gw.data_ptr(), gb.data_ptr()
        e.a_gn_groups, e.a_gn_silu = int(groups), int(gsilu)
    with _Timed("conv3x3", 2.0 * n * oh * ow * cout * 9 * cin, f"{n}x{h}x{wd} Cin{cin} Cout{cout} s{stride}"):
        rc = _lib.load().b200sr_conv3x3_bf16(
            x.data_ptr(), w.data_ptr(), n, h, wd, cin, cout, stride, pad_lo, C.byref(e), force_bn, _stream()
        )
    check(rc, f"conv3x3 N={n} H={h} W={wd} Cin={cin} Cout={cout} s={stride}")
    return out


def conv3x3_small(
    x: torch.Tensor,
    w: torch.Tensor,
    bias: Optional[torch.Tensor],
    *,
    addend: Optional[torch.Tensor] = None,
    out_nchw_f32: bool = False,
) -> torch.Tensor:
    _req(x, bf16, "conv3x3_small.x")
    _req(w, bf16, "conv3x3_small.w")
    n, h, wd, cin = x.shape
    cout = w.shape[0]
    if out_nchw_f32:
        out = torch.empty(n, cout, h, wd, dtype=torch.float32, device=x.device)
    else:
        out = torch.empty(n, h, wd, cout, dtype=bf16, device=x.device)
    rc = _lib.load().b200sr_conv3x3_small(
        x.data_ptr(), w.data_ptr(), _ptr(bias), _ptr(addend), out.data_ptr(), n, h, wd, cin, cout, int(out_nchw_f32),
        _stream()
    )
    check(rc, f"conv3x3_small Cin={cin} Cout={cout}")
    return out


# ------------------------------------------------------------------------------------------------
# normalisation
# ------------------------------------------------------------------------------------------------
def group_norm(
    x: torch.Tensor,
    weight: Optional[torch.Tensor],
    bias: Optional[torch.Tensor],
    *,
    groups: int = 32,
    eps: float = 1e-5,
    silu: bool = False,
    sft_gamma: Optional[torch.Tensor] = None,
    sft_beta: Optional[torch.Tensor] = None,
    raw: Optional[torch.Tensor] = None,
    control_scale: float = 1.0,
) -> torch.Tensor:
    """GroupNorm over channels-last x: [N, ..., C] bf16 (+SiLU) (+ZeroSFT modulation)."""
    _req(x, bf16, "group_norm.x")
    n, c = x.shape[0], x.shape[-1]
    hw = x.numel() // (n * c)
    lib = _lib.load()
    ws = _workspace(x.device, lib.b200sr_group_norm_workspace_bytes(n, hw, c, groups))
    y = torch.empty_like(x)
    nbytes = 2.0 * x.numel() * (2 + (2 if sft_gamma is not None else 0) + (1 if raw is not None and control_scale != 1.0 else 0))
    with _Timed("group_norm", nbytes, f"N{n} HW{hw} C{c}{' sft' if sft_gamma is not None else ''}"):
        rc = lib.b200sr_group_norm_nhwc(
            x.data_ptr(), y.data_ptr(), _ptr(weight), _ptr(bias), n, hw, c, groups, eps, int(silu), _ptr(sft_gamma),
            _ptr(sft_beta), _ptr(raw), float(control_scale), ws.data_ptr(), _stream()
        )
    check(rc, f"group_norm N={n} HW={hw} C={c}", kernels=max(1, lib.b200sr_group_norm_launches(n, hw, c, groups)))
    return y


GN_FUSE_MAX_COUT = 256   # one N tile: every staged input tile is normalised exactly once


def conv3x3_gn_fusable(x: torch.Tensor, stride: int = 1, cout: Optional[int] = None) -> bool:
    """Shapes the halo-path convolution (and with it the fused input GroupNorm) covers; with `cout`, also whether fusing
    pays: measured in-graph (tools/bench_graph_ops.py gnconv), stats + fused conv vs GroupNorm + conv is 263 vs 343 us at
    1x1024^2 64->64 and 136 vs 169 us at 1x512^2 128->128, but 74 vs 66 us at 2x32^2 1280->1280, where five N tiles each
    re-normalise the same input tile and the transform no longer hides under the MMAs."""
    ok = stride == 1 and x.dim() == 4 and x.shape[2] % 8 == 0 and x.shape[1] >= 16 and x.shape[3] % 64 == 0
    return ok and (cout is None or cout <= GN_FUSE_MAX_COUT)


def group_norm_stats(x: torch.Tensor, groups: int = 32, eps: float = 1e-5) -> torch.Tensor:
    """(mean, rstd) per (image, group) of channels-last x: fp32 [N, groups, 2] (the statistics pass of group_norm)."""
    _req(x, bf16, "group_norm_stats.x")
    n, c = x.shape[0], x.shape[-1]
    hw = x.numel() // (n * c)
    lib = _lib.load()
    ws = _workspace(x.device, lib.b200sr_group_norm_workspace_bytes(n, hw, c, groups))
    stats = torch.empty(n, groups, 2, dtype=torch.float32, device=x.device)
    with _Timed("group_norm", 2.0 * x.numel(), f"N{n} HW{hw} C{c} stats"):
        rc = lib.b200sr_group_norm_stats(x.data_ptr(), n, hw, c, groups, eps, stats.data_ptr(), ws.data_ptr(), _stream())
    check(rc, f"group_norm_stats N={n} HW={hw} C={c}")
    return stats


def layer_norm(x: torch.Tensor, weight: torch.Tensor, bias: torch.Tensor, eps: float = 1e-5) -> torch.Tensor:
    _req(x, bf16, "layer_norm.x")
    c = x.shape[-1]
    m = x.numel() // c
    y = torch.empty_like(x)
    with _Timed("layer_norm", 4.0 * x.numel(), f"M{m} C{c}"):
        rc = _lib.load().b200sr_layer_norm(x.data_ptr(), y.data_ptr(), weight.data_ptr(), bias.data_ptr(), m, c, eps, _stream())
    check(rc, f"layer_norm M={m} C={c}")
    return y


# ------------------------------------------------------------------------------------------------
# attention
# ------------------------------------------------------------------------------------------------
def attention(
    q: torch.Tensor, k: torch.Tensor, v: torch.Tensor, heads: int, *, q_col: int = 0, k_col: int = 0, v_col: int = 0,
    scale: Optional[float] = None, causal: bool = False
) -> torch.Tensor:
    """q: [B, Nq, ldq], k / v: [B, Nk, ld] row-major bf16 matrices; head h of q occupies columns
    [q_col + 64h, q_col + 64h + 64) (likewise k_col / v_col) so a fused QKV buffer can be passed
    three times with different offsets.  Returns [B, Nq, heads*64]."""
    for t, nme in ((q, "q"), (k, "k"), (v, "v")):
        _req(t, bf16, f"attention.{nme}")
    b, nq, ldq = q.shape
    nk = k.shape[1]
    out = torch.empty(b, nq, heads * 64, dtype=bf16, device=q.device)
    lib = _lib.load()
    ws_bytes = lib.b200sr_attention_d64_workspace_bytes(b, heads, nq, nk)
    ws = _workspace(q.device, ws_bytes, "attn") if ws_bytes else None
    with _Timed("attention", 4.0 * b * heads * nq * nk * 64, f"B{b} H{heads} Nq{nq} Nk{nk}"):
        rc = lib.b200sr_attention_d64(
            q.data_ptr(), ldq, q_col, k.data_ptr(), k.shape[2], k_col, v.data_ptr(), v.shape[2], v_col, out.data_ptr(),
            heads * 64, b, heads, nq, nk, float(scale if scale is not None else 0.125), int(causal), _ptr(ws), _stream()
        )
    check(rc, f"attention B={b} H={heads} Nq={nq} Nk={nk}")
    return out


def softmax_rows(x: torch.Tensor, scale: float = 1.0, valid_cols: Optional[int] = None) -> torch.Tensor:
    """softmax(x * scale) over the first `valid_cols` columns (others -> 0): fp32 [..., cols] -> bf16."""
    _req(x, torch.float32, "softmax_rows.x")
    cols = x.shape[-1]
    y = torch.empty(x.shape, dtype=bf16, device=x.device)
    check(_lib.load().b200sr_softmax_rows(x.data_ptr(), y.data_ptr(), x.numel() // cols, cols,
                                          cols if valid_cols is None else valid_cols, float(scale), _stream()),
          "softmax_rows")
    return y


SCORE_CHUNK_BYTES = 1 << 30   # fp32 score rows held at once by single_head_attention (T = 16384: the whole 1 GB matrix)


def gemm_row_softmax(a: torch.Tensor, w: torch.Tensor, scale: float, valid_cols: Optional[int] = None,
                     w_dynamic: bool = True) -> torch.Tensor:
    """softmax(scale * a @ w.T) over whole rows as bf16 [M, N] (columns >= valid_cols: 0), in two passes of the same GEMM:
    pass 1 leaves only per-tile (max, sum) statistics, pass 2 recomputes the tile and writes the probabilities — the fp32
    score matrix never travels through HBM (6 B per score in the three-kernel form, 2 B here)."""
    _req(w, bf16, "gemm_row_softmax.w")
    _req(a, bf16, "gemm_row_softmax.a")
    K, N = a.shape[-1], w.shape[0]
    a2 = a.reshape(-1, K)
    if a2.stride(-1) != 1:
        a2 = a2.contiguous()
    M, lda = a2.shape[0], a2.stride(0)
    parts = -(-N // gemm_n_tile(M, N, K))
    stats = torch.empty(parts, M, 2, dtype=torch.float32, device=a.device)
    out = torch.empty(M, N, dtype=bf16, device=a.device)
    lib = _lib.load()
    folded = torch.empty(M, 2, dtype=torch.float32, device=a.device) if parts > 1 else stats
    for which in (1, 2):
        e = _epilogue(out, N, None, None, 0, None, 0, False, False, float(scale) * 1.4426950408889634, 0, 0, 0, 0, w_dynamic)
        e.row_softmax, e.row_softmax_valid = which, int(valid_cols) if valid_cols is not None else N
        if which == 1:
            e.out, e.ln_stats_out = None, stats.data_ptr()
        else:
            if parts > 1:
                check(lib.b200sr_row_softmax_fold(stats.data_ptr(), parts, M, folded.data_ptr(), _stream()), "row_softmax_fold")
            e.ln_stats, e.ln_parts = folded.data_ptr(), 1
        with _Timed("gemm", 2.0 * M * N * K, f"M{M} N{N} K{K} row softmax pass {which}"):
            rc = lib.b200sr_gemm_bf16(a2.data_ptr(), lda, w.data_ptr(), M, N, K, C.byref(e), 0, _stream())
        check(rc, f"gemm_row_softmax pass {which} M={M} N={N} K={K}")
    return out


TWO_PASS_SOFTMAX = True   # single_head_attention: scores recomputed instead of stored (False: score GEMM -> softmax_rows)


def single_head_attention(q: torch.Tensor, k: torch.Tensor, v_t: torch.Tensor, scale: float,
                          out_bias: Optional[torch.Tensor] = None, valid_keys: Optional[int] = None) -> torch.Tensor:
    """softmax(q k^T * scale) v for ONE head of width C = 512 (SR3 SelfAttention, sr3_modules/unet.py:114-143; the
    first stage's AttnBlock, sgm/modules/diffusionmodules/model.py:158-199).  q, k: [T, C] bf16; v_t: [C, Tk] bf16
    (V transposed = the B operand of P V); returns [T, C] bf16 (+ out_bias[C]).

    The output accumulator of a 128-row tile at C = 512 fills all 512 TMEM columns, which leaves no room for the score
    tile, so this shape runs as score GEMM -> row softmax -> P V GEMM over query chunks sized to keep the fp32 scores
    within SCORE_CHUNK_BYTES (never the T x T matrix: 17 GB at T = 65536)."""
    t, c = q.shape
    tk = k.shape[0]
    two_pass = TWO_PASS_SOFTMAX and tk % 8 == 0
    rows = (SCORE_CHUNK_BYTES // ((2 if two_pass else 4) * tk)) // 256 * 256
    rows = max(256, min(rows, t))
    out = torch.empty(t, c, dtype=bf16, device=q.device)
    for r0 in range(0, t, rows):
        r1 = min(t, r0 + rows)
        if two_pass:
            p = gemm_row_softmax(q[r0:r1], k, scale, valid_keys)                    # [rows, Tk] bf16 probabilities
        else:
            s = gemm(q[r0:r1], k, out_fp32=True, w_dynamic=True)                    # [rows, Tk] fp32 scores
            p = softmax_rows(s, scale, valid_cols=valid_keys)
        gemm(p, v_t, out_bias, w_dynamic=True, out=out[r0:r1])
    return out


# ------------------------------------------------------------------------------------------------
# layout / elementwise
# ------------------------------------------------------------------------------------------------
def nchw_to_nhwc_bf16(x: torch.Tensor, scale: float = 1.0) -> torch.Tensor:
    """[N, C, H, W] fp32 -> [N, H, W, C] bf16 (times `scale`)."""
    _req(x, torch.float32, "nchw_to_nhwc.x")
    n, c, h, w = x.shape
    y = torch.empty(n, h, w, c, dtype=bf16, device=x.device)
    check(_lib.load().b200sr_nchw_f32_to_nhwc_bf16(x.data_ptr(), y.data_ptr(), n, c, h * w, float(scale), _stream()),
          "nchw_to_nhwc")
    return y


def cast_bf16(x: torch.Tensor) -> torch.Tensor:
    """fp32 -> bf16 of an arbitrary contiguous tensor (conditioning vectors, context tokens)."""
    if x.dtype == bf16:
        return x if x.is_contiguous() else x.contiguous()
    _req(x, torch.float32, "cast_bf16.x")
    y = torch.empty(x.shape, dtype=bf16, device=x.device)
    check(_lib.load().b200sr_nchw_f32_to_nhwc_bf16(x.data_ptr(), y.data_ptr(), 1, 1, x.numel(), 1.0, _stream()),
          "cast_bf16")
    return y


def nhwc_to_nchw_f32(x: torch.Tensor) -> torch.Tensor:
    _req(x, bf16, "nhwc_to_nchw.x")
    n, h, w, c = x.shape
    y = torch.empty(n, c, h, w, dtype=torch.float32, device=x.device)
    check(_lib.load().b200sr_nhwc_bf16_to_nchw_f32(x.data_ptr(), y.data_ptr(), n, c, h * w, _stream()), "nhwc_to_nchw")
    return y


def pack_conv3x3_few_out(weight: torch.Tensor, bias: Optional[torch.Tensor]):
    """[Cout <= 4, Cin, 3, 3] (+ bias) -> packed bf16 [8, 9*Cin] / fp32 [8]: output channels zero-padded to 8 so the
    convolution runs on the tcgen05 path (the direct warp-per-pixel kernel is 10-50x slower at 128^2 .. 1024^2)."""
    co = weight.shape[0]
    w = torch.zeros(8, *weight.shape[1:], dtype=weight.dtype, device=weight.device)
    w[:co] = weight.detach()
    b = torch.zeros(8, dtype=torch.float32, device=weight.device)
    if bias is not None:
        b[:co] = bias.detach().float()
    return pack_conv3x3(w), b


def conv3x3_to_nchw_f32(x: torch.Tensor, w8: torch.Tensor, b8: torch.Tensor, cout: int) -> torch.Tensor:
    """3x3 conv (pad 1) to `cout` <= 4 channels, returned as fp32 NCHW: tensor-core conv with the output padded to 8
    channels (bf16, the reference's autocast output dtype), then the first `cout` channels converted."""
    y8 = conv3x3(x, w8, b8)
    n, h, wd, cs = y8.shape
    out = torch.empty(n, cout, h, wd, dtype=torch.float32, device=x.device)
    check(_lib.load().b200sr_nhwc_bf16_to_nchw_f32_strided(y8.data_ptr(), out.data_ptr(), n, cout, cs, h * wd, _stream()),
          "nhwc_to_nchw_strided")
    return out


def upsample2x(x: torch.Tensor) -> torch.Tensor:
    _req(x, bf16, "upsample2x.x")
    n, h, w, c = x.shape
    y = torch.empty(n, 2 * h, 2 * w, c, dtype=bf16, device=x.device)
    check(_lib.load().b200sr_upsample2x_nhwc(x.data_ptr(), y.data_ptr(), n, h, w, c, _stream()), "upsample2x")
    return y


def concat_add(a: Optional[torch.Tensor], b: torch.Tensor, c: Optional[torch.Tensor] = None) -> torch.Tensor:
    """cat([a, b (+ c)], channel dim) for channels-last bf16 tensors."""
    _req(b, bf16, "concat_add.b")
    ca = 0 if a is None else a.shape[-1]
    cb = b.shape[-1]
    rows = b.numel() // cb
    out = torch.empty(*b.shape[:-1], ca + cb, dtype=bf16, device=b.device)
    check(_lib.load().b200sr_concat_add(_ptr(a), ca, b.data_ptr(), cb, _ptr(c), out.data_ptr(), rows, _stream()),
          "concat_add")
    return out


def axpy(a: torch.Tensor, b: torch.Tensor, alpha: float = 1.0) -> torch.Tensor:
    _req(a, bf16, "axpy.a")
    _req(b, bf16, "axpy.b")
    y = torch.empty_like(a)
    check(_lib.load().b200sr_axpy_bf16(a.data_ptr(), b.data_ptr(), y.data_ptr(), float(alpha), a.numel(), _stream()),
          "axpy")
    return y


def pad_channels(x: torch.Tensor, cpad: int) -> torch.Tensor:
    """[..., C] bf16 -> [..., cpad] bf16 with zero fill."""
    _req(x, bf16, "pad_channels.x")
    c = x.shape[-1]
    y = torch.empty(*x.shape[:-1], cpad, dtype=bf16, device=x.device)
    check(_lib.load().b200sr_pad_channels(x.data_ptr(), y.data_ptr(), c, cpad, x.numel() // c, _stream()), "pad_channels")
    return y


def pack_conv3x3_padded(weight: torch.Tensor, cin_pad: int) -> torch.Tensor:
    """[Cout, Cin, 3, 3] -> bf16 [Cout, 9*cin_pad] (zero weights for the padded input channels)."""
    co, ci, kh, kw = weight.shape
    w = torch.zeros(co, 3, 3, cin_pad, dtype=weight.dtype, device=weight.device)
    w[..., :ci] = weight.detach().permute(0, 2, 3, 1)
    return w.reshape(co, 9 * cin_pad).to(bf16).contiguous()


def pointwise_small(x: torch.Tensor, w: torch.Tensor, bias: Optional[torch.Tensor], *, out_nchw_f32: bool = False,
                    scale: float = 1.0) -> torch.Tensor:
    """1x1 convolution between <= 8 channels: x bf16 [N, H, W, Cin], w fp32 [Cout, Cin] -> (w x + b) * scale as bf16
    [N, H, W, Cout] or fp32 [N, Cout, H, W]."""
    _req(x, bf16, "pointwise_small.x")
    n, h, wd, cin = x.shape
    cout = w.shape[0]
    y = (torch.empty(n, cout, h, wd, dtype=torch.float32, device=x.device) if out_nchw_f32
         else torch.empty(n, h, wd, cout, dtype=bf16, device=x.device))
    check(_lib.load().b200sr_pointwise_small(x.data_ptr(), w.data_ptr(), _ptr(bias), y.data_ptr(), cin, cout, n * h * wd,
                                             h * wd, int(out_nchw_f32), float(scale), _stream()), "pointwise_small")
    return y


def diag_gaussian(moments: torch.Tensor, noise: Optional[torch.Tensor], scale: float = 1.0) -> torch.Tensor:
    """moments fp32 [N, 2C, H, W] -> (mean + exp(clamp(logvar) / 2) * noise) * scale (noise None: the mode)."""
    _req(moments, torch.float32, "diag_gaussian.moments")
    n, c2, h, w = moments.shape
    z = torch.empty(n, c2 // 2, h, w, dtype=torch.float32, device=moments.device)
    check(_lib.load().b200sr_diag_gaussian(moments.data_ptr(), _ptr(noise), z.data_ptr(), n, c2 // 2, h * w, float(scale),
                                           _stream()), "diag_gaussian")
    return z


def silu(x: torch.Tensor) -> torch.Tensor:
    _req(x, bf16, "silu.x")
    y = torch.empty_like(x)
    check(_lib.load().b200sr_silu_bf16(x.data_ptr(), y.data_ptr(), x.numel(), _stream()), "silu")
    return y


def embed_tokens(ids: torch.Tensor, tok: torch.Tensor, pos: torch.Tensor) -> torch.Tensor:
    """tok[ids] + pos: ids int64 [B, T], tok fp32 [vocab, C], pos fp32 [T, C] -> bf16 [B, T, C]."""
    _req(ids, torch.int64, "embed_tokens.ids")
    _req(tok, torch.float32, "embed_tokens.tok")
    _req(pos, torch.float32, "embed_tokens.pos")
    b, t = ids.shape
    c = tok.shape[1]
    out = torch.empty(b, t, c, dtype=bf16, device=ids.device)
    check(_lib.load().b200sr_embed_tokens(ids.data_ptr(), tok.data_ptr(), pos.data_ptr(), out.data_ptr(), b, t, c, tok.shape[0],
                                          _stream()), "embed_tokens")
    return out


def sinusoid_embedding(t: torch.Tensor, dim: int, max_period: float = 10000.0, sin_first: bool = False) -> torch.Tensor:
    t = t.reshape(-1).to(torch.float32).contiguous()
    if not t.is_cuda:
        raise _lib.B200SRError("sinusoid_embedding: expected a CUDA tensor")
    out = torch.empty(t.numel(), dim, dtype=bf16, device=t.device)
    check(_lib.load().b200sr_sinusoid_embedding(t.data_ptr(), out.data_ptr(), t.numel(), dim, float(max_period),
                                                int(sin_first), _stream()), "sinusoid_embedding")
    return out


# ------------------------------------------------------------------------------------------------
# sampler-side kernels
# ------------------------------------------------------------------------------------------------
def sampler_pre(x: torch.Tensor, noise: Optional[torch.Tensor], scalars: torch.Tensor, cfg_copies: int = 2):
    """Returns (x_hat fp32 NCHW, net_in bf16 NHWC [cfg_copies*B, H, W, C])."""
    _req(x, torch.float32, "sampler_pre.x")
    b, c, h, w = x.shape
    x_hat = torch.empty_like(x)
    net_in = torch.empty(cfg_copies * b, h, w, c, dtype=bf16, device=x.device)
    check(_lib.load().b200sr_sampler_pre(x.data_ptr(), _ptr(noise), scalars.data_ptr(), x_hat.data_ptr(),
                                         net_in.data_ptr(), b, c, h * w, cfg_copies, _stream()), "sampler_pre")
    return x_hat, net_in


def sampler_post(eps: torch.Tensor, x_hat: torch.Tensor, scalars: torch.Tensor, use_cfg: bool = True,
                 want_denoised: bool = True):
    """eps: fp32 NCHW [2B or B, C, H, W].  Returns (x_next, denoised)."""
    _req(eps, torch.float32, "sampler_post.eps")
    b, c, h, w = x_hat.shape
    x_next = torch.empty_like(x_hat)
    den = torch.empty_like(x_hat) if want_denoised else None
    check(_lib.load().b200sr_sampler_post(eps.data_ptr(), x_hat.data_ptr(), scalars.data_ptr(), _ptr(den),
                                          x_next.data_ptr(), b, c, h * w, int(use_cfg), _stream()), "sampler_post")
    return x_next, den


def euler_from_denoised(denoised: torch.Tensor, x_hat: torch.Tensor, scalars: torch.Tensor) -> torch.Tensor:
    x_next = torch.empty_like(x_hat)
    check(_lib.load().b200sr_euler_from_denoised(denoised.data_ptr(), x_hat.data_ptr(), scalars.data_ptr(),
                                                 x_next.data_ptr(), x_hat.numel(), _stream()), "euler_from_denoised")
    return x_next


def tile_accumulate(tile: torch.Tensor, weight: torch.Tensor, acc: torch.Tensor, cnt: Optional[torch.Tensor], h0: int,
                    w0: int):
    """acc[win] += tile * weight (product and sum rounded separately); cnt[win] += weight unless cnt is None."""
    b, c, th, tw = tile.shape
    H, W = acc.shape[-2:]
    check(_lib.load().b200sr_tile_accumulate(tile.data_ptr(), weight.data_ptr(), acc.data_ptr(), _ptr(cnt), b * c,
                                             th, tw, H, W, h0, w0, _stream()), "tile_accumulate")


def tile_weighted_strip(tile: torch.Tensor, weight: torch.Tensor, y0: int, x0: int, sh: int, sw: int,
                        out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """(tile * weight)[:, :, y0:y0+sh, x0:x0+sw] packed contiguously (fp32): what a peer rank's overlapping window needs."""
    _req(tile, torch.float32, "tile_weighted_strip.tile")
    b, c, th, tw = tile.shape
    if out is None:
        out = torch.empty(b, c, sh, sw, dtype=torch.float32, device=tile.device)
    check(_lib.load().b200sr_tile_weighted_strip(tile.data_ptr(), weight.data_ptr(), out.data_ptr(), b * c, th, tw, y0, x0,
                                                 sh, sw, _stream()), "tile_weighted_strip")
    return out


def strip_add(strip: torch.Tensor, acc: torch.Tensor, h0: int, w0: int) -> None:
    """acc[:, :, h0:h0+sh, w0:w0+sw] += strip (fp32, contiguous strip [B, C, sh, sw])."""
    _req(strip, torch.float32, "strip_add.strip")
    b, c, sh, sw = strip.shape
    H, W = acc.shape[-2:]
    check(_lib.load().b200sr_strip_add(strip.data_ptr(), acc.data_ptr(), b * c, sh, sw, H, W, h0, w0, _stream()),
          "strip_add")


def copy_batch(pairs) -> None:
    """Up to 8 (dst, src) copies between contiguous device tensors of equal byte size in ONE kernel launch."""
    n = len(pairs)
    arr = (_lib.Copy * n)()
    for i, (dst, src) in enumerate(pairs):
        nb = src.numel() * src.element_size()
        if not (dst.is_cuda and src.is_cuda and dst.is_contiguous() and src.is_contiguous()) or \
                dst.numel() * dst.element_size() != nb:
            raise _lib.B200SRError("copy_batch: contiguous CUDA tensors of equal byte size expected")
        arr[i].src, arr[i].dst, arr[i].bytes = src.data_ptr(), dst.data_ptr(), nb
    check(_lib.load().b200sr_copy_batch(arr, n, _stream()), "copy_batch")


def tile_normalize(acc: torch.Tensor, cnt: torch.Tensor) -> torch.Tensor:
    out = torch.empty_like(acc)
    check(_lib.load().b200sr_tile_normalize(acc.data_ptr(), cnt.data_ptr(), out.data_ptr(), acc.numel(), _stream()),
          "tile_normalize")
    return out


_rel_ws: dict = {}


def rel_l1_similarity(prev: torch.Tensor, cur: torch.Tensor, threshold: torch.Tensor) -> torch.Tensor:
    """Returns a device fp32[2]: (diff, diff < threshold) — DFBCache.are_two_tensors_similar."""
    _req(prev, bf16, "rel_l1.prev")
    _req(cur, bf16, "rel_l1.cur")
    key = (prev.device.type, prev.device.index, _ws_slot[0])
    ws = _rel_ws.get(key)
    if ws is None:
        ws = torch.zeros(2, dtype=torch.float64, device=prev.device)
        _rel_ws[key] = ws
    res = torch.empty(2, dtype=torch.float32, device=prev.device)
    check(_lib.load().b200sr_rel_l1_similarity(prev.data_ptr(), cur.data_ptr(), prev.numel(), threshold.data_ptr(),
                                               ws.data_ptr(), res.data_ptr(), _stream()), "rel_l1_similarity", kernels=2)
    return res


def sr3_update(x: torch.Tensor, eps: torch.Tensor, noise: Optional[torch.Tensor], scalars: torch.Tensor) -> torch.Tensor:
    out = torch.empty_like(x)
    check(_lib.load().b200sr_sr3_update(x.data_ptr(), eps.data_ptr(), _ptr(noise), scalars.data_ptr(), out.data_ptr(),
                                        x.numel(), _stream()), "sr3_update")
    return out


# ------------------------------------------------------------------------------------------------
# output side: wavelet colour fix, Tensor2PIL
# ------------------------------------------------------------------------------------------------
def wavelet_level(img: torch.Tensor, radius: int, high: Optional[torch.Tensor] = None, first: bool = False) -> torch.Tensor:
    """One level of wavelet_decomposition (utils/colorfix.py:73-106): returns low = blur(img, radius); `high`
    (optional, in place) accumulates img - low."""
    _req(img, torch.float32, "wavelet_level.img")
    b, c, h, w = img.shape
    low = torch.empty_like(img)
    check(_lib.load().b200sr_wavelet_level(img.data_ptr(), low.data_ptr(), _ptr(high), int(first), b * c, h, w, int(radius),
                                           _stream()), "wavelet_level")
    return low


def add_f32(a: torch.Tensor, b: torch.Tensor) -> torch.Tensor:
    _req(a, torch.float32, "add_f32.a")
    _req(b, torch.float32, "add_f32.b")
    out = torch.empty_like(a)
    check(_lib.load().b200sr_add_f32(a.data_ptr(), b.data_ptr(), out.data_ptr(), a.numel(), _stream()), "add_f32")
    return out


def image_to_u8(x: torch.Tensor, oh: int, ow: int) -> torch.Tensor:
    """fp32 [C, H, W] in [-1, 1] -> uint8 [oh, ow, C] (bicubic resize, *127.5 + 127.5, clip, truncate)."""
    _req(x, torch.float32, "image_to_u8.x")
    c, h, w = x.shape
    out = torch.empty(oh, ow, c, dtype=torch.uint8, device=x.device)
    check(_lib.load().b200sr_image_to_u8(x.data_ptr(), out.data_ptr(), c, h, w, oh, ow, _stream()), "image_to_u8")
    return out


# ------------------------------------------------------------------------------------------------
# stage-1 -> stage-2 hand-off: tensor2img, PIL2Tensor's Image.resize(BICUBIC) and uint8 -> [-1, 1]
# ------------------------------------------------------------------------------------------------
PILLOW_PRECISION_BITS = 22


def _pillow_bicubic(x):
    """libImaging/Resample.c bicubic_filter (a = -0.5, support 2), float64, same operation order."""
    a = -0.5
    x = np.abs(x)
    near = ((a + 2.0) * x - (a + 3.0)) * x * x + 1
    far = (((x - 5) * x + 8) * x - 4) * a
    return np.where(x < 1.0, near, np.where(x < 2.0, far, 0.0))


def pillow_bicubic_tables(in_len: int, out_len: int):
    """Pillow's precompute_coeffs + normalize_coeffs_8bpc (libImaging/Resample.c) for one axis of
    ``Image.resize(..., Image.BICUBIC)`` over the whole image (box = (0, in_len)), as numpy arrays:
    (bounds int32 [out_len, 2] = (first tap, tap count), coeffs int32 [out_len, ksize], ksize).

    Per output index o: center = (o + 0.5) * scale with scale = in / out; the filter is stretched by
    fs = max(scale, 1) (antialiasing when reducing); taps xmin .. xmin + n - 1 with xmin = int(center - support + 0.5)
    and support = 2 * fs; w_k = filter((k + xmin - center + 0.5) * (1 / fs)), divided by their sequential double sum
    (unless it is 0); the fixed-point coefficient is w * 2^22 rounded half away from zero."""
    if in_len <= 0 or out_len <= 0:
        raise ValueError(f"resample lengths must be positive, got {in_len} -> {out_len}")
    scale = float(in_len) / out_len
    fs = max(scale, 1.0)
    support = 2.0 * fs
    ksize = int(math.ceil(support)) * 2 + 1
    center = (np.arange(out_len, dtype=np.float64) + 0.5) * scale
    xmin = np.maximum((center - support + 0.5).astype(np.int64), 0)           # C (int) cast: toward zero
    xmax = np.minimum((center + support + 0.5).astype(np.int64), in_len)
    n = xmax - xmin
    k = np.arange(ksize, dtype=np.int64)
    pos = (k[None, :] + xmin[:, None]).astype(np.float64)
    w = _pillow_bicubic((pos - center[:, None] + 0.5) * (1.0 / fs))
    w = np.where(k[None, :] < n[:, None], w, 0.0)
    ww = np.zeros(out_len, dtype=np.float64)
    for j in range(ksize):                                                      # sequential sum, as the C loop
        ww = ww + w[:, j]
    w = np.where(ww[:, None] != 0.0, w / np.where(ww == 0.0, 1.0, ww)[:, None], w)
    one = float(1 << PILLOW_PRECISION_BITS)
    fixed = np.where(w < 0, (-0.5 + w * one).astype(np.int64), (0.5 + w * one).astype(np.int64))
    bounds = np.stack((xmin, n), 1).astype(np.int32)
    return bounds, fixed.astype(np.int32), ksize


_resample_tables: dict = {}


def _device_tables(in_len: int, out_len: int, device: torch.device):
    key = (in_len, out_len, device.type, device.index)
    t = _resample_tables.get(key)
    if t is None:
        bounds, coeffs, ksize = pillow_bicubic_tables(in_len, out_len)
        t = (torch.from_numpy(bounds).to(device), torch.from_numpy(coeffs).to(device), ksize)
        _resample_tables[key] = t
    return t


def tensor2img_u8(x: torch.Tensor) -> torch.Tensor:
    """fp32 [C, H, W] in [-1, 1] -> uint8 [H, W, C]: rint((clamp(x, -1, 1) + 1) / 2 * 255) in fp32."""
    _req(x, torch.float32, "tensor2img_u8.x")
    c, h, w = x.shape
    out = torch.empty(h, w, c, dtype=torch.uint8, device=x.device)
    check(_lib.load().b200sr_tensor2img_u8(x.data_ptr(), out.data_ptr(), c, h, w, _stream()), "tensor2img_u8")
    return out


def resample_u8_axis(src: torch.Tensor, out_len: int, axis: int, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """One Pillow bicubic pass of a uint8 [H, W, C] image along axis 1 (width) or 0 (height).  `out` (optional) is
    the destination; its shape must be the result's."""
    _req(src, torch.uint8, "resample_u8.src")
    h, w, c = src.shape
    if axis == 1:
        outer, in_len, inner, shape = h, w, c, (h, out_len, c)
    elif axis == 0:
        outer, in_len, inner, shape = 1, h, w * c, (out_len, w, c)
    else:
        raise ValueError("axis must be 0 (height) or 1 (width)")
    if out is None:
        out = torch.empty(shape, dtype=torch.uint8, device=src.device)
    elif tuple(out.shape) != shape:
        raise ValueError(f"resample_u8: out has shape {tuple(out.shape)}, expected {shape}")
    _req(out, torch.uint8, "resample_u8.out")
    bounds, coeffs, ksize = _device_tables(in_len, out_len, src.device)
    check(_lib.load().b200sr_resample_u8(src.data_ptr(), out.data_ptr(), outer, in_len, out_len, inner,
                                         bounds.data_ptr(), coeffs.data_ptr(), ksize, _stream()), "resample_u8")
    return out


def resize_bicubic_u8(img: torch.Tensor, oh: int, ow: int) -> torch.Tensor:
    """``PIL.Image.fromarray(img).resize((ow, oh), Image.BICUBIC)`` of a uint8 [H, W, C] image, byte for byte: the
    horizontal pass first (when the width changes), then the vertical pass (when the height changes); an unchanged
    size is a copy."""
    _req(img, torch.uint8, "resize_bicubic_u8.img")
    h, w, _ = img.shape
    if ow != w:
        img = resample_u8_axis(img, ow, 1)
    if oh != h:
        img = resample_u8_axis(img, oh, 0)
    return img.clone() if (oh, ow) == (h, w) else img


def img_u8_to_tensor(img: torch.Tensor) -> torch.Tensor:
    """uint8 [H, W, C] -> fp32 [C, H, W]: (float)(x / 255 * 2 - 1) computed in double."""
    _req(img, torch.uint8, "img_u8_to_tensor.img")
    h, w, c = img.shape
    out = torch.empty(c, h, w, dtype=torch.float32, device=img.device)
    check(_lib.load().b200sr_img_u8_to_tensor(img.data_ptr(), out.data_ptr(), c, h, w, _stream()), "img_u8_to_tensor")
    return out
