"""Drop-in stage-2 denoiser modules: same constructor arguments, ``forward`` signatures and
``state_dict`` keys as the reference classes, with the compute routed to the sm_100a kernels.

Mirrored reference classes (file:line relative to the reference root):
  TimestepBlock / TimestepEmbedSequential   sgm/modules/diffusionmodules/openaimodel.py:63-99
  Upsample / Downsample / ResBlock          openaimodel.py:102-145, :164-204, :207-350
  UNetModel                                 openaimodel.py:500-1007
  GEGLU / FeedForward / CrossAttention      sgm/modules/attention.py:84-110, :196-285
  BasicTransformerBlock / SpatialTransformer  attention.py:376-486, :533-635
  ZeroSFT / ZeroCrossAttn / GLVControl / LightGLVUNet   models/modules/SR_modules.py:59-149, :152-537, :540-883
  ControlWrapper                            sgm/modules/diffusionmodules/wrappers.py:68-110

Tensor convention at every public ``forward``: images are NCHW-*shaped* tensors.  fp32 / arbitrary
inputs are converted once; everything these modules return is a bf16 tensor whose memory is
channels-last (``y.permute(0, 2, 3, 1)`` is contiguous), so chained modules exchange NHWC views
without copies, while any torch consumer still sees an ordinary ``[N, C, H, W]`` tensor.  Tokens
are ``[B, T, C]`` bf16.  Parameters remain ordinary fp32 ``nn.Parameter``s under the reference's
names; bf16 K-major copies for the tensor cores are packed lazily and re-packed when a parameter
changes (``load_state_dict`` / ``.to()``).

Numerics follow the reference's autocast policy (SURVEY.md section 3.4): bf16 operands, fp32
accumulation, fp32 normalisation statistics and softmax; activations are stored in bf16.
"""
from __future__ import annotations

from typing import Dict, List, Optional

import torch
import torch.nn as nn

from . import ops

bf16 = torch.bfloat16


# ------------------------------------------------------------------------------------------------
# helpers
# ------------------------------------------------------------------------------------------------
def exists(x):
    return x is not None


def zero_module(module: nn.Module) -> nn.Module:
    """util.py:233-239."""
    for p in module.parameters():
        p.detach().zero_()
    return module


def to_nhwc(x: torch.Tensor) -> torch.Tensor:
    """NCHW-shaped tensor -> contiguous [N, H, W, C] bf16 (zero-copy for our own outputs)."""
    if x.dim() != 4:
        raise ValueError(f"expected a 4-D NCHW tensor, got {tuple(x.shape)}")
    v = x.permute(0, 2, 3, 1)
    if x.dtype == bf16 and v.is_contiguous():
        return v
    if x.dtype == torch.float32 and x.is_contiguous():
        return ops.nchw_to_nhwc_bf16(x)
    return v.to(bf16).contiguous()  # exotic layouts / dtypes: plain layout plumbing


def from_nhwc(y: torch.Tensor) -> torch.Tensor:
    return y.permute(0, 3, 1, 2)


def tokens_bf16(x: torch.Tensor) -> torch.Tensor:
    if x.dtype == bf16 and x.is_contiguous():
        return x
    if x.dtype == torch.float32:
        return ops.cast_bf16(x.contiguous())
    return x.to(bf16).contiguous()


class Packed:
    """Mixin: lazily packed (bf16 / fused) copies of parameters, invalidated when they change."""

    def _pk(self, name: str, params, fn):
        cache = self.__dict__.setdefault("_pk_cache", {})
        key = tuple((p.data_ptr(), p._version, str(p.device)) for p in params)
        hit = cache.get(name)
        if hit is None or hit[0] != key:
            with torch.no_grad():
                hit = (key, fn(*params))
            cache[name] = hit
        return hit[1]


_F32 = lambda p: p.detach().float().contiguous()  # noqa: E731


def _silu_of(emb: torch.Tensor) -> torch.Tensor:
    """SiLU(emb), shared by every ResBlock of one forward (openaimodel.py:281-283)."""
    # The result rides on the emb tensor *object* (never keyed by address: the caching allocator
    # hands the same address to the next step's emb).
    s = getattr(emb, "_b200sr_silu", None)
    if s is None:
        s = ops.silu(tokens_bf16(emb))
        try:
            emb._b200sr_silu = s
        except Exception:  # pragma: no cover - exotic tensor subclasses
            pass
    return s


class EmbSlot:
    """Stand-in for the `emb` argument when every ResBlock's projection of it is already known (the engine
    precomputes them for all sampler steps): only carries the per-block table ``_b200sr_rb``."""

    def __init__(self, table):
        self._b200sr_rb = table


def _resblocks_of(root: nn.Module):
    blocks = root.__dict__.get("_b200sr_resblocks")
    if blocks is None:
        blocks = [m for m in root.modules() if isinstance(m, ResBlock)]
        root.__dict__["_b200sr_resblocks"] = blocks
    return blocks


def rb_table(root: nn.Module, proj: torch.Tensor):
    """proj: fp32 [B, sum Cout] (row stride arbitrary) -> {id(ResBlock): its [B, Cout] column window}."""
    table, off = {}, 0
    for blk in _resblocks_of(root):
        table[id(blk)] = proj[:, off:off + blk.out_channels]
        off += blk.out_channels
    return table


def _project_emb_for_resblocks(holder: Packed, root: nn.Module, emb: torch.Tensor) -> Optional[torch.Tensor]:
    """Every ResBlock applies its own Linear to the same SiLU(emb) (openaimodel.py:281-283, :337-341).
    They only depend on emb, so all of a network's projections run as ONE GEMM against the row-wise
    concatenation of the weights right after emb is known; each block then reads its column window
    (fp32 [B, sum Cout], consumed through ``ld_rowvec``) instead of launching an M = B GEMM of its own.
    Returns the [B, sum Cout] projection (also attached to `emb` as a per-block table)."""
    blocks = _resblocks_of(root)
    if not blocks:
        return None
    params = tuple(p for blk in blocks for p in (blk.emb_layers[1].weight, blk.emb_layers[1].bias))
    w_all, b_all = holder._pk("rb_emb", params, lambda *ps: (
        torch.cat([ops.pack_linear(w) for w in ps[0::2]], 0).contiguous(),
        torch.cat([_F32(b) for b in ps[1::2]], 0).contiguous()))
    proj = ops.gemm(_silu_of(emb), w_all, b_all, out_fp32=True)  # [B, sum Cout]
    try:
        emb._b200sr_rb = rb_table(root, proj)
        emb._b200sr_proj = proj
    except Exception:  # pragma: no cover - exotic tensor subclasses
        pass
    return proj


def timestep_embedding(timesteps: torch.Tensor, dim: int, max_period: float = 10000.0) -> torch.Tensor:
    """util.py:206-230 (cos | sin); returns bf16 [B, dim]."""
    return ops.sinusoid_embedding(timesteps, dim, max_period, sin_first=False)


class GroupNorm32(nn.GroupNorm):
    """util.py:258-276 — parameter container; the fused kernel is invoked by the owning block."""


def normalization(channels: int) -> nn.GroupNorm:
    return GroupNorm32(32, channels)


def _gn(norm: nn.GroupNorm, x_nhwc: torch.Tensor, silu: bool = False, **kw) -> torch.Tensor:
    return ops.group_norm(x_nhwc, norm.weight, norm.bias, groups=norm.num_groups, eps=norm.eps, silu=silu, **kw)


def _conv3x3(holder: Packed, name: str, conv: nn.Conv2d, x_nhwc: torch.Tensor, **kw) -> torch.Tensor:
    w = holder._pk(name + ".w", (conv.weight,), ops.pack_conv3x3)
    b = holder._pk(name + ".b", (conv.bias,), _F32) if conv.bias is not None else None
    return ops.conv3x3(x_nhwc, w, b, **kw)


def _gn_silu_conv3x3(holder: Packed, name: str, norm: nn.GroupNorm, conv: nn.Conv2d, x_nhwc: torch.Tensor, **kw) -> torch.Tensor:
    """conv3x3(SiLU(GroupNorm(x))) (openaimodel.py:254-258, :289-300; model.py:127-141; sr3 unet.py:81-92).  Where the
    halo-path convolution applies (stride 1, W % 8 == 0, H >= 16) and the output fits one N tile (<= 256 channels: the
    high-resolution levels of SR3 and of the first stage) only the statistics pass runs as a kernel of its own: the
    convolution normalises its input tiles in shared memory.  Same arithmetic, same bf16 rounding point, so the result
    equals the two-kernel form bit for bit."""
    if ops.conv3x3_gn_fusable(x_nhwc, 1, conv.out_channels) and norm.affine:
        stats = ops.group_norm_stats(x_nhwc, norm.num_groups, norm.eps)
        return _conv3x3(holder, name, conv, x_nhwc, gn=(stats, norm.weight, norm.bias, norm.num_groups, True), **kw)
    return _conv3x3(holder, name, conv, _gn(norm, x_nhwc, silu=True), **kw)


def _linear(holder: Packed, name: str, lin, x: torch.Tensor, **kw) -> torch.Tensor:
    w = holder._pk(name + ".w", (lin.weight,), ops.pack_linear)
    b = holder._pk(name + ".b", (lin.bias,), _F32) if lin.bias is not None else None
    return ops.gemm(x, w, b, **kw)


# ------------------------------------------------------------------------------------------------
# openaimodel.py blocks
# ------------------------------------------------------------------------------------------------
class TimestepBlock(nn.Module):
    """openaimodel.py:63-72."""


class Upsample(nn.Module, Packed):
    """openaimodel.py:102-145: nearest x2 (+ 3x3 conv)."""

    def __init__(self, channels, use_conv, dims=2, out_channels=None, padding=1, third_up=False):
        super().__init__()
        assert dims == 2 and padding == 1
        self.channels, self.out_channels, self.use_conv, self.dims = channels, out_channels or channels, use_conv, dims
        if use_conv:
            self.conv = nn.Conv2d(self.channels, self.out_channels, 3, padding=padding)

    def forward_nhwc(self, x):
        assert x.shape[-1] == self.channels
        x = ops.upsample2x(x)
        return _conv3x3(self, "conv", self.conv, x) if self.use_conv else x

    def forward(self, x):
        return from_nhwc(self.forward_nhwc(to_nhwc(x)))


class Downsample(nn.Module, Packed):
    """openaimodel.py:164-204: 3x3 conv, stride 2, pad 1."""

    def __init__(self, channels, use_conv, dims=2, out_channels=None, padding=1, third_down=False):
        super().__init__()
        assert dims == 2 and use_conv and padding == 1, "only the learned stride-2 convolution is on the hot path"
        self.channels, self.out_channels, self.use_conv, self.dims = channels, out_channels or channels, use_conv, dims
        self.op = nn.Conv2d(self.channels, self.out_channels, 3, stride=2, padding=padding)

    def forward_nhwc(self, x):
        assert x.shape[-1] == self.channels
        return _conv3x3(self, "op", self.op, x, stride=2)

    def forward(self, x):
        return from_nhwc(self.forward_nhwc(to_nhwc(x)))


class ResBlock(TimestepBlock, Packed):
    """openaimodel.py:207-350 (the configuration the YAML selects: no up/down, additive emb)."""

    def __init__(self, channels, emb_channels, dropout, out_channels=None, use_conv=False, use_scale_shift_norm=False,
                 dims=2, use_checkpoint=False, up=False, down=False, kernel_size=3, exchange_temb_dims=False,
                 skip_t_emb=False):
        super().__init__()
        assert dims == 2 and kernel_size == 3 and not (up or down or use_scale_shift_norm or skip_t_emb or use_conv)
        self.channels, self.emb_channels, self.dropout = channels, emb_channels, dropout
        self.out_channels = out_channels or channels
        self.use_checkpoint, self.use_scale_shift_norm = use_checkpoint, use_scale_shift_norm
        self.in_layers = nn.Sequential(normalization(channels), nn.SiLU(),
                                       nn.Conv2d(channels, self.out_channels, 3, padding=1))
        self.updown = False
        self.h_upd = self.x_upd = nn.Identity()
        self.emb_layers = nn.Sequential(nn.SiLU(), nn.Linear(emb_channels, self.out_channels))
        self.out_layers = nn.Sequential(normalization(self.out_channels), nn.SiLU(), nn.Dropout(p=dropout),
                                        zero_module(nn.Conv2d(self.out_channels, self.out_channels, 3, padding=1)))
        if self.out_channels == channels:
            self.skip_connection = nn.Identity()
        else:
            self.skip_connection = nn.Conv2d(channels, self.out_channels, 1)

    def forward_nhwc(self, x, emb):
        # emb add is fused into conv1's epilogue, the skip add into conv2's (openaimodel.py:337-350)
        pre = getattr(emb, "_b200sr_rb", None)
        emb_out = pre.get(id(self)) if pre is not None else None
        if emb_out is None:  # stand-alone use of the block
            emb_out = _linear(self, "emb", self.emb_layers[1], _silu_of(emb), out_fp32=True)
        h = _gn_silu_conv3x3(self, "conv1", self.in_layers[0], self.in_layers[2], x, rowvec=emb_out)
        skip = x if isinstance(self.skip_connection, nn.Identity) else _linear(self, "skip", self.skip_connection, x)
        return _gn_silu_conv3x3(self, "conv2", self.out_layers[0], self.out_layers[3], h, residual=skip)

    def forward(self, x, emb):
        return from_nhwc(self.forward_nhwc(to_nhwc(x), emb))


# ------------------------------------------------------------------------------------------------
# attention.py blocks
# ------------------------------------------------------------------------------------------------
class GEGLU(nn.Module, Packed):
    """attention.py:84-91; value * gelu(gate) fused into the projection's epilogue."""

    def __init__(self, dim_in, dim_out):
        super().__init__()
        self.proj = nn.Linear(dim_in, dim_out * 2)

    def forward(self, x, ln=None):
        """`ln` = (LayerNorm module, RowStats of x): x is the raw residual stream and the norm is folded into the GEMM."""
        if ln is not None:
            norm, stats = ln
            w, colsum, shift = self._pk("proj_ln", (self.proj.weight, self.proj.bias, norm.weight, norm.bias),
                                        ops.pack_geglu_ln)
            return ops.gemm(tokens_bf16(x), w, None, geglu=True, ln=(stats, colsum, shift, norm.eps))
        w, b = self._pk("proj", (self.proj.weight, self.proj.bias), ops.pack_geglu)
        return ops.gemm(tokens_bf16(x), w, b, geglu=True)


class FeedForward(nn.Module, Packed):
    """attention.py:94-110 (glu=True on this path)."""

    def __init__(self, dim, dim_out=None, mult=4, glu=False, dropout=0.0):
        super().__init__()
        assert glu, "only the gated feed-forward is on the hot path"
        inner_dim = int(dim * mult)
        dim_out = dim_out or dim
        self.net = nn.Sequential(GEGLU(dim, inner_dim), nn.Dropout(dropout), nn.Linear(inner_dim, dim_out))

    def forward(self, x, residual: Optional[torch.Tensor] = None, ln=None, want_stats: bool = False):
        return _linear(self, "out", self.net[2], self.net[0](x, ln=ln), residual=residual, want_stats=want_stats)


class CrossAttention(nn.Module, Packed):
    """attention.py:196-285: q/k/v without bias, heads of 64, SDPA scale 1/8, out Linear with bias.
    Self-attention runs one fused QKV GEMM whose output the attention kernel reads in place."""

    def __init__(self, query_dim, context_dim=None, heads=8, dim_head=64, dropout=0.0, backend=None):
        super().__init__()
        assert dim_head == 64, "the tcgen05 attention kernel is specialised for head_dim 64"
        inner_dim = dim_head * heads
        context_dim = context_dim or query_dim
        self.scale, self.heads = dim_head**-0.5, heads
        self.to_q = nn.Linear(query_dim, inner_dim, bias=False)
        self.to_k = nn.Linear(context_dim, inner_dim, bias=False)
        self.to_v = nn.Linear(context_dim, inner_dim, bias=False)
        self.to_out = nn.Sequential(nn.Linear(inner_dim, query_dim), nn.Dropout(dropout))
        self.backend = backend

    def attend(self, x, context=None, kv=None, ln=None):
        """x: [B, T, C] bf16 -> attention output before to_out, [B, T, inner].  `kv`: precomputed [B, Tk, 2*inner].
        `ln` (self-attention only) = (LayerNorm, RowStats of x): the norm is folded into the QKV GEMM."""
        inner = self.to_q.weight.shape[0]
        if context is None:
            if ln is not None:
                norm, stats = ln
                w, colsum, shift = self._pk(
                    "qkv_ln", (self.to_q.weight, self.to_k.weight, self.to_v.weight, norm.weight, norm.bias),
                    lambda q, k, v, g, b: ops.pack_linear_ln(torch.cat([q, k, v], 0), g, b))
                qkv = ops.gemm(x, w, ln=(stats, colsum, shift, norm.eps))
            else:
                w = self._pk("qkv", (self.to_q.weight, self.to_k.weight, self.to_v.weight),
                             lambda q, k, v: torch.cat([q, k, v], 0).to(bf16).contiguous())
                qkv = ops.gemm(x, w)
            return ops.attention(qkv, qkv, qkv, self.heads, q_col=0, k_col=inner, v_col=2 * inner, scale=self.scale)
        q = _linear(self, "q", self.to_q, x)
        bound = self._bound_entry(context)
        if kv is not None:
            pass
        elif bound is not None:
            kv = bound[1]  # hoisted by bind_static_context(): the text context is constant over the steps
        else:
            kv = ops.gemm(context, self._wkv())
        if kv.shape[0] != q.shape[0]:
            # a context shared by n latents per CFG half ([uncond; cond] captions of a batch of tiles): rows of q are
            # ordered [uncond x n; cond x n].  Only shapes that miss the folded path get here (tokens % 256 != 0).
            if q.shape[0] % kv.shape[0]:
                raise ValueError(f"context batch {kv.shape[0]} does not divide the query batch {q.shape[0]}")
            kv = kv.repeat_interleave(q.shape[0] // kv.shape[0], dim=0)
        return ops.attention(q, kv, kv, self.heads, q_col=0, k_col=0, v_col=inner, scale=self.scale)

    def _wkv(self):
        return self._pk("kv", (self.to_k.weight, self.to_v.weight), lambda k, v: torch.cat([k, v], 0).to(bf16).contiguous())

    def _fold_norm(self) -> Optional[nn.LayerNorm]:
        """The LayerNorm in front of this attention (set by BasicTransformerBlock), folded into the bound keys; None
        when there is none."""
        return self.__dict__.get("_pre_norm")

    def _weights_key(self):
        ps = [self.to_q.weight, self.to_k.weight, self.to_v.weight, self.to_out[0].weight]
        norm = self._fold_norm()
        if norm is not None:
            ps += [norm.weight, norm.bias]
        return tuple((p.data_ptr(), p._version) for p in ps)

    def _bound_entry(self, context):
        """The (context, kv, folded, weights_key) entry bound for this very tensor object, or None.  An entry made
        from projection weights that have changed since (load_state_dict, .to()) is re-bound on the spot."""
        if context is None:
            return None
        table = self.__dict__.get("_static")
        if not table:
            return None
        e = table.get(id(context))
        if e is None or e[0] is not context:
            return None
        if e[3] != self._weights_key():
            if torch.cuda.is_current_stream_capturing():
                raise RuntimeError("cross-attention weights changed after bind_static_context(); re-bind before capture")
            self.bind_static_context(context)
            e = table[id(context)]
        return e

    def bind_static_context(self, context: Optional[torch.Tensor]) -> None:
        """Precompute K/V of a context that stays constant across sampler steps (the text embedding:
        SURVEY.md 8(a) a8 notes the reference re-projects it every step).  `context` must be the very
        tensor object later passed to forward(); several contexts may be bound (one per CFG half).
        Results are written in place when a buffer for that object exists, so captured CUDA graphs stay
        valid.  Pass None to unbind everything."""
        table = self.__dict__.setdefault("_static", {})
        if context is None:
            table.clear()
            return
        old = table.get(id(context))
        shape = (*context.shape[:-1], 2 * self.to_q.weight.shape[0])
        same = old is not None and old[0] is context and tuple(old[1].shape) == shape
        kv = ops.gemm(context, self._wkv(), out=old[1] if same else None)
        fused = self._fold_projections(context)
        if same and old[2] is not None and fused is not None and len(old[2]) == len(fused):
            for dst, src in zip(old[2], fused):
                dst.copy_(src)
            fused = old[2]
        table[id(context)] = (context, kv, fused, self._weights_key())

    def bound_tensors(self, context):
        """The device tensors bound for `context` (K/V, folded K', folded V'): snapshot / restore by the engine
        when it switches between captions."""
        e = self.__dict__.get("_static", {}).get(id(context))
        if e is None or e[0] is not context:
            return []
        return [e[1]] + ([t for t in e[2] if t.is_cuda or t.dim() > 0] if e[2] is not None else [])

    SEG = 80  # key slots per head in the folded form (77 text tokens, padded)

    @torch.no_grad()
    def _fold_projections(self, context: torch.Tensor):
        """With a context that is constant over the steps, to_q folds into the keys and to_out into the values:
            softmax(x Wq^T K_h^T * s) V_h Wo_h^T  =  softmax(x K'_h^T) V'_h,   K'_h = s K_h Wq_h,  V'_h = V_h Wo_h^T
        so a cross-attention is two GEMMs (the first with a per-head softmax epilogue) instead of q-projection +
        attention + out-projection.  One-time fp32 preparation per bound context, like weight packing.
        Returns (K' [B, H*80, C] bf16 in log2 units, V'^T [B, C, H*80] bf16, number of keys) or None.
        With a LayerNorm to fold (`_fold_norm`) K' additionally absorbs its gain, and two more tensors follow: the column
        sums of the rounded K' gamma and the shift K' beta, both [B, H*80] fp32 (ops.gemm's `ln` operands):
            LN(x) K'^T = rstd * (x (K' gamma)^T - mean * colsum) + K' beta."""
        b, tk = context.shape[0], context.shape[1]
        if context.dim() != 3 or tk > self.SEG:
            return None
        h, c = self.heads, self.to_q.weight.shape[1]
        ctx = context.float()
        k = (ctx @ self.to_k.weight.float().t()).view(b, tk, h, 64)
        v = (ctx @ self.to_v.weight.float().t()).view(b, tk, h, 64)
        wq = self.to_q.weight.float().view(h, 64, c)
        wo = self.to_out[0].weight.float().view(-1, h, 64)
        kp = torch.zeros(b, h, self.SEG, c, device=context.device)
        kp[:, :, :tk] = torch.einsum("bjhd,hdc->bhjc", k, wq) * (self.scale * 1.4426950408889634)
        vp = torch.zeros(b, h, self.SEG, wo.shape[0], device=context.device)
        vp[:, :, :tk] = torch.einsum("bjhd,chd->bhjc", v, wo)
        kp = kp.reshape(b, h * self.SEG, c)
        vpt = vp.reshape(b, h * self.SEG, -1).transpose(1, 2).to(bf16).contiguous()
        norm = self._fold_norm()
        if norm is None:
            return (kp.to(bf16).contiguous(), vpt, torch.tensor(tk))
        kg = (kp * norm.weight.float()).to(bf16).contiguous()
        return (kg, vpt, torch.tensor(tk), kg.float().sum(-1).contiguous(), (kp @ norm.bias.float()).contiguous())

    def forward(self, x, context=None, mask=None, additional_tokens=None, n_times_crossframe_attn_in_self=0,
                residual: Optional[torch.Tensor] = None, alpha: float = 1.0, kv: Optional[torch.Tensor] = None,
                ln=None, want_stats: bool = False):
        """`ln` = (LayerNorm, RowStats of x): x is the RAW residual stream; the norm is folded into the first GEMM
        (QKV projection, or the folded-key product of a bound context) where that exists, otherwise applied by the
        LayerNorm kernel here.  `want_stats`: return (out, RowStats of out) for the next folded norm."""
        if mask is not None or additional_tokens is not None or n_times_crossframe_attn_in_self:
            raise NotImplementedError("masks / additional tokens / cross-frame attention are not on the hot path")
        x = tokens_bf16(x)
        ctx = tokens_bf16(context) if context is not None else None
        if ctx is not None and kv is None and x.dim() == 3 and x.shape[1] % 256 == 0:
            bound = self._bound_entry(ctx)
            folds_ln = bound is not None and bound[2] is not None and len(bound[2]) == 5
            if folds_ln and (ln is None or ln[0] is not self._fold_norm()):
                bound = None    # the bound keys carry a LayerNorm this call does not ask for: take the general path
            if bound is not None and bound[2] is not None and x.shape[0] % bound[2][0].shape[0] == 0:
                # The bound context may have fewer rows than x: [uncond; cond] captions shared by several latents
                # (tiles of one image batched into one step).  Rows of x are ordered [uncond x n; cond x n], so
                # each context row serves a contiguous block of n * T query rows.
                k_fold, v_fold, tk = bound[2][:3]
                rpg = x.shape[1] * (x.shape[0] // k_fold.shape[0])
                if folds_ln:
                    p = ops.gemm(x, k_fold, softmax_valid=int(tk), w_rows_per_group=rpg,
                                 ln=(ln[1], bound[2][3], bound[2][4], ln[0].eps))
                else:
                    if ln is not None:
                        x = ops.layer_norm(x, ln[0].weight, ln[0].bias, ln[0].eps)
                    p = ops.gemm(x, k_fold, softmax_valid=int(tk), w_rows_per_group=rpg)
                bias = self._pk("out.b", (self.to_out[0].bias,), _F32)
                return ops.gemm(p, v_fold, bias, residual=residual, alpha=alpha, w_rows_per_group=rpg,
                                want_stats=want_stats)
        if ln is not None and ctx is not None:
            x, ln = ops.layer_norm(x, ln[0].weight, ln[0].bias, ln[0].eps), None
        return _linear(self, "out", self.to_out[0], self.attend(x, ctx, kv, ln=ln), residual=residual, alpha=alpha,
                       want_stats=want_stats)


MemoryEfficientCrossAttention = CrossAttention  # attention.py:288-373 computes the same function


class BasicTransformerBlock(nn.Module):
    """attention.py:376-486; the three residual adds are fused into the producing GEMMs."""

    def __init__(self, dim, n_heads, d_head, dropout=0.0, context_dim=None, gated_ff=True, checkpoint=True,
                 disable_self_attn=False, attn_mode="softmax", sdp_backend=None):
        super().__init__()
        self.disable_self_attn = disable_self_attn
        self.attn1 = CrossAttention(query_dim=dim, heads=n_heads, dim_head=d_head, dropout=dropout,
                                    context_dim=context_dim if disable_self_attn else None)
        self.ff = FeedForward(dim, dropout=dropout, glu=gated_ff)
        self.attn2 = CrossAttention(query_dim=dim, context_dim=context_dim, heads=n_heads, dim_head=d_head,
                                    dropout=dropout)
        self.norm1, self.norm2, self.norm3 = nn.LayerNorm(dim), nn.LayerNorm(dim), nn.LayerNorm(dim)
        self.checkpoint = checkpoint
        self.attn2.__dict__["_pre_norm"] = self.norm2   # not a submodule of attn2: folded into its bound keys

    @staticmethod
    def _ln(norm: nn.LayerNorm, x):
        return ops.layer_norm(x, norm.weight, norm.bias, norm.eps)

    def forward(self, x, context=None, additional_tokens=None, n_times_crossframe_attn_in_self=0, stats=None,
                want_stats: bool = False):
        """`stats`: RowStats of x written by the GEMM that produced it.  With them no LayerNorm kernel runs: each norm is
        folded into the GEMM behind it and every residual GEMM hands the statistics of its output to the next one
        (DESIGN.md section 4).  `want_stats`: return (x, RowStats) for the next block."""
        x = tokens_bf16(x)
        if stats is None:
            x = self.attn1(self._ln(self.norm1, x), context=context if self.disable_self_attn else None, residual=x)
            x = self.attn2(self._ln(self.norm2, x), context=context, residual=x)
            return self.ff(self._ln(self.norm3, x), residual=x, want_stats=want_stats)
        x, stats = self.attn1(x, context=context if self.disable_self_attn else None, residual=x,
                              ln=(self.norm1, stats), want_stats=True)
        x, stats = self.attn2(x, context=context, residual=x, ln=(self.norm2, stats), want_stats=True)
        return self.ff(x, residual=x, ln=(self.norm3, stats), want_stats=want_stats)


class SpatialTransformer(nn.Module, Packed):
    """attention.py:533-635 with use_linear=True.  NHWC pixels *are* the token matrix, so both
    rearranges are free; proj_out's epilogue adds the block input."""

    def __init__(self, in_channels, n_heads, d_head, depth=1, dropout=0.0, context_dim=None, disable_self_attn=False,
                 use_linear=False, attn_type="softmax", use_checkpoint=True, sdp_backend=None):
        super().__init__()
        assert use_linear, "the YAML selects use_linear_in_transformer=True"
        if exists(context_dim) and not isinstance(context_dim, (list, tuple)):
            context_dim = [context_dim]
        if exists(context_dim):
            context_dim = list(context_dim)
            if depth != len(context_dim):
                assert all(c == context_dim[0] for c in context_dim)
                context_dim = depth * [context_dim[0]]
        else:
            context_dim = [None] * depth
        self.in_channels = in_channels
        inner_dim = n_heads * d_head
        self.norm = nn.GroupNorm(num_groups=32, num_channels=in_channels, eps=1e-6, affine=True)
        self.proj_in = nn.Linear(in_channels, inner_dim)
        self.transformer_blocks = nn.ModuleList([
            BasicTransformerBlock(inner_dim, n_heads, d_head, dropout=dropout, context_dim=context_dim[d],
                                  disable_self_attn=disable_self_attn, attn_mode=attn_type, checkpoint=use_checkpoint)
            for d in range(depth)])
        self.proj_out = zero_module(nn.Linear(inner_dim, in_channels))
        self.use_linear = use_linear

    def forward_nhwc(self, x, context=None):
        if not isinstance(context, list):
            context = [context]
        context = [tokens_bf16(c) if c is not None else None for c in context]
        b, h, w, c = x.shape
        t = _gn(self.norm, x).view(b, h * w, c)
        t, stats = _linear(self, "proj_in", self.proj_in, t, want_stats=True)
        last = len(self.transformer_blocks) - 1
        for i, block in enumerate(self.transformer_blocks):
            r = block(t, context=context[i if len(context) > 1 else 0], stats=stats, want_stats=i < last)
            t, stats = r if isinstance(r, tuple) else (r, None)
        t = _linear(self, "proj_out", self.proj_out, t, residual=x.view(b, h * w, c))
        return t.view(b, h, w, c)

    def forward(self, x, context=None):
        return from_nhwc(self.forward_nhwc(to_nhwc(x), context))


class TimestepEmbedSequential(nn.Sequential, TimestepBlock):
    """openaimodel.py:75-99."""

    def forward_nhwc(self, x, emb, context=None):
        for layer in self:
            if isinstance(layer, TimestepBlock):
                x = layer.forward_nhwc(x, emb)
            elif isinstance(layer, SpatialTransformer):
                x = layer.forward_nhwc(x, context)
            elif isinstance(layer, nn.Conv2d):
                x = _stem_conv(layer, x)
            else:
                x = layer.forward_nhwc(x)
        return x

    def forward(self, x, emb, context=None, **unused):
        return from_nhwc(self.forward_nhwc(to_nhwc(x), emb, context))


def _stem_conv(conv: nn.Conv2d, x_nhwc: torch.Tensor, addend: Optional[torch.Tensor] = None) -> torch.Tensor:
    """latent (<= 8 channels) -> features (input_blocks.0.0, input_hint_block.0): the input is zero-padded to
    one 64-channel K chunk so the convolution runs on the tcgen05 implicit-GEMM path (the direct
    few-channel kernel is 60x slower at 128^2)."""
    cache = conv.__dict__.setdefault("_pk_cache", {})
    key = (conv.weight.data_ptr(), conv.weight._version, conv.bias.data_ptr(), conv.bias._version)
    if cache.get("key") != key:
        with torch.no_grad():
            cache["key"], cache["w"], cache["b"] = key, ops.pack_conv3x3_padded(conv.weight, 64), _F32(conv.bias)
    return ops.conv3x3(ops.pad_channels(x_nhwc, 64), cache["w"], cache["b"], residual=addend)


# ------------------------------------------------------------------------------------------------
# UNetModel (constructor only builds what the YAML configuration uses)
# ------------------------------------------------------------------------------------------------
class UNetModel(nn.Module, Packed):
    """openaimodel.py:500-1007 for use_spatial_transformer=True, dims=2, conv resampling,
    num_classes in {None, "sequential"}.  Produces the reference's module tree / state_dict keys."""

    def __init__(self, in_channels, model_channels, out_channels, num_res_blocks, attention_resolutions, dropout=0,
                 channel_mult=(1, 2, 4, 8), conv_resample=True, dims=2, num_classes=None, use_checkpoint=False,
                 use_fp16=False, num_heads=-1, num_head_channels=-1, num_heads_upsample=-1, use_scale_shift_norm=False,
                 resblock_updown=False, use_new_attention_order=False, use_spatial_transformer=False,
                 transformer_depth=1, context_dim=None, n_embed=None, legacy=True, disable_self_attentions=None,
                 num_attention_blocks=None, disable_middle_self_attn=False, use_linear_in_transformer=False,
                 spatial_transformer_attn_type="softmax", adm_in_channels=None, use_fairscale_checkpoint=False,
                 offload_to_cpu=False, transformer_depth_middle=None, _build_output_blocks=True):
        super().__init__()
        assert use_spatial_transformer and context_dim is not None and dims == 2 and conv_resample
        assert not resblock_updown and not use_scale_shift_norm and n_embed is None
        assert num_head_channels != -1 or num_heads != -1
        if isinstance(context_dim, (list, tuple)) or type(context_dim).__name__ == "ListConfig":
            context_dim = list(context_dim)
        self.in_channels, self.model_channels, self.out_channels = in_channels, model_channels, out_channels
        if isinstance(transformer_depth, int):
            transformer_depth = len(channel_mult) * [transformer_depth]
        transformer_depth = list(transformer_depth)
        transformer_depth_middle = transformer_depth[-1] if transformer_depth_middle is None else transformer_depth_middle
        if isinstance(num_res_blocks, int):
            self.num_res_blocks = len(channel_mult) * [num_res_blocks]
        else:
            if len(num_res_blocks) != len(channel_mult):
                raise ValueError("provide num_res_blocks either as an int (globally constant) or as a list/tuple "
                                 "(per-level) with the same length as channel_mult")
            self.num_res_blocks = list(num_res_blocks)
        self.attention_resolutions, self.dropout, self.channel_mult = attention_resolutions, dropout, channel_mult
        self.conv_resample, self.num_classes, self.use_checkpoint = conv_resample, num_classes, use_checkpoint
        self.num_heads, self.num_head_channels = num_heads, num_head_channels
        self.num_heads_upsample = num_heads if num_heads_upsample == -1 else num_heads_upsample
        self.predict_codebook_ids = False

        time_embed_dim = model_channels * 4
        self.time_embed = nn.Sequential(nn.Linear(model_channels, time_embed_dim), nn.SiLU(),
                                        nn.Linear(time_embed_dim, time_embed_dim))
        if num_classes is not None:
            if num_classes != "sequential":
                raise ValueError("only num_classes='sequential' (SDXL vector conditioning) is on the hot path")
            assert adm_in_channels is not None
            self.label_emb = nn.Sequential(nn.Sequential(nn.Linear(adm_in_channels, time_embed_dim), nn.SiLU(),
                                                         nn.Linear(time_embed_dim, time_embed_dim)))

        def heads_for(ch):
            if num_head_channels == -1:
                return num_heads, ch // num_heads
            return ch // num_head_channels, num_head_channels

        def transformer(ch, depth, level=None, middle=False):
            nh, dh = heads_for(ch)
            if legacy:
                dh = ch // nh
            disabled = disable_middle_self_attn if middle else (
                disable_self_attentions[level] if exists(disable_self_attentions) else False)
            return SpatialTransformer(ch, nh, dh, depth=depth, context_dim=context_dim, disable_self_attn=disabled,
                                      use_linear=use_linear_in_transformer, attn_type=spatial_transformer_attn_type,
                                      use_checkpoint=use_checkpoint)

        self.input_blocks = nn.ModuleList([TimestepEmbedSequential(nn.Conv2d(in_channels, model_channels, 3, padding=1))])
        input_block_chans = [model_channels]
        ch, ds = model_channels, 1
        for level, mult in enumerate(channel_mult):
            for nr in range(self.num_res_blocks[level]):
                layers = [ResBlock(ch, time_embed_dim, dropout, out_channels=mult * model_channels, dims=dims,
                                   use_checkpoint=use_checkpoint)]
                ch = mult * model_channels
                if ds in attention_resolutions and (not exists(num_attention_blocks) or nr < num_attention_blocks[level]):
                    layers.append(transformer(ch, transformer_depth[level], level))
                self.input_blocks.append(TimestepEmbedSequential(*layers))
                input_block_chans.append(ch)
            if level != len(channel_mult) - 1:
                self.input_blocks.append(TimestepEmbedSequential(Downsample(ch, conv_resample, dims=dims, out_channels=ch)))
                input_block_chans.append(ch)
                ds *= 2
        self.middle_block = TimestepEmbedSequential(
            ResBlock(ch, time_embed_dim, dropout, dims=dims, use_checkpoint=use_checkpoint),
            transformer(ch, transformer_depth_middle, middle=True),
            ResBlock(ch, time_embed_dim, dropout, dims=dims, use_checkpoint=use_checkpoint))
        if not _build_output_blocks:
            return
        self.output_blocks = nn.ModuleList([])
        for level, mult in list(enumerate(channel_mult))[::-1]:
            for i in range(self.num_res_blocks[level] + 1):
                ich = input_block_chans.pop()
                layers = [ResBlock(ch + ich, time_embed_dim, dropout, out_channels=model_channels * mult, dims=dims,
                                   use_checkpoint=use_checkpoint)]
                ch = model_channels * mult
                if ds in attention_resolutions and (not exists(num_attention_blocks) or i < num_attention_blocks[level]):
                    layers.append(transformer(ch, transformer_depth[level], level))
                if level and i == self.num_res_blocks[level]:
                    layers.append(Upsample(ch, conv_resample, dims=dims, out_channels=ch))
                    ds //= 2
                self.output_blocks.append(TimestepEmbedSequential(*layers))
        self.out = nn.Sequential(normalization(ch), nn.SiLU(),
                                 zero_module(nn.Conv2d(model_channels, out_channels, 3, padding=1)))

    # -- shared pieces ------------------------------------------------------------------------
    def _embed(self, timesteps, y):
        """time_embed(t_emb) + label_emb(y) -> bf16 [B, 4*model_channels] (openaimodel.py:987-992)."""
        t_emb = timestep_embedding(timesteps, self.model_channels)
        h = _linear(self, "te0", self.time_embed[0], t_emb, act=1)
        if self.num_classes is None:
            emb = _linear(self, "te2", self.time_embed[2], h)
        else:
            emb_t = _linear(self, "te2", self.time_embed[2], h)
            l = _linear(self, "le0", self.label_emb[0][0], tokens_bf16(y), act=1)
            emb = _linear(self, "le2", self.label_emb[0][2], l, residual=emb_t)
        _project_emb_for_resblocks(self, self, emb)
        return emb

    def _out_nchw_f32(self, h_nhwc):
        """self.out: GN32 + SiLU + 3x3 conv to the latent channels, written as fp32 NCHW (openaimodel.py:941-947)."""
        h = _gn(self.out[0], h_nhwc, silu=True)
        conv = self.out[2]
        w8, b8 = self._pk("out.wb8", (conv.weight, conv.bias), ops.pack_conv3x3_few_out)
        return ops.conv3x3_to_nchw_f32(h, w8, b8, conv.weight.shape[0])

    def forward(self, x, timesteps=None, context=None, y=None, **kwargs):
        """openaimodel.py:973-1007 (plain UNet, skip connections by concatenation)."""
        assert (y is not None) == (self.num_classes is not None)
        emb = self._embed(timesteps, y)
        ctx = tokens_bf16(context)
        h, hs = to_nhwc(x), []
        for module in self.input_blocks:
            h = module.forward_nhwc(h, emb, ctx)
            hs.append(h)
        h = self.middle_block.forward_nhwc(h, emb, ctx)
        for module in self.output_blocks:
            h = module.forward_nhwc(ops.concat_add(h, hs.pop()), emb, ctx)
        return self._out_nchw_f32(h)


# ------------------------------------------------------------------------------------------------
# SR_modules.py: adapters, control net, adapted UNet
# ------------------------------------------------------------------------------------------------
class ZeroSFT(nn.Module, Packed):
    """SR_modules.py:59-110.  zero_conv's epilogue adds the skip feature; the concat, GroupNorm,
    (1 + gamma) / beta modulation and control_scale lerp run as one normalisation kernel."""

    def __init__(self, label_nc, norm_nc, concat_channels=0, norm=True, mask=False):
        super().__init__()
        assert norm
        self.norm = norm
        self.param_free_norm = normalization(norm_nc + concat_channels)
        nhidden = 128
        self.mlp_shared = nn.Sequential(nn.Conv2d(label_nc, nhidden, kernel_size=3, padding=1), nn.SiLU())
        self.zero_mul = zero_module(nn.Conv2d(nhidden, norm_nc + concat_channels, kernel_size=3, padding=1))
        self.zero_add = zero_module(nn.Conv2d(nhidden, norm_nc + concat_channels, kernel_size=3, padding=1))
        self.zero_conv = zero_module(nn.Conv2d(label_nc, norm_nc, 1, 1, 0))
        self.pre_concat = bool(concat_channels != 0)
        self.mask = mask

    def precompute(self, c):
        """Everything that depends only on the control feature c (zero_conv(c), gamma, beta): can run on another
        stream while the UNet is still producing h."""
        actv = _conv3x3(self, "mlp", self.mlp_shared[0], c, act=1)
        return {"zc": _linear(self, "zero_conv", self.zero_conv, c),
                "gamma": _conv3x3(self, "mul", self.zero_mul, actv), "beta": _conv3x3(self, "add", self.zero_add, actv)}

    def forward_nhwc(self, c, h, h_ori=None, control_scale=1, pre=None):
        assert self.mask is False
        cat = h_ori is not None and self.pre_concat
        if h_ori is not None and not self.pre_concat:
            raise NotImplementedError("post-concat ZeroSFT is not used by LightGLVUNet")
        control_scale = float(control_scale)
        if pre is None:
            hz = _linear(self, "zero_conv", self.zero_conv, c, residual=h)  # h + zero_conv(c)
            hc = ops.concat_add(h_ori, hz) if cat else hz
            actv = _conv3x3(self, "mlp", self.mlp_shared[0], c, act=1)
            gamma = _conv3x3(self, "mul", self.zero_mul, actv)
            beta = _conv3x3(self, "add", self.zero_add, actv)
        else:
            hc = ops.concat_add(h_ori, h, pre["zc"]) if cat else ops.axpy(h, pre["zc"], 1.0)
            gamma, beta = pre["gamma"], pre["beta"]
        raw = None
        if control_scale != 1.0:
            raw = ops.concat_add(h_ori, h) if cat else h
        return _gn(self.param_free_norm, hc, sft_gamma=gamma, sft_beta=beta, raw=raw, control_scale=control_scale)

    def forward(self, c, h, h_ori=None, control_scale=1):
        return from_nhwc(self.forward_nhwc(to_nhwc(c), to_nhwc(h), None if h_ori is None else to_nhwc(h_ori),
                                           control_scale))


class ZeroCrossAttn(nn.Module, Packed):
    """SR_modules.py:113-149: x + CrossAttention(GN(x), GN(context)) * control_scale."""

    def __init__(self, context_dim, query_dim, zero_out=True, mask=False):
        super().__init__()
        self.attn = CrossAttention(query_dim=query_dim, context_dim=context_dim, heads=query_dim // 64, dim_head=64)
        self.norm1 = normalization(query_dim)
        self.norm2 = normalization(context_dim)
        self.mask = mask

    def precompute(self, context):
        """GN(context) tokens -> K/V projection: depends only on the control feature."""
        b, h, w, cc = context.shape
        ct = _gn(self.norm2, context).view(b, h * w, cc)
        return {"kv": ops.gemm(ct, self.attn._wkv())}

    def forward_nhwc(self, context, x, control_scale=1, pre=None):
        assert self.mask is False
        b, h, w, c = x.shape
        xt = _gn(self.norm1, x).view(b, h * w, c)
        if pre is None:
            ct = _gn(self.norm2, context).view(b, h * w, context.shape[-1])
            out = self.attn(xt, ct, residual=x.view(b, h * w, c), alpha=float(control_scale))
        else:
            out = self.attn(xt, xt, residual=x.view(b, h * w, c), alpha=float(control_scale), kv=pre["kv"])
        return out.view(b, h, w, c)

    def forward(self, context, x, control_scale=1):
        return from_nhwc(self.forward_nhwc(to_nhwc(context), to_nhwc(x), control_scale))


class GLVControl(UNetModel):
    """SR_modules.py:152-537: encoder half + middle block of the SDXL UNet run on the noisy latent,
    with the LQ latent injected through a (zero-initialised) hint convolution after the stem."""

    def __init__(self, *args, input_upscale=1, **kwargs):
        super().__init__(*args, _build_output_blocks=False, **kwargs)
        assert input_upscale == 1
        self.input_upscale = input_upscale
        self.input_hint_block = TimestepEmbedSequential(
            zero_module(nn.Conv2d(self.in_channels, self.model_channels, 3, padding=1)))

    def forward_nhwc(self, x, timesteps, xt, context, y, emb=None) -> List[torch.Tensor]:
        if emb is None:
            emb = self._embed(timesteps, y)
        hint = _stem_conv(self.input_hint_block[0], x)
        hs = []
        h = _stem_conv(self.input_blocks[0][0], xt, addend=hint)  # h = conv(xt); h += guided_hint
        hs.append(h)
        for module in list(self.input_blocks)[1:]:
            h = module.forward_nhwc(h, emb, context)
            hs.append(h)
        hs.append(self.middle_block.forward_nhwc(h, emb, context))
        return hs

    def forward(self, x, timesteps, xt, context=None, y=None, **kwargs):
        assert (y is not None) == (self.num_classes is not None)
        hs = self.forward_nhwc(to_nhwc(x), timesteps, to_nhwc(xt), tokens_bf16(context), y)
        return [from_nhwc(h) for h in hs]


class LightGLVUNet(UNetModel):
    """SR_modules.py:540-883: SDXL UNet whose skip concatenations are replaced by ZeroSFT adapters fed
    with the control features, plus two ZeroCrossAttn adapters before the upsamplers; fbcache modes
    "none", "input_stage1", "input_stage2" (the ones RestoreEDMSampler.fb_mode selects, sampling.py:543)."""

    def __init__(self, mode="", project_type="ZeroSFT", project_channel_scale=1, *args, **kwargs):
        super().__init__(*args, **kwargs)
        if mode == "XL-base":
            cond_output_channels = [320] * 4 + [640] * 3 + [1280] * 3
            project_channels = [160] * 4 + [320] * 3 + [640] * 3
            concat_channels = [320] * 2 + [640] * 3 + [1280] * 4 + [0]
            cross_attn_insert_idx = [6, 3]
            self.progressive_mask_nums = [0, 3, 7, 11]
        elif mode == "XL-refine":
            cond_output_channels = [384] * 4 + [768] * 3 + [1536] * 6
            project_channels = [192] * 4 + [384] * 3 + [768] * 6
            concat_channels = [384] * 2 + [768] * 3 + [1536] * 7 + [0]
            cross_attn_insert_idx = [9, 6, 3]
            self.progressive_mask_nums = [0, 3, 6, 10, 14]
        else:
            raise NotImplementedError
        project_channels = [int(c * project_channel_scale) for c in project_channels]
        self.cache_threshold = 0.1
        self.project_modules = nn.ModuleList()
        for i in range(len(cond_output_channels)):
            if project_type == "ZeroSFT":
                self.project_modules.append(ZeroSFT(project_channels[i], cond_output_channels[i],
                                                    concat_channels=concat_channels[i]))
            elif project_type == "ZeroCrossAttn":
                self.project_modules.append(ZeroCrossAttn(cond_output_channels[i], project_channels[i]))
            else:
                raise NotImplementedError
        for i in cross_attn_insert_idx:
            self.project_modules.insert(i, ZeroCrossAttn(cond_output_channels[i], concat_channels[i]))

    def step_progressive_mask(self):
        if len(self.progressive_mask_nums) > 0:
            mask_num = self.progressive_mask_nums.pop()
            for i in range(len(self.project_modules)):
                self.project_modules[i].mask = i < mask_num

    # -- the two halves of the network --------------------------------------------------------
    def _input_stage(self, x, emb, context):
        hs, h = [], x
        for module in self.input_blocks:
            if isinstance(module[0], nn.Conv2d):
                h = _stem_conv(module[0], h)
            else:
                h = module.forward_nhwc(h, emb, context)
            hs.append(h)
        return h, hs

    def _adapter_controls(self, n_control: int):
        """adapter index -> control index, in the order forward() consumes them (SR_modules.py:628-655)."""
        plan = {}
        a, ci = len(self.project_modules) - 1, n_control - 1
        plan[a] = ci
        a -= 1
        ci -= 1
        for module in self.output_blocks:
            plan[a] = ci
            a -= 1
            if len(module) == 3:
                plan[a] = ci
                a -= 1
            ci -= 1
        return plan

    def precompute_adapters(self, control):
        """Adapter work that needs only the control features (runs on the control stream in the engine)."""
        return {a: self.project_modules[a].precompute(control[ci]) for a, ci in self._adapter_controls(len(control)).items()}

    def _middle(self, h, emb, context):
        return self.middle_block.forward_nhwc(h, emb, context)

    def _output_stage(self, h, hs, emb, context, control, control_scale, pre=None, middle_done=False):
        hs = list(hs)
        pre = pre or {}
        adapter_idx = len(self.project_modules) - 1
        control_idx = len(control) - 1
        if not middle_done:
            h = self.middle_block.forward_nhwc(h, emb, context)
        h = self.project_modules[adapter_idx].forward_nhwc(control[control_idx], h, control_scale=control_scale,
                                                           pre=pre.get(adapter_idx))
        adapter_idx -= 1
        control_idx -= 1
        for module in self.output_blocks:
            _h = hs.pop()
            h = self.project_modules[adapter_idx].forward_nhwc(control[control_idx], _h, h, control_scale=control_scale,
                                                               pre=pre.get(adapter_idx))
            adapter_idx -= 1
            if len(module) == 3:
                assert isinstance(module[2], Upsample)
                h = module[0].forward_nhwc(h, emb)
                h = module[1].forward_nhwc(h, context)
                h = self.project_modules[adapter_idx].forward_nhwc(control[control_idx], h, control_scale=control_scale,
                                                                   pre=pre.get(adapter_idx))
                adapter_idx -= 1
                h = module[2].forward_nhwc(h)
            else:
                h = module.forward_nhwc(h, emb, context)
            control_idx -= 1
        return self._out_nchw_f32(h)

    @torch.no_grad()
    def forward(self, x, timesteps=None, context=None, y=None, control=None, control_scale=1.0, fbcache_mode="none",
                partial_info=None, **kwargs):
        assert (y is not None) == (self.num_classes is not None)
        if fbcache_mode in ("none", "input_stage1"):
            emb = self._embed(timesteps, y)
            ctx = tokens_bf16(context)
            ctrl = [to_nhwc(c) for c in control]
            h, hs = self._input_stage(to_nhwc(x), emb, ctx)
            if fbcache_mode == "input_stage1":
                return {"mode": "input", "h": from_nhwc(h), "hs": [from_nhwc(t) for t in hs], "emb": emb,
                        "context": ctx, "control": [from_nhwc(c) for c in ctrl],
                        "adapter_idx": len(self.project_modules) - 1, "control_idx": len(ctrl) - 1}
            return self._output_stage(h, hs, emb, ctx, ctrl, control_scale)
        if fbcache_mode == "input_stage2":
            if partial_info is None or partial_info.get("mode", "") != "input":
                raise ValueError("input_stage2 requires partial_info from input_stage1")
            return self._output_stage(to_nhwc(partial_info["h"]), [to_nhwc(t) for t in partial_info["hs"]],
                                      partial_info["emb"], tokens_bf16(partial_info["context"]),
                                      [to_nhwc(c) for c in partial_info["control"]], control_scale)
        if fbcache_mode in ("middle_stage1", "middle_stage2", "output_stage1", "output_stage2"):
            raise NotImplementedError(f"fbcache_mode={fbcache_mode}: RestoreEDMSampler.fb_mode is fixed to 'input_stage' "
                                      "(sampling.py:543); the middle/output variants are not on the hot path")
        raise ValueError(f"Unknown fbcache_mode={fbcache_mode}")


class ControlWrapper(nn.Module):
    """wrappers.py:68-110.  `dtype` is kept for interface compatibility (SR_model.py:41 sets it); the
    kernels always compute bf16 x bf16 -> fp32.  Differences from the reference, both semantics-
    preserving: no torch.autocast context is needed, and in "input_stage2" the control net is not
    re-run (the reference recomputes it and then uses the copy stored in partial_info, SR_modules.py:694)."""

    def __init__(self, diffusion_model, compile_model: bool = False, dtype=torch.float32):
        super().__init__()
        self.diffusion_model = diffusion_model
        self.control_model = None
        self.dtype = dtype

    def load_control_model(self, control_model):
        self.control_model = control_model

    def forward(self, x: torch.Tensor, t: torch.Tensor, c: dict, control_scale=1, fbcache_mode="none",
                partial_info=None, **kwargs):
        ops.require_cuda(x, "b200sr.ControlWrapper")
        control = None
        if fbcache_mode != "input_stage2":
            control = self.control_model(x=c.get("control", None), timesteps=t, xt=x,
                                         control_vector=c.get("control_vector", None), mask_x=c.get("mask_x", None),
                                         context=c.get("crossattn", None), y=c.get("vector", None))
        out = self.diffusion_model(x, timesteps=t, context=c.get("crossattn", None), y=c.get("vector", None),
                                   control=control, control_scale=control_scale, fbcache_mode=fbcache_mode,
                                   partial_info=partial_info, **kwargs)
        if "stage1" in fbcache_mode:
            return out
        return out.float()


def bind_text_context(wrapper: nn.Module, context: Optional[torch.Tensor]) -> int:
    """Hoist the text K/V projections of every cross-attention (attn2) out of the step loop."""
    n = 0
    for m in wrapper.modules():
        if isinstance(m, BasicTransformerBlock) and not m.disable_self_attn:
            m.attn2.bind_static_context(context)
            n += 1
    return n


def unbind_text_context(wrapper: nn.Module, context: torch.Tensor) -> None:
    """Drop what bind_text_context(wrapper, context) stored for this one context tensor (an engine going away)."""
    for m in wrapper.modules():
        if isinstance(m, BasicTransformerBlock) and not m.disable_self_attn:
            table = m.attn2.__dict__.get("_static")
            if table:
                e = table.get(id(context))
                if e is not None and e[0] is context:
                    del table[id(context)]


def text_binding_tensors(wrapper: nn.Module, context: torch.Tensor) -> List[torch.Tensor]:
    """All tensors bind_text_context(wrapper, context) produced, in module order."""
    out = []
    for m in wrapper.modules():
        if isinstance(m, BasicTransformerBlock) and not m.disable_self_attn:
            out.extend(m.attn2.bound_tensors(context))
    return out


def build_stage2(network_params: Dict, control_params: Dict) -> ControlWrapper:
    """Convenience: what SR_backbone.__init__ does through instantiate_from_config (SR_model.py:17-51)."""
    wrapper = ControlWrapper(LightGLVUNet(**network_params))
    wrapper.load_control_model(GLVControl(**control_params))
    return wrapper
