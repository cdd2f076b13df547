"""The normalisation edge-case infrastructure checked on the CPU: the GroupNorm geometry port agrees with the path table
the GPU suite relies on, float32 restatements of the kernels' algorithms (in their summation order) stay within the
per-element float64 bounds at every input regime, and every planted defect -- each confined to one (image, group) or one
row -- is rejected, several of them by a margin the whole-tensor ``rel_l2 < 5e-3`` of the older tests cannot see."""
import math

import pytest
import torch

import norm_ref as nr

f32, f64, bf16 = torch.float32, torch.float64, torch.bfloat16


# ---------------------------------------------------------------------------------------------------------------------
# float32 restatements (with switchable defects)
# ---------------------------------------------------------------------------------------------------------------------
def gn_two_kernel(x, w, b, *, groups=32, eps=1e-5, silu=False, gamma=None, beta=None, raw=None, cs=1.0, num_sms=148,
                  defect=None, at=(0, 0)):
    """gn_stats_kernel -> gn_apply_kernel in float32: thread (pl, cv) sums pixels pl, pl + P, ... of its chunk, the CTA
    folds its [P][C] sums per group (thread rows outer, channels inner), the last CTA folds the chunk partials in
    float64 and forms (mean, rstd) as gn_mean_rstd does; the apply pass computes x * sc + sh.  ``defect`` hits the one
    (image, group) ``at``."""
    N, HW, C = x.shape
    geo = nr.gn_geometry(N, HW, C, groups, num_sms)
    P, ppc, chunks, cpg, C8 = geo["P"], geo["ppc"], geo["chunks"], C // groups, C // 8
    n0, g0 = at
    steps = -(-ppc // P)
    xc = torch.zeros(N, chunks * ppc, C)
    xc[:, :HW] = x.float()
    xs = torch.zeros(N, chunks, steps * P, C)
    xs[:, :, :ppc] = xc.view(N, chunks, ppc, C)
    xs = xs.view(N, chunks, steps, P, C)
    s = torch.zeros(N, chunks, P, C)
    q = torch.zeros(N, chunks, P, C)
    for i in range(steps):
        v = xs[:, :, i]
        s, q = s + v, q + v * v
    if defect == "skip_lane":                # the thread of the last channel vector never accumulates (C / 8 % 32 != 0)
        cv = C8 - 1
        assert C8 % 32 != 0 and cv * 8 // cpg == g0
        s[n0, :, 0, cv * 8:cv * 8 + 8] = 0
        q[n0, :, 0, cv * 8:cv * 8 + 8] = 0
    s5, q5 = s.view(N, chunks, P, groups, cpg), q.view(N, chunks, P, groups, cpg)
    pa = torch.zeros(N, chunks, groups)
    pb = torch.zeros(N, chunks, groups)
    for pp in range(P):
        for c in range(cpg):
            pa, pb = pa + s5[:, :, pp, :, c], pb + q5[:, :, pp, :, c]
    keep = torch.ones(N, chunks, groups, dtype=f64)
    if defect == "drop_last_chunk":
        assert geo["last_chunk"] < ppc, "the defect is about a ragged last chunk"
        keep[n0, -1, g0] = 0
    a64, b64 = (pa.double() * keep).sum(1), (pb.double() * keep).sum(1)
    inv = 1.0 / (HW * cpg)
    mean = a64 * inv
    var = (b64 * inv - mean * mean).clamp_min(0.0)
    if defect == "unbiased":
        var[n0, g0] = var[n0, g0] * (HW * cpg) / (HW * cpg - 1)
    var32 = var.float()
    rstd = 1.0 / torch.sqrt(var32 + torch.tensor(eps, dtype=f32))
    if defect == "rsqrt_plus_eps":
        rstd[n0, g0] = 1.0 / torch.sqrt(var32[n0, g0]) + eps
    mean = mean.float()
    if defect == "stale_image":
        assert n0 > 0
        mean[n0, g0], rstd[n0, g0] = mean[n0 - 1, g0], rstd[n0 - 1, g0]
    mc, rc = mean.repeat_interleave(cpg, 1), rstd.repeat_interleave(cpg, 1)       # [N, C]
    if defect == "stale_group":
        assert g0 > 0
        mc[n0, g0 * cpg], rc[n0, g0 * cpg] = mean[n0, g0 - 1], rstd[n0, g0 - 1]
    sc = rc * w[None]
    sh = b[None] - mc * sc
    v = x.float() * sc[:, None] + sh[:, None]
    sel = torch.zeros(N, 1, C, dtype=torch.bool)
    sel[n0, 0, g0 * cpg:(g0 + 1) * cpg] = True
    silu_f = lambda t: t / (1.0 + torch.exp(-t))   # noqa: E731
    late_silu = defect == "silu_after_sft"
    if silu:
        v = torch.where(sel, v, silu_f(v)) if late_silu else silu_f(v)
    if gamma is not None:
        v = v * (1.0 + gamma.float()) + beta.float()
        if late_silu:
            v = torch.where(sel, silu_f(v), v)
        cs32 = torch.tensor(cs, dtype=f32)
        if raw is not None and float(cs32) != 1.0:
            lerp = v * cs32 + raw.float() * (1.0 - cs32)
            swap = v * (1.0 - cs32) + raw.float() * cs32
            v = torch.where(sel, swap, lerp) if defect == "swap_cs" else lerp
    return v.to(bf16)


def _warp_sum(t):
    """[M, 32] lane values -> [M] through the xor-shuffle tree of warp_sum."""
    lane = torch.arange(32)
    for o in (16, 8, 4, 2, 1):
        t = t + t[:, lane ^ o]
    return t[:, 0]


def layer_norm_kernel(x, w, b, eps=1e-5, defect=None, at=0):
    """layer_norm_kernel<VEC> in float32: per lane ``sum += f.x + f.y`` over its vectors, warp tree, ``/ C``; the
    centred second pass likewise; rsqrt; ``(v - mean) * rstd * w + b``.  ``defect`` "next_row_mean": row ``at`` uses the
    mean of row at + 1."""
    M, C = x.shape
    vec = nr.ln_template(C)
    width = vec * 32 * 8
    xp = torch.zeros(M, width)
    xp[:, :C] = x.float()
    lanes = xp.view(M, vec, 32, 8)                  # vector vi = lane + 32 i
    s = torch.zeros(M, 32)
    for i in range(vec):
        for j in range(0, 8, 2):
            s = s + (lanes[:, i, :, j] + lanes[:, i, :, j + 1])
    mean = _warp_sum(s) / C
    if defect == "next_row_mean":
        mean[at] = mean[at + 1]
    valid = torch.zeros(width, dtype=torch.bool)
    valid[:C] = True
    d = torch.where(valid.view(vec, 32, 8)[None], lanes - mean[:, None, None, None], torch.zeros(()))
    sq = torch.zeros(M, 32)
    for i in range(vec):
        for j in range(8):
            sq = sq + d[:, i, :, j] * d[:, i, :, j]
    rstd = torch.rsqrt(_warp_sum(sq) / C + torch.tensor(eps, dtype=f32))
    return ((x.float() - mean[:, None]) * rstd[:, None] * w[None] + b[None]).to(bf16)


def fold_producer(v32, bn):
    """The producer epilogue's partials of fp32 values v32 [M, N] (before their bf16 rounding): per N tile two lanes
    (even / odd columns) accumulate ``bn / 2`` terms each, then add: [parts, M, 2] fp32."""
    M, N = v32.shape
    parts = -(-N // bn)
    vp = torch.zeros(M, parts * bn)
    vp[:, :N] = v32
    t = vp.view(M, parts, bn)
    a1, a2 = torch.zeros(2, M, parts), torch.zeros(2, M, parts)
    for j in range(0, bn, 2):
        pair = t[:, :, j:j + 2].permute(2, 0, 1)
        a1, a2 = a1 + pair, a2 + pair * pair
    return torch.stack([a1[0] + a1[1], a2[0] + a2[1]], -1).transpose(0, 1).contiguous()


def fold_consumer(a, w, buf, colsum, shift, eps=1e-5, *, w_rows_per_group=0, defect=None, at=0):
    """The consumer epilogue in float32: s1, s2 = fp32 sums of the ``parts`` partials, mean = s1 * (1 / K), var =
    max(s2 * (1 / K) - mean^2, 0), rstd = rsqrt(var + eps), nm = -mean * rstd; ``rstd * acc + (nm * colsum + shift)``
    with acc the (accurately rounded) fp32 accumulator.  Defects on row ``at``: "drop_part" (``parts - 1`` partials),
    "next_row_mean" (mean of row at + 1), "wrong_group_colsum" (colsum of the previous weight group)."""
    M, K = a.shape
    w3 = w if w.dim() == 3 else w[None]
    cs3, sh3 = colsum.reshape(w3.shape[0], -1), shift.reshape(w3.shape[0], -1)
    parts = buf.shape[0]
    s1, s2 = torch.zeros(M), torch.zeros(M)
    for q in range(parts):
        use = torch.ones(M, dtype=torch.bool)
        if defect == "drop_part" and q == parts - 1:
            use[at] = False
        s1 = torch.where(use, s1 + buf[q, :, 0], s1)
        s2 = torch.where(use, s2 + buf[q, :, 1], s2)
    inv_k = torch.tensor(1.0 / K, dtype=f32)
    mean = s1 * inv_k
    if defect == "next_row_mean":
        mean[at] = mean[at + 1]
    var = (s2 * inv_k - mean * mean).clamp_min(0.0)
    rstd = torch.rsqrt(var + torch.tensor(eps, dtype=f32))
    nm = -mean * rstd
    rpg = w_rows_per_group or M
    grp = torch.arange(M) // rpg if w_rows_per_group else torch.zeros(M, dtype=torch.long)
    cgrp = grp.clone()
    if defect == "wrong_group_colsum":
        assert grp[at] > 0
        cgrp[at] = grp[at] - 1
    acc = torch.einsum("mk,mnk->mn", a.double(), w3.double()[grp]).float()
    return (rstd[:, None] * acc + (nm[:, None] * cs3[cgrp] + sh3[grp])).to(bf16)


# ---------------------------------------------------------------------------------------------------------------------
# the geometry port
# ---------------------------------------------------------------------------------------------------------------------
PATHS_148 = {
    (2, 64 * 64, 640): 1, (2, 32 * 32, 1280): 1, (2, 32 * 32, 2560): 1, (4, 32 * 32, 1280): 1, (2, 1000, 1280): 1,
    (1, 136, 128): 1, (2, 1024, 960): 1, (128, 8 * 8, 64): 1,
    (8, 32 * 32, 1280): 2, (129, 8 * 8, 64): 2, (2, 128 * 128, 320): 2, (2, 64 * 64, 1920): 2, (1, 1024 * 1024, 128): 2,
}


@pytest.mark.parametrize("shape,launches", list(PATHS_148.items()))
def test_gn_geometry_port_path_table(shape, launches):
    assert nr.gn_geometry(*shape)["launches"] == launches


def test_gn_geometry_port_edges():
    g = nr.gn_geometry(4, 32 * 32, 1280)
    assert g["chunks"] * 4 == 148                               # exactly at the SM count
    assert nr.gn_geometry(8, 32 * 32, 1280)["chunks"] * 8 > 148
    assert nr.gn_geometry(2, 1000, 1280)["last_chunk"] == 6      # ragged
    g = nr.gn_geometry(1, 136, 128)
    assert g["last_chunk"] == 8 and g["P"] == 16                 # fewer pixels than thread rows
    g = nr.gn_geometry(2, 1024, 960)
    assert (g["active"], g["threads"]) == (240, 256)             # idle thread rows
    assert nr.gn_geometry(1, 1024 * 1024, 128)["chunks"] == 296
    assert nr.gn_geometry(4, 32 * 32, 1280, num_sms=150)["launches"] == 2   # 38 chunks of 27 pixels: 152 > 150
    assert [nr.ln_template(c) for c in (8, 248, 264, 768, 1280, 2560, 2568, 5120)] == [1, 1, 3, 3, 5, 10, 20, 20]


def test_generators_reach_every_regime():
    x = nr.gn_inputs(2, 1000, 1280, eps=1e-5, seed=0).double()
    st = nr.gn_stats(x, 32, 1e-5)
    kind = nr.gn_regimes(2, 32)
    assert set(kind.reshape(-1).tolist()) == set(range(len(nr.REGIMES)))
    assert bool((st["var"][kind == nr.REGIMES.index("const")] == 0).all())
    tiny = st["var"][kind == nr.REGIMES.index("tiny")]
    assert bool(((tiny > 0.3e-5) & (tiny < 3e-5)).all())
    r64 = kind == nr.REGIMES.index("r64")
    assert bool((st["mean"][r64].abs() / st["var"][r64].sqrt() > 50).all())
    assert bool((x.abs().amax((1, 2)) > 5e3).all())


# ---------------------------------------------------------------------------------------------------------------------
# restatements within the bounds
# ---------------------------------------------------------------------------------------------------------------------
GN_CASES = [((2, 1000, 1280), 1e-5, True, None), ((1, 136, 128), 1e-6, False, 1.0), ((2, 1024, 960), 1e-5, True, 0.6),
            ((3, 64, 64), 1e-6, True, 0.6), ((2, 8, 64), 1e-5, False, None)]


@pytest.mark.parametrize("shape,eps,silu,cs", GN_CASES)
def test_group_norm_restatement_within_bound(shape, eps, silu, cs):
    N, HW, C = shape
    x = nr.gn_inputs(N, HW, C, eps=eps, seed=HW)
    w, b, gam, bet, raw = nr.gn_params(C, seed=C, sft_shape=shape)
    kw = dict(gamma=gam, beta=bet, raw=raw, cs=cs) if cs is not None else {}
    out = gn_two_kernel(x, w, b, eps=eps, silu=silu, **kw)
    ref, bound = nr.group_norm(x, w, b, eps=eps, silu=silu, sft_gamma=kw.get("gamma"), sft_beta=kw.get("beta"),
                               raw=kw.get("raw"), control_scale=cs if cs is not None else 1.0)
    worst = nr.assert_within(out, ref, bound, f"group norm {shape}")
    print(f"\n[err/bound] fp32 restatement group norm {shape}: {worst:.3f}")
    const = nr.gn_regimes(N, 32) == nr.REGIMES.index("const")
    if not silu and cs is None:                # a constant group's reference is exactly its bias (var = 0)
        sel = const.repeat_interleave(C // 32, 1)[:, None, :].expand(N, HW, C)
        assert bool(sel.any()) and torch.equal(ref[sel], b.double().expand(N, HW, C)[sel])


@pytest.mark.parametrize("C", [8, 264, 1280, 2568])
def test_layer_norm_restatement_within_bound(C):
    x = nr.ln_rows(45, C, seed=C)
    w, b = nr.gn_params(C, seed=C)
    ref, bound = nr.layer_norm(x, w, b)
    worst = nr.assert_within(layer_norm_kernel(x, w, b), ref, bound, f"layer norm C={C}")
    print(f"\n[err/bound] fp32 restatement layer norm C={C}: {worst:.3f}")


def _fold_case(M=384, K=320, N=160, bn=64, groups=1, rpg=0):
    a, w0, res = nr.fold_producer_inputs(M, K, seed=M)
    v32 = (a.double() @ w0.double().T + res.double()).float()
    x = v32.to(bf16)
    buf = fold_producer(v32, bn)
    wp, colsum, shift = nr.fold_weights(N, K, groups=groups, seed=N)
    return x, buf, wp, colsum, shift


def test_fold_producer_restatement_within_bound():
    M, K, bn = 384, 320, 64
    a, w0, res = nr.fold_producer_inputs(M, K, seed=1)
    v32 = (a.double() @ w0.double().T + res.double()).float()
    ref, bound = nr.ln_partials(v32.to(bf16), bn)
    worst = nr.assert_within(fold_producer(v32, bn).reshape(-1, 2), ref.reshape(-1, 2), bound.reshape(-1, 2), "partials")
    print(f"\n[err/bound] fp32 restatement fold producer: {worst:.3f}")


@pytest.mark.parametrize("groups", [1, 3])
def test_fold_consumer_restatement_within_bound(groups):
    rpg = 128 if groups > 1 else 0
    x, buf, wp, colsum, shift = _fold_case(groups=groups)
    out = fold_consumer(x, wp, buf, colsum, shift, w_rows_per_group=rpg)
    ref, bound = nr.ln_fold(x, wp, buf, colsum, shift, w_rows_per_group=rpg)
    worst = nr.assert_within(out, ref, bound, "fold consumer")
    print(f"\n[err/bound] fp32 restatement fold consumer groups={groups}: {worst:.3f}")


# ---------------------------------------------------------------------------------------------------------------------
# planted defects: each rejected, several invisible to the whole-tensor metric
# ---------------------------------------------------------------------------------------------------------------------
def _at(N, kind_name, n=1, skip_first=True):
    """(n, g) of image n's first group in regime ``kind_name`` (g > 0)."""
    kind = nr.gn_regimes(N, 32)[n]
    g = next(i for i in range(1 if skip_first else 0, 32) if nr.REGIMES[int(kind[i])] == kind_name)
    return n, g


GN_DEFECTS = [
    ("drop_last_chunk", (2, 1000, 1280), "outlier", {}),
    ("stale_group", (2, 1024, 1280), "r8", {}),
    ("stale_image", (2, 1024, 1280), "r1", {}),
    ("rsqrt_plus_eps", (2, 1024, 640), "tiny", {}),
    ("unbiased", (2, 8, 64), "r0", {}),
    ("swap_cs", (2, 1024, 640), "r0", dict(sft=True, cs=0.6)),
    ("silu_after_sft", (2, 1024, 640), "r1", dict(sft=True, silu=True)),
    ("skip_lane", (2, 1024, 960), None, {}),
]


MISSED_BY_REL_L2 = ("drop_last_chunk", "stale_group", "stale_image", "unbiased")


def _rejected(out, ref, bound):
    ratio = ((out.double() - ref).abs() / bound).nan_to_num(nan=math.inf).max()
    return float(ratio)


@pytest.mark.parametrize("defect,shape,regime,opt", GN_DEFECTS, ids=[d[0] for d in GN_DEFECTS])
def test_group_norm_planted_defect_rejected(defect, shape, regime, opt):
    N, HW, C = shape
    x = nr.gn_inputs(N, HW, C, seed=3)
    w, b, gam, bet, raw = nr.gn_params(C, seed=4, sft_shape=shape)
    cs = opt.get("cs", 1.0)
    kw = dict(gamma=gam, beta=bet, raw=raw, cs=cs) if opt.get("sft") else {}
    at = (1, C // 32 * 0 + (C // 8 - 1) * 8 // (C // 32)) if regime is None else _at(N, regime)
    out = gn_two_kernel(x, w, b, silu=opt.get("silu", False), defect=defect, at=at, **kw)
    ref, bound = nr.group_norm(x, w, b, silu=opt.get("silu", False), sft_gamma=kw.get("gamma"), sft_beta=kw.get("beta"),
                               raw=kw.get("raw"), control_scale=cs)
    ratio = _rejected(out, ref, bound)
    print(f"\n[defect] {defect} at (image, group) {at}: worst err/bound {ratio:.3g}")
    assert ratio > 1, f"{defect} not rejected"
    if defect in MISSED_BY_REL_L2:
        # the older tests' input (mean 0.7, std 2 everywhere): the defect stays confined and small, rel_l2 passes it
        g = torch.Generator().manual_seed(8)
        xb = (torch.randn(N, HW, C, generator=g) * 2 + 0.7).to(bf16)
        out = gn_two_kernel(xb, w, b, silu=opt.get("silu", False), defect=defect, at=at, **kw)
        ref, bound = nr.group_norm(xb, w, b, silu=opt.get("silu", False), sft_gamma=kw.get("gamma"),
                                   sft_beta=kw.get("beta"), raw=kw.get("raw"), control_scale=cs)
        ratio, l2 = _rejected(out, ref, bound), nr.rel_l2(out.reshape(-1, C), ref.reshape(-1, C))
        print(f"[defect] {defect} on the benign input: worst err/bound {ratio:.3g}, whole-tensor rel_l2 {l2:.2e}")
        assert ratio > 1 and l2 < 5e-3


@pytest.mark.parametrize("defect", ["drop_part", "next_row_mean", "wrong_group_colsum"])
def test_fold_consumer_planted_defect_rejected(defect):
    groups, rpg = 3, 128
    x, buf, wp, colsum, shift = _fold_case(groups=groups)
    at = 128 + 3 if defect == "wrong_group_colsum" else 7    # row 7: offset 8 (FOLD_OFFSETS[7 % 5])
    out = fold_consumer(x, wp, buf, colsum, shift, w_rows_per_group=rpg, defect=defect, at=at)
    ref, bound = nr.ln_fold(x, wp, buf, colsum, shift, w_rows_per_group=rpg)
    ratio = _rejected(out, ref, bound)
    l2 = nr.rel_l2(out, ref)
    print(f"\n[defect] fold consumer {defect} at row {at}: worst err/bound {ratio:.3g}, whole-tensor rel_l2 {l2:.2e}")
    assert ratio > 1, f"{defect} not rejected"


def test_layer_norm_planted_defect_rejected():
    x = nr.ln_rows(333, 768, seed=5)
    w, b = nr.gn_params(768, seed=6)
    ref, bound = nr.layer_norm(x, w, b)
    out = layer_norm_kernel(x, w, b, defect="next_row_mean", at=10)
    ratio = _rejected(out, ref, bound)
    print(f"\n[defect] layer norm next_row_mean: worst err/bound {ratio:.3g}, rel_l2 {nr.rel_l2(out, ref):.2e}")
    assert ratio > 1
