"""The softmax edge-case infrastructure checked on the CPU: the designed inputs reach the attention kernel's lazy rescale
and split merge (by the emulator of its decisions), the attention work plan port agrees with the kernel's, and the
per-element float64 bounds accept a float32 restatement of each kernel's blockwise algorithm while rejecting every
planted defect -- defects that the whole-tensor ``rel_l2 < 8e-3`` of the older tests lets through."""
import math

import pytest
import torch

import softmax_ref as sr

f64, bf16 = torch.float64, torch.bfloat16


# ---------------------------------------------------------------------------------------------------------------------
# float32 restatements of the kernels' algorithms (with switchable defects, each confined to one row)
# ---------------------------------------------------------------------------------------------------------------------
def blockwise_attention(q, k, v, heads, scale=0.125, bps=None, defect=None, at=(0, 0, 0)):
    """attention_d64_kernel's algorithm in float32: per 128-key block S = Q K^T, block maximum, lazy rescale of O and l
    when the maximum grew by more than 8 since m_used, P = ex2(S c - m_used) rounded to bf16 before P.V, l from the
    unrounded P; key ranges of ``bps`` blocks publish (O, m_used, l) and are merged with weights ex2(m_used - max).
    Keys beyond Nk read as zeros (the TMA fill) and are masked.  ``defect`` applies to the one row ``at = (b, h, r)``."""
    B, Nq, _ = q.shape
    Nk = k.shape[1]
    nblk = -(-Nk // 128)
    c = torch.tensor(scale * sr.LOG2E, dtype=torch.float32)
    out = torch.empty(B, Nq, heads * 64, dtype=bf16)
    ranges = [(s, min(s + bps, nblk)) for s in range(0, nblk, bps)] if bps else [(0, nblk)]
    for b in range(B):
        for h in range(heads):
            Q = q[b, :, 64 * h:64 * h + 64].float()
            K = torch.zeros(nblk * 128, 64)
            V = torch.zeros(nblk * 128, 64)
            K[:Nk] = k[b, :, 64 * h:64 * h + 64].float()
            V[:Nk] = v[b, :, 64 * h:64 * h + 64].float()
            sel = torch.zeros(Nq, dtype=torch.bool)
            if (b, h) == tuple(at[:2]):
                sel[at[2]] = True
            parts = []
            for j0, j1 in ranges:
                m_used = torch.full((Nq,), -math.inf)
                true_m = torch.full((Nq,), -math.inf)
                l = torch.zeros(Nq)
                O = torch.zeros(Nq, 64)
                skipped = torch.zeros(Nq, dtype=torch.bool)
                for j in range(j0, j1):
                    s = Q @ K[128 * j:128 * j + 128].T
                    keep = (128 * j + torch.arange(128)) < Nk
                    keep = keep[None, :] | (sel[:, None] if defect == "unmasked" else torch.zeros(Nq, 1, dtype=torch.bool))
                    s = torch.where(keep, s, torch.tensor(-math.inf))
                    mx = s.amax(1) * c
                    true_m = torch.maximum(true_m, mx)
                    if j == j0:
                        m_used = mx
                    else:
                        grow = mx > m_used + sr.RESCALE_LOG2
                        alpha = torch.where(grow, torch.exp2(m_used - mx), torch.ones(Nq))
                        alpha_o, alpha_l = alpha, alpha
                        if defect == "no_rescale_o":
                            hit = sel & grow & ~skipped
                            alpha_o = torch.where(hit, torch.ones(Nq), alpha)
                            skipped |= hit
                        if defect == "l_not_rescaled":
                            alpha_l = torch.where(sel, torch.ones(Nq), alpha)
                        O = O * alpha_o[:, None]
                        l = l * alpha_l
                        m_used = torch.where(grow, mx, m_used)
                    e = torch.exp2(s * c - m_used[:, None])
                    l = l + e.sum(1)
                    O = O + e.to(bf16).float() @ V[128 * j:128 * j + 128]
                parts.append((O, m_used, l, true_m))
            if len(parts) == 1:
                O, _, l, _ = parts[0]
            else:
                ms = torch.stack([p[1] for p in parts])
                if defect == "merge_true_max":
                    ms = torch.where(sel[None, :], torch.stack([p[3] for p in parts]), ms)
                w = torch.exp2(ms - ms.amax(0))
                l = sum(w[i] * parts[i][2] for i in range(len(parts)))
                O = sum(w[i][:, None] * parts[i][0] for i in range(len(parts)))
            out[b, :, 64 * h:64 * h + 64] = (O / l[:, None]).to(bf16)
    return out


def segment_softmax(a, w, valid, defect_row=None):
    """The per-head softmax epilogue in float32: fp32 logits, columns >= valid of each 80-column segment masked, ex2 of
    (v - max), one sum, probabilities rounded to bf16.  ``defect_row``: that row's pad columns are not masked."""
    t = a.float() @ w.float().T
    M, N = t.shape
    t = t.view(M, N // 80, 80)
    keep = (torch.arange(80) < valid)[None, None, :].expand(M, N // 80, 80).clone()
    if defect_row is not None:
        keep[defect_row] = True
    t = torch.where(keep, t, torch.tensor(-math.inf))
    e = torch.exp2(t - t.amax(-1, keepdim=True))
    return (e / e.sum(-1, keepdim=True)).to(bf16).view(M, N)


# ---------------------------------------------------------------------------------------------------------------------
# the work plan and the generators
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("shape,split,bps", [((2, 20, 1024, 1024), 4, 2), ((1, 33, 1152, 512), 4, 1),
                                             ((1, 4, 256, 1000), 4, 2), ((1, 4, 200, 513), 3, 2),
                                             ((2, 20, 1000, 1025), 3, 3), ((1, 37, 1000, 2049), 1, 17)])
def test_attention_plan_port(shape, split, bps):
    """The shapes the GPU tests use, with the plan a 148-SM B200 gives them (the GPU test compares the workspace size
    with the library's): split over key ranges or not, and how many key blocks a range holds."""
    plan = sr.attention_plan(*shape)
    assert (plan["split"], plan["blocks_per_split"]) == (split, bps)
    assert (plan["workspace_bytes"] > 0) == (split > 1)
    if shape == (1, 4, 200, 513):   # the ragged 1-key last block is a key range of its own
        assert plan["nblk"] - (plan["split"] - 1) * plan["blocks_per_split"] == 1


@pytest.mark.parametrize("shape", [(1, 4, 256, 1000), (1, 4, 200, 513), (2, 20, 1000, 1025)])
def test_designed_attention_inputs_reach_rescale_and_merge(shape):
    B, H, Nq, Nk = shape
    q, k, v = sr.attention_inputs(B, H, Nq, Nk, seed=1)
    cov = sr.attention_coverage(q, k, H)
    print(f"[coverage] {shape}: {cov}")
    assert cov["rows_rescaled"] >= 0.2 * cov["rows"]
    assert cov["near_below"] > 0 and cov["near_above"] > 0
    assert cov["max_in_last_block"] > 0
    if cov["plan"]["blocks_per_split"] > 1 and cov["plan"]["tail"]:
        assert cov["rescales_in_split"] >= 0.05 * cov["split_rows"]
    if Nk % 128 == 1:
        # spike rows (+12, +40) put their row maximum on the one valid key of the ragged last block
        nblk = -(-Nk // 128)
        hits = 0
        for h in range(H):
            t = sr.attention_logits(q, k, H, 0, h)
            _, kind = sr.attention_offsets(Nq, nblk, 0, h, seed=1)
            rows = (kind == sr.ROW_KINDS.index("spike")) & (t[:, -1] - t[:, :-1].amax(1) > 4)
            hits += int(rows.sum())
            assert bool((t[rows].argmax(1) == Nk - 1).all())
        assert hits > 0


@pytest.mark.parametrize("B,H,N", [(1, 8, 1024), (1, 2, 4096)])
def test_random_attention_inputs_never_rescale(B, H, N):
    """The inputs test_attention draws (randn q, k; scale 1/8) never trigger the lazy rescale: 0 of 8192 rows.  This is
    the gap the designed inputs close."""
    g = torch.Generator().manual_seed(N)
    q = torch.randn(B, N, H * 64, generator=g).to(bf16)
    k = torch.randn(B, N, H * 64, generator=g).to(bf16)
    cov = sr.attention_coverage(q, k, H)
    assert cov["rows"] == 8192 and cov["rescales"] == 0


# ---------------------------------------------------------------------------------------------------------------------
# the checker: the honest restatement passes, each planted defect fails, rel_l2 misses every one of them
# ---------------------------------------------------------------------------------------------------------------------
ATT_SHAPE = (1, 16, 1024, 1025)   # 16384 rows; ragged 1-key last block; key ranges of 3 blocks as in a split plan
ATT_BPS = 3


@pytest.fixture(scope="module")
def att_case():
    B, H, Nq, Nk = ATT_SHAPE
    q, k, v = sr.attention_inputs(B, H, Nq, Nk, seed=3)
    ref, bound = sr.attention(q, k, v, H)
    honest = blockwise_attention(q, k, v, H, bps=ATT_BPS)
    return q, k, v, ref, bound, honest


def _defect_row(q, k, H, defect):
    """A row where the defect changes the arithmetic: (b, h, r)."""
    Nq, Nk = q.shape[1], k.shape[1]
    nblk = -(-Nk // 128)
    for h in range(H):
        bm = sr.block_maxima(sr.attention_logits(q, k, H, 0, h))
        _, kind = sr.attention_offsets(Nq, nblk, 0, h, seed=3)
        if defect in ("no_rescale_o", "l_not_rescaled"):
            cnt, _ = sr.emulate_lazy_rescale(bm, ATT_BPS)
            rows = (cnt > 0) & (kind == sr.ROW_KINDS.index("random"))
        elif defect == "merge_true_max":
            # the last range's maximum is stale (grew by 0.5 .. 8 after its first block) while the others' are not
            rng = [bm[:, s:s + ATT_BPS] for s in range(0, nblk, ATT_BPS)]
            stale = [(x.amax(1) - x[:, 0]) for x in rng]
            rows = (stale[-2] > 2) & (stale[-2] < 8) & (stale[0] < 0.5) & (kind == sr.ROW_KINDS.index("random"))
        else:   # unmasked: a row whose maximum is not far above the zero logits of the padding keys
            rows = (kind == sr.ROW_KINDS.index("decreasing")) & (bm.amax(1) < 4)
        idx = rows.nonzero()
        if len(idx):
            return 0, h, int(idx[0])
    raise AssertionError(f"no row for {defect}")


def test_attention_restatement_within_bounds(att_case):
    q, k, v, ref, bound, honest = att_case
    worst = sr.assert_within(honest, ref, bound, "float32 restatement")
    assert worst < 0.6, worst
    assert sr.rel_l2(honest, ref) < 8e-3


@pytest.mark.parametrize("defect", ["no_rescale_o", "merge_true_max", "unmasked", "l_not_rescaled"])
def test_attention_defects_caught(att_case, defect):
    q, k, v, ref, bound, honest = att_case
    at = _defect_row(q, k, ATT_SHAPE[1], defect)
    bad = blockwise_attention(q, k, v, ATT_SHAPE[1], bps=ATT_BPS, defect=defect, at=at)
    changed = (bad != honest).any(-1)
    assert changed.sum() == 1 and bool(changed[0, at[2]])          # the defect is confined to its row
    with pytest.raises(AssertionError, match="err/bound"):
        sr.assert_within(bad, ref, bound, defect)
    assert sr.rel_l2(bad, ref) < 8e-3, "the old whole-tensor check sees this defect too"


def test_segment_softmax_pad_defect_caught():
    M, K, heads, valid = 4096, 128, 3, 77
    a, w = sr.head_softmax_inputs(M, K, heads, 30.0, seed=5)
    ref, bound = sr.head_softmax(a, w[0], valid)
    honest = segment_softmax(a, w[0], valid)
    assert sr.assert_within(honest, ref, bound, "segment softmax") < 0.6
    assert bool((honest.view(M, heads, 80)[..., valid:] == 0).all())
    bad = segment_softmax(a, w[0], valid, defect_row=1234)
    with pytest.raises(AssertionError, match="err/bound"):
        sr.assert_within(bad, ref, bound, "pad defect")
    assert sr.rel_l2(bad, ref) < 8e-3


def test_row_softmax_reference_agrees_with_a_float32_two_pass_fold():
    """gemm_row_softmax's two-pass arithmetic restated in float32 (per-tile (max, sum), folded with the -inf guard,
    then ex2(t - M) / L) lies within the bound, including rows whose tile maxima differ by more than 126 and a
    fully masked tile."""
    M, N, K, tile = 512, 1024, 64, 128
    a, w = sr.row_softmax_inputs(M, N, K, tile, seed=2)
    valid = 3 * tile + 5     # tile 3 partly, tiles 4.. fully masked
    ref, bound = sr.gemm_row_softmax(a, w, 0.125, valid)
    t = (a.float() @ w.float().T) * torch.tensor(0.125 * sr.LOG2E, dtype=torch.float32)
    t[:, valid:] = -math.inf
    tm = t.view(M, N // tile, tile).amax(-1)
    tl = torch.where(torch.isfinite(tm), torch.exp2(t.view(M, N // tile, tile) - tm[..., None]).sum(-1), torch.zeros_like(tm))
    m = tm.amax(1, keepdim=True)
    lsum = (tl * torch.where(torch.isfinite(tm), torch.exp2(tm - m), torch.zeros_like(tm))).sum(1, keepdim=True)
    p = (torch.exp2(t - m) / lsum).to(bf16)
    assert sr.assert_within(p, ref, bound, "two-pass restatement") < 0.6
    assert bool((p[:, valid:] == 0).all())
    assert float((tm.amax(1) - tm[:, :4].amin(1)).max()) > 126
