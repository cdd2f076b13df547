"""Every softmax path of the library against float64, element by element, on inputs designed to reach its rescale and
merge code: the attention kernel's lazy rescale and split merge, the per-head segment softmax epilogue (with and without
the LayerNorm fold), the two-pass whole-row softmax of the GEMM, both row-softmax kernels, and CUDA-graph replays of the
stateful ones.  References, bounds (derived in softmax_ref's docstrings) and generators live in tests/softmax_ref.py;
each test prints its worst err / bound."""
import pytest
import torch

import softmax_ref as sr

pytestmark = pytest.mark.gpu
bf16 = torch.bfloat16


@pytest.fixture(scope="module")
def ops():
    from b200sr import ops as _ops

    return _ops


@pytest.fixture(scope="module")
def lib():
    from b200sr import _lib

    return _lib.load()


@pytest.fixture(scope="module")
def num_sms():
    return torch.cuda.get_device_properties(torch.cuda.current_device()).multi_processor_count


def _report(what, worst):
    print(f"\n[err/bound] {what}: {worst:.3f}")


def _attn_counters_zero(ops):
    ws = [w for key, w in ops._ws_cache.items() if key[-1] == "attn"]
    assert ws, "a split plan should have asked for a workspace"
    for w in ws:
        assert int(w[:sr.ATT_WS_COUNTERS].view(torch.int32).abs().sum()) == 0


# ---------------------------------------------------------------------------------------------------------------------
# attention: growth ladder, thresholds, spikes in the ragged last block, uniform rows; split and unsplit plans
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("shape,fused", [
    ((2, 20, 1024, 1024), True),    # 24 tail tiles split 4 ways, 2 blocks per range; fused QKV column windows
    ((1, 33, 1152, 512), False),    # one tail tile split 4 ways, 1 block per range (merge only)
    ((1, 4, 256, 1000), False),     # every tile split, ragged last block
    ((1, 4, 200, 513), False),      # the 1-key last block is a range of its own; Nq not a multiple of 128
    ((2, 20, 1000, 1025), False),   # 3-block ranges, the last ending on the 1-key block
    ((1, 37, 1000, 2049), False),   # 296 tiles = 1 full wave: no split; 17 key blocks, the last with 1 key
])
def test_attention_designed_rows(ops, lib, num_sms, shape, fused):
    B, H, Nq, Nk = shape
    C = H * 64
    q, k, v = (t.cuda() for t in sr.attention_inputs(B, H, Nq, Nk, seed=11))
    plan = sr.attention_plan(B, H, Nq, Nk, num_sms)
    assert lib.b200sr_attention_d64_workspace_bytes(B, H, Nq, Nk) == plan["workspace_bytes"]
    cov = sr.attention_coverage(q, k, H, num_sms=num_sms)
    print(f"\n[coverage] attention {shape}: " + ", ".join(f"{key} {val}" for key, val in cov.items() if key != "plan")
          + f"; split {plan['split']} x {plan['blocks_per_split']} blocks")
    assert cov["rows_rescaled"] > 0 and cov["max_in_last_block"] > 0
    if plan["tail"] and plan["blocks_per_split"] > 1:
        assert cov["rescales_in_split"] > 0
    if fused:
        g = torch.Generator(device="cuda").manual_seed(5)
        buf = torch.randn(B, Nq, 3 * C + 64, generator=g, device="cuda").to(bf16)   # column 0..63: not part of any window
        buf[..., 64:64 + C], buf[..., 64 + C:64 + 2 * C], buf[..., 64 + 2 * C:] = q, k, v
        args, kw = (buf, buf, buf, H), dict(q_col=64, k_col=64 + C, v_col=64 + 2 * C)
    else:
        args, kw = (q, k, v, H), {}
    outs = [ops.attention(*args, **kw) for _ in range(4)]
    torch.cuda.synchronize()
    for o in outs[1:]:
        assert torch.equal(o, outs[0])
    if plan["tail"]:
        _attn_counters_zero(ops)
    ref, bound = sr.attention(q, k, v, H)
    _report(f"attention {shape}", sr.assert_within(outs[0], ref, bound, f"attention {shape}"))


@pytest.mark.parametrize("N", [1, 77, 128])
def test_attention_causal(ops, N):
    q, k, v = (t.cuda() for t in sr.causal_inputs(2, 3, N, seed=N))
    out = ops.attention(q, k, v, 3, causal=True)
    ref, bound = sr.attention(q, k, v, 3, causal=True)
    _report(f"causal attention N={N}", sr.assert_within(out, ref, bound, f"causal attention N={N}"))


def test_attention_causal_beyond_one_key_block_is_refused(ops):
    from b200sr import _lib

    x = torch.zeros(1, 129, 64, dtype=bf16, device="cuda")
    with pytest.raises(_lib.B200SRError):
        ops.attention(x, x, x, 1, causal=True)


# ---------------------------------------------------------------------------------------------------------------------
# per-head segment softmax epilogue (folded text cross-attention), plain and with the LayerNorm fold
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("heads,valid,log2_range,ln", [
    (1, 77, 30.0, False),     # N = 80: one segment per N tile
    (2, 80, 1.0, False),      # N = 160: two segments, no padding
    (3, 2, 30.0, False),      # N = 240: three segments (BN = 240)
    (5, 1, 30.0, False),      # N = 400: tiles of three and two segments; one valid column -> exactly 1
    (3, 77, 200.0, False),    # logits over > 126 log2 units: exponentials flush to zero
    (5, 80, 200.0, True),
    (2, 77, 30.0, True),
    (3, 1, 1.0, True),
    (1, 2, 200.0, True),
])
def test_head_softmax_epilogue(ops, heads, valid, log2_range, ln):
    M, K, groups = 1024, 128, 2
    rpg = M // groups                     # per-group weights, as the folded cross-attention binds two captions
    a, w = sr.head_softmax_inputs(M, K, heads, log2_range, seed=heads * 100 + valid, groups=groups)
    a, w = a.cuda(), w.cuda()
    N = heads * sr.SOFTMAX_SEG
    if ln:
        g = torch.Generator(device="cuda").manual_seed(valid)
        w0 = (torch.randn(K, K, generator=g, device="cuda") * K ** -0.5).to(bf16)
        res = (torch.randn(M, K, generator=g, device="cuda") * 2 - 0.4).to(bf16)
        x, st = ops.gemm(a, w0, None, residual=res, want_stats=True)
        gamma = 1 + 0.3 * torch.randn(K, generator=g, device="cuda")
        beta = 0.2 * torch.randn(K, generator=g, device="cuda")
        kp = w.float()
        kg = (kp * gamma).to(bf16).contiguous()
        colsum, shift = kg.float().sum(-1).contiguous(), (kp @ beta).contiguous()
        lnargs = (st, colsum, shift, 1e-5)
        p = ops.gemm(x, kg, softmax_valid=valid, w_rows_per_group=rpg, ln=lnargs)
        ref, bound = sr.head_softmax(x, kg, valid, w_rows_per_group=rpg, ln=lnargs)
    else:
        p = ops.gemm(a, w, softmax_valid=valid, w_rows_per_group=rpg)
        ref, bound = sr.head_softmax(a, w, valid, w_rows_per_group=rpg)
    seg = p.view(M, heads, sr.SOFTMAX_SEG)
    assert bool((seg[..., valid:] == 0).all())                       # pad columns: exactly 0 (bound 0 says so too)
    if valid == 1:
        assert bool((seg[..., 0] == 1.0).all())
    what = f"head softmax heads={heads} valid={valid} range={log2_range}{' ln' if ln else ''}"
    _report(what, sr.assert_within(p, ref, bound, what))


# ---------------------------------------------------------------------------------------------------------------------
# whole-row softmax: two-pass GEMM, both row-softmax kernels, chunked single-head attention
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("M,N,cut", [(1000, 2048, "tile"), (1000, 2048, "inside"), (1000, 2048, "one"), (700, 4104, None)])
def test_gemm_row_softmax_far_apart_tiles(ops, M, N, cut):
    K = 128
    tile = ops.gemm_n_tile(M, N, K)
    valid = {"tile": 2 * tile, "inside": tile + 37, "one": 1, None: None}[cut]
    a, w = (t.cuda() for t in sr.row_softmax_inputs(M, N, K, tile, seed=N + len(str(cut))))
    p = ops.gemm_row_softmax(a, w, 0.125, valid)
    ref, bound = sr.gemm_row_softmax(a, w, 0.125, valid)
    v = N if valid is None else valid
    assert bool((p[:, v:] == 0).all())
    if v == 1:
        assert bool((p[:, 0] == 1.0).all())
    what = f"gemm_row_softmax M={M} N={N} tile={tile} valid={valid}"
    _report(what, sr.assert_within(p, ref, bound, what))


def _softmax_rows_kernel(x: torch.Tensor) -> str:
    """Which kernel norm.cu's softmax_rows picks for this input (the output is freshly allocated, hence aligned)."""
    cols = x.shape[-1]
    return "block" if 1024 < cols <= 32768 and cols % 4 == 0 and x.data_ptr() % 16 == 0 else "warp"


@pytest.mark.parametrize("rows,cols,valid,offset,kernel", [
    (64, 1024, 1, 0, "warp"),
    (40, 1028, 1000, 0, "block"),
    (8, 32768, 32768, 0, "block"),
    (8, 32772, 30001, 0, "warp"),      # longer than the block kernel holds
    (16, 4099, 4099, 0, "warp"),       # cols % 4 != 0
    (16, 4096, 4000, 1, "warp"),       # a view one float into its buffer: not 16-byte aligned
    (16, 4096, 4000, 0, "block"),
])
def test_softmax_rows_wide_range(ops, rows, cols, valid, offset, kernel):
    data = sr.wide_range_rows(rows, cols, 200.0, seed=cols + offset).cuda()
    buf = torch.empty(rows * cols + 4, device="cuda")
    x = buf[offset:offset + rows * cols].view(rows, cols)
    x.copy_(data)
    assert _softmax_rows_kernel(x) == kernel
    y = ops.softmax_rows(x, 1.0, valid_cols=valid)
    ref, bound = sr.softmax_rows(data, 1.0, valid)
    assert bool((y[:, valid:] == 0).all())
    what = f"softmax_rows {rows}x{cols} valid={valid} ({kernel} kernel)"
    _report(what, sr.assert_within(y, ref, bound, what))


def test_single_head_attention_valid_keys_across_query_chunks(ops, monkeypatch):
    t, tk, c, valid = 1000, 1000, 512, 777
    monkeypatch.setattr(ops, "SCORE_CHUNK_BYTES", 2 * tk * 256)     # 256 query rows per chunk: 4 chunks, the last ragged
    scale = c ** -0.5
    tile = ops.gemm_n_tile(256, tk, c)
    q, k = (x.cuda() for x in sr.row_softmax_inputs(t, tk, c, tile, far=60.0, seed=3, scale=scale))
    g = torch.Generator(device="cuda").manual_seed(4)
    v_t = torch.randn(c, tk, generator=g, device="cuda").to(bf16)
    bias = torch.randn(c, generator=g, device="cuda")
    o = ops.single_head_attention(q, k, v_t, scale, out_bias=bias, valid_keys=valid)
    ref, bound = sr.single_head_attention(q, k, v_t, scale, valid_keys=valid, out_bias=bias)
    _report("single_head_attention", sr.assert_within(o, ref, bound, "single_head_attention"))


# ---------------------------------------------------------------------------------------------------------------------
# CUDA-graph replay of the stateful paths (arrival counters, statistics buffers)
# ---------------------------------------------------------------------------------------------------------------------
def test_graph_replay_switches_rescale_rows(ops, num_sms):
    B, H, N = 2, 20, 1024                       # split plan: 24 tail tiles
    M, NR, K, valid = 1000, 2048, 128, 1500     # several N tiles
    tile = ops.gemm_n_tile(M, NR, K)
    g = torch.Generator().manual_seed(9)
    plain = tuple(torch.randn(B, N, H * 64, generator=g).to(bf16) for _ in range(3))   # never rescales
    att_variants = [sr.attention_inputs(B, H, N, N, seed=21), plain, sr.attention_inputs(B, H, N, N, seed=22)]
    rs_variants = [sr.row_softmax_inputs(M, NR, K, tile, seed=1), sr.row_softmax_inputs(M, NR, K, tile, far=0.0, seed=2),
                   sr.row_softmax_inputs(M, NR, K, tile, seed=3)]
    rescaled = []
    for q, k, _ in att_variants:
        per_row = []
        plan = sr.attention_plan(B, H, N, N, num_sms)
        tail = sr.split_tiles(B, H, N, plan)
        for b in range(B):
            for h in range(H):
                bm = sr.block_maxima(sr.attention_logits(q.cuda(), k.cuda(), H, b, h))
                cnt_full, _ = sr.emulate_lazy_rescale(bm)
                cnt_split, _ = sr.emulate_lazy_rescale(bm, plan["blocks_per_split"])
                per_row.append(torch.where(tail[b, h].cuda(), cnt_split, cnt_full) > 0)
        rescaled.append(torch.cat(per_row))
    for r0, r1 in zip(rescaled, rescaled[1:]):
        assert bool((r0 != r1).any())           # rows switch between rescaling and not from one replay to the next

    qs, ks, vs = (torch.empty(B, N, H * 64, dtype=bf16, device="cuda") for _ in range(3))
    a_s, w_s = torch.empty(M, K, dtype=bf16, device="cuda"), torch.empty(NR, K, dtype=bf16, device="cuda")

    def load(i):
        for dst, src in zip((qs, ks, vs), att_variants[i]):
            dst.copy_(src)
        a_s.copy_(rs_variants[i][0])
        w_s.copy_(rs_variants[i][1])

    def run():
        return ops.attention(qs, ks, vs, H), ops.gemm_row_softmax(a_s, w_s, 0.125, valid)

    load(0)
    run()                                       # eager warm-up: workspaces exist before the capture
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        o_g, p_g = run()
    for i in range(3):
        load(i)
        graph.replay()
        torch.cuda.synchronize()
        o_e, p_e = run()
        torch.cuda.synchronize()
        assert torch.equal(o_g, o_e) and torch.equal(p_g, p_e)
        _attn_counters_zero(ops)
        ref, bound = sr.attention(qs, ks, vs, H)
        _report(f"graph replay {i} attention", sr.assert_within(o_g, ref, bound, f"replay {i} attention"))
        ref, bound = sr.gemm_row_softmax(a_s, w_s, 0.125, valid)
        _report(f"graph replay {i} gemm_row_softmax", sr.assert_within(p_g, ref, bound, f"replay {i} row softmax"))
