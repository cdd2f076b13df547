"""Per-op in-graph timing: each op is captured REP times into one CUDA graph (cycling through enough
distinct weight tensors to keep them cold in L2, like the real step) and the replay is timed.
This is the steady-state cost of one launch inside the step graph (PDL edges included)."""
import math, os, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "remote-sensing-vision-language-diffusion-model_b200"))
import torch
from b200sr import ops
bf16 = torch.bfloat16
dev = "cuda"
REP = 48
def r(*s, scale=0.5): return (torch.randn(*s, device=dev) * scale).to(bf16)

def graph_time(make_calls):
    """make_calls(i) enqueues the i-th launch."""
    for i in range(REP): make_calls(i)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        for i in range(REP): make_calls(i)
    for _ in range(2): g.replay()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(5): g.replay()
    e1.record(); torch.cuda.synchronize()
    return e0.elapsed_time(e1) / 5 / REP * 1e3  # us per launch

rows = []
def gemm_case(M, N, K, geglu=False, residual=False, n_in_step=0):
    nw = max(2, min(REP, int(160e6 / (N * K * 2)) + 1))
    ws = [r(N, K, scale=0.03) for _ in range(nw)]
    bs = torch.randn(N, device=dev)
    a = r(M, K); res = r(M, N) if residual else None
    out = torch.empty(M, N // 2 if geglu else N, device=dev, dtype=bf16)
    t = graph_time(lambda i: ops.gemm(a, ws[i % nw], bs, residual=res, geglu=geglu, out=out))
    fl = 2.0 * M * N * K
    rows.append((f"gemm M{M} N{N} K{K}{' geglu' if geglu else ''}", t, fl / t / 1e6, n_in_step))
def conv_case(N, H, W, Cin, Cout, n_in_step=0):
    nw = max(2, min(REP, int(160e6 / (Cout * 9 * Cin * 2)) + 1))
    ws = [r(Cout, 9 * Cin, scale=0.02) for _ in range(nw)]
    x = r(N, H, W, Cin); b = torch.randn(Cout, device=dev); emb = torch.randn(N, Cout, device=dev)
    t = graph_time(lambda i: ops.conv3x3(x, ws[i % nw], b, rowvec=emb))
    fl = 2.0 * N * H * W * Cout * 9 * Cin
    rows.append((f"conv {N}x{H}x{W} {Cin}->{Cout}", t, fl / t / 1e6, n_in_step))
def attn_case(B, H, Nq, Nk, n_in_step=0):
    C = H * 64
    if Nq == Nk:
        qkv = r(B, Nq, 3 * C)
        t = graph_time(lambda i: ops.attention(qkv, qkv, qkv, H, q_col=0, k_col=C, v_col=2 * C))
    else:
        q = r(B, Nq, C); kv = r(B, Nk, 2 * C)
        t = graph_time(lambda i: ops.attention(q, kv, kv, H, q_col=0, k_col=0, v_col=C))
    fl = 4.0 * B * H * Nq * Nk * 64
    rows.append((f"attn B{B} H{H} Nq{Nq} Nk{Nk}", t, fl / t / 1e6, n_in_step))
def ln_case(M, C, n_in_step=0):
    x = r(M, C); g = torch.ones(C, device=dev); b = torch.zeros(C, device=dev)
    t = graph_time(lambda i: ops.layer_norm(x, g, b))
    rows.append((f"layer_norm M{M} C{C}", t, 4.0 * M * C / t / 1e6, n_in_step))   # "TF/s" column = TB/s here
def gn_case(N, HW, C, n_in_step=0):
    x = r(N, HW, C); g = torch.ones(C, device=dev); b = torch.zeros(C, device=dev)
    t = graph_time(lambda i: ops.group_norm(x, g, b, silu=True))
    rows.append((f"group_norm N{N} HW{HW} C{C} (2 kernels)", t, 6.0 * N * HW * C / t / 1e6, n_in_step))

which = sys.argv[1] if len(sys.argv) > 1 else "all"
if which in ("all", "gemm"):
    gemm_case(2048, 10240, 1280, geglu=True, n_in_step=90)
    gemm_case(2048, 1280, 1280, residual=True, n_in_step=293)
    gemm_case(2048, 1280, 5120, residual=True, n_in_step=90)
    gemm_case(2048, 3840, 1280, n_in_step=90)
    gemm_case(8192, 5120, 640, geglu=True, n_in_step=14)
    gemm_case(8192, 640, 640, residual=True, n_in_step=60)
    gemm_case(8192, 640, 2560, residual=True, n_in_step=14)
    gemm_case(8192, 1920, 640, n_in_step=14)
    conv_case(2, 32, 32, 1280, 1280, 17)
    conv_case(2, 128, 128, 320, 320, 11)
    conv_case(2, 64, 64, 640, 640, 9)
if which == "xattn":
    for (B, T, C, H) in ((2, 1024, 1280, 20), (2, 4096, 640, 10)):
        x = r(B, T, C); kf = [r(B, H * 80, C, scale=0.05) for _ in range(8)]; vf = [r(B, C, H * 80, scale=0.1) for _ in range(8)]
        bias = torch.randn(C, device=dev); res = r(B, T, C)
        p_ = ops.gemm(x, kf[0], softmax_valid=77, w_rows_per_group=T)
        t1 = graph_time(lambda i: ops.gemm(x, kf[i % 8], softmax_valid=77, w_rows_per_group=T))
        t2 = graph_time(lambda i: ops.gemm(p_, vf[i % 8], bias, residual=res, w_rows_per_group=T))
        rows.append((f"xattn gemm1 softmax B{B} T{T} C{C}", t1, 2.0 * B * T * H * 80 * C / t1 / 1e6, 0))
        rows.append((f"xattn gemm2 B{B} T{T} C{C}", t2, 2.0 * B * T * H * 80 * C / t2 / 1e6, 0))
    gemm_case(2048, 10240, 1280, geglu=True, n_in_step=90)
    gemm_case(2048, 1280, 1280, residual=True, n_in_step=293)
    gemm_case(2048, 3840, 1280, n_in_step=90)
if which in ("all", "attn"):
    attn_case(2, 20, 1024, 1024, 91)
    attn_case(2, 10, 4096, 4096, 15)
    attn_case(2, 20, 1024, 77, 90)
    attn_case(2, 10, 4096, 77, 14)
if which in ("all", "norm"):
    ln_case(2048, 1280, 270); ln_case(8192, 640, 42)
    gn_case(2, 1024, 1280, 28); gn_case(2, 16384, 320, 12); gn_case(2, 4096, 640, 17)
if which == "gnconv":
    for (N, H, W, Cin, Cout) in ((2, 32, 32, 1280, 1280), (2, 64, 64, 640, 640), (2, 128, 128, 320, 320), (2, 32, 32, 2560, 1280),
                                 (1, 1024, 1024, 64, 64), (1, 512, 512, 128, 128)):
        nw = max(2, min(REP, int(160e6 / (Cout * 9 * Cin * 2)) + 1))
        ws = [r(Cout, 9 * Cin, scale=0.02) for _ in range(nw)]
        x = r(N, H, W, Cin); b = torch.randn(Cout, device=dev)
        gw = torch.ones(Cin, device=dev); gb = torch.zeros(Cin, device=dev)
        fl = 2.0 * N * H * W * Cout * 9 * Cin
        t0 = graph_time(lambda i: ops.conv3x3(x, ws[i % nw], b))
        t1 = graph_time(lambda i: ops.conv3x3(ops.group_norm(x, gw, gb, silu=True), ws[i % nw], b))
        t2 = graph_time(lambda i: ops.conv3x3(x, ws[i % nw], b, gn=(ops.group_norm_stats(x), gw, gb, 32, True)))
        st = ops.group_norm_stats(x)
        t3 = graph_time(lambda i: ops.conv3x3(x, ws[i % nw], b, gn=(st, gw, gb, 32, True)))
        t4 = graph_time(lambda i: ops.conv3x3(x, ws[i % nw], b, gn=(st, gw, gb, 32, False)))
        t5 = graph_time(lambda i: ops.group_norm_stats(x))
        print(f"conv {N}x{H}x{W} {Cin}->{Cout}: plain conv {t0:6.1f} us | GN(2 kernels)+conv {t1:6.1f} | stats+fused conv {t2:6.1f} | "
              f"fused conv alone {t3:6.1f} (no SiLU {t4:6.1f}) | stats kernel {t5:5.1f}")
if which == "scores":
    # fp32 attention scores of the single-head attention (SR3 / first stage): M = N = 16384 tokens, K = 512
    for (M, N, K) in ((16384, 16384, 512), (4096, 4096, 512)):
        q = r(M, K); k_ = r(N, K)
        out = torch.empty(M, N, device=dev)
        t = graph_time(lambda i: ops.gemm(q, k_, None, alpha=0.044, out=out, out_fp32=True))
        print(f"scores gemm M{M} N{N} K{K} fp32 out: {t:8.1f} us  {2.0 * M * N * K / t / 1e6:7.1f} TF/s  write {M * N * 4 / t / 1e6:6.2f} TB/s"
              f"  (B200SR_EPI_TMA={os.environ.get('B200SR_EPI_TMA', '1')})")
if which == "rowsoftmax":
    for (M, N, K) in ((16384, 16384, 512), (4096, 4096, 512)):
        q = r(M, K); k_ = r(N, K); v_t = r(K, N)
        o = torch.empty(M, K, device=dev, dtype=bf16)
        def two(i):
            p_ = ops.gemm_row_softmax(q, k_, K ** -0.5)
            ops.gemm(p_, v_t, None, w_dynamic=True, out=o)
        t2 = graph_time(two)
        t1 = graph_time(lambda i: ops.gemm_row_softmax(q, k_, K ** -0.5))
        print(f"single-head attention T{M} C{K}: two-pass softmax GEMM + PV {t2:8.1f} us (the two passes alone {t1:8.1f} us)")
if which == "lnfold":
    # (1) single GEMMs back to back: plain / writing row statistics / LayerNorm folded in / both
    for (M, N, K, geglu, residual) in ((2048, 1280, 1280, False, True), (2048, 3840, 1280, False, False),
                                       (2048, 10240, 1280, True, False), (2048, 1280, 5120, False, True),
                                       (8192, 640, 640, False, True), (8192, 1920, 640, False, False)):
        nw = max(2, min(REP, int(160e6 / (N * K * 2)) + 1))
        ws = [r(N, K, scale=0.03) for _ in range(nw)]
        bs = torch.randn(N, device=dev); a = r(M, K); res = r(M, N) if residual else None
        _, st = ops.gemm(r(M, 64), r(K, 64), None, want_stats=True)
        cs = torch.randn(1, N, device=dev); sh = torch.randn(1, N, device=dev)
        out = torch.empty(M, N // 2 if geglu else N, device=dev, dtype=bf16)
        t0 = graph_time(lambda i: ops.gemm(a, ws[i % nw], bs, residual=res, geglu=geglu, out=out))
        t1 = graph_time(lambda i: ops.gemm(a, ws[i % nw], bs, residual=res, geglu=geglu, out=out, ln=(st, cs, sh, 1e-5)))
        t2 = t3 = float("nan")
        if not geglu:
            t2 = graph_time(lambda i: ops.gemm(a, ws[i % nw], bs, residual=res, out=out, want_stats=True))
            t3 = graph_time(lambda i: ops.gemm(a, ws[i % nw], bs, residual=res, out=out, want_stats=True, ln=(st, cs, sh, 1e-5)))
        t4 = graph_time(lambda i: ops.layer_norm(a, torch.ones(K, device=dev), torch.zeros(K, device=dev)))
        print(f"gemm M{M} N{N} K{K} geglu={int(geglu)} res={int(residual)}: plain {t0:6.1f} us | ln in {t1:6.1f} | stats out {t2:6.1f} | "
              f"both {t3:6.1f} | layer_norm of A alone {t4:5.1f}")
    # (2) whole transformer blocks in one graph, text context bound
    from b200sr import modules as md
    for (B, T, C, H) in ((2, 1024, 1280, 20), (2, 4096, 640, 10)):
        nblk = 6
        blocks = [md.BasicTransformerBlock(C, H, 64, context_dim=2048).to(dev) for _ in range(nblk)]
        ctx = r(2, 77, 2048)
        for b_ in blocks:
            b_.attn2.bind_static_context(ctx)
        x0 = r(B, T, 64); w0 = r(C, 64)
        def run(fused):
            if fused:
                x, st = ops.gemm(x0, w0, None, want_stats=True)
            else:
                x, st = ops.gemm(x0, w0, None), None
            for b_ in blocks:
                rr = b_(x, context=ctx, stats=st, want_stats=fused)
                x, st = rr if fused else (rr, None)
            return x
        res_ = {}
        for fused in (True, False):
            with torch.no_grad():
                y = run(fused); torch.cuda.synchronize()
                g = torch.cuda.CUDAGraph()
                with torch.cuda.graph(g):
                    y = run(fused)
                for _ in range(3): g.replay()
                torch.cuda.synchronize()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                for _ in range(10): g.replay()
                e1.record(); torch.cuda.synchronize()
                res_[fused] = (e0.elapsed_time(e1) / 10 / nblk * 1e3, y.float().clone())
        msg = " | ".join(f"{'folded' if k else 'LayerNorm kernels'} {v[0]:7.1f} us/block" for k, v in res_.items())
        msg += f" | rel diff {((res_[True][1] - res_[False][1]).norm() / res_[False][1].norm()).item():.2e}"
        print(f"transformer block B{B} T{T} C{C}: {msg}")
tot = 0.0
print(f"{'op':46s} {'us/launch':>9s} {'TF/s|TB/s':>9s} {'n/step':>6s} {'ms/step':>8s}")
for name, t, rate, n in rows:
    tot += t * n / 1e3
    print(f"{name:46s} {t:9.1f} {rate:9.1f} {n:6d} {t * n / 1e3:8.3f}")
print("sum ms/step of listed ops:", round(tot, 3))
if which == "fixed":
    rows.clear()
    def g2(M, N, K, residual=False, bias=True, bn=0, label=""):
        nw = max(2, min(REP, int(160e6 / (N * K * 2)) + 1))
        ws = [r(N, K, scale=0.03) for _ in range(nw)]
        bs = torch.randn(N, device=dev) if bias else None
        a = r(M, K); res = r(M, N) if residual else None
        out = torch.empty(M, N, device=dev, dtype=bf16)
        t = graph_time(lambda i: ops.gemm(a, ws[i % nw], bs, residual=res, out=out, force_bn=bn))
        rows.append((f"gemm M{M} N{N} K{K} res={int(residual)} bias={int(bias)} bn={bn} {label}", t, 2.0 * M * N * K / t / 1e6, 0))
    for K in (64, 128, 256, 640, 1280, 2560):
        g2(2048, 1280, K)
    g2(2048, 1280, 1280, residual=True)
    g2(2048, 1280, 1280, bias=False)
    for bn in (96, 128, 160, 192, 256):
        g2(2048, 1280, 1280, bn=bn)
    g2(128, 1280, 1280, label="(1 m-block, cluster 1)")
    g2(256, 1280, 1280, label="(1 pair)")
    g2(2048, 160, 1280, label="(8 pairs only)")
    x = r(2048, 1280)
    t = graph_time(lambda i: ops.silu(x))
    rows.append(("silu 2048x1280 (trivial elementwise kernel)", t, 0.0, 0))
    print(f"{'op':70s} {'us/launch':>9s} {'TF/s':>8s}")
    for name, t, rate, n in rows:
        print(f"{name:70s} {t:9.1f} {rate:8.1f}")
