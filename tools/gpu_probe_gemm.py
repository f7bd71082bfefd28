"""GPU probe for the tcgen05 tile kernel: prints one line per case (never asserts) so a single gpurun call
shows every failing descriptor / layout combination at once. Not part of the test-suite."""
import ctypes
import os
import sys
import time

import torch
import torch.nn.functional as F

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from cadre_b200 import _lib  # noqa: E402

L = _lib.lib()
dev = torch.device("cuda:0")
ENC16 = _lib.enc_dtype()
torch.manual_seed(0)


def report(name, got, ref, tol):
    got = got.float()
    ref = ref.float()
    err = (got - ref).abs().max().item()
    scale = ref.abs().max().item() + 1e-30
    bad = not (err <= tol * scale) or not torch.isfinite(got).all().item()
    print(f"{'FAIL' if bad else 'ok  '} {name}: max_abs_err={err:.3e} ref_max={scale:.3e} rel={err/scale:.3e}",
          flush=True)
    return not bad


def run_gemm(kind, a_mn, b_mn, M, N, K, batch=1, out_f32=1, act=0, bias=False, res=False, block_n=0,
             rows=None, name=""):
    dt = torch.float32 if kind else ENC16
    es = 4 if kind else 2
    al = 16 // es

    def pad(x):
        return (x + al - 1) // al * al
    # logical A [batch, M, K], B [batch, N, K]
    A = torch.randn(batch, M, K, device=dev).to(dt)
    Bm = torch.randn(batch, N, K, device=dev).to(dt)
    if a_mn:
        lda = pad(M)
        As = torch.zeros(batch, K, lda, device=dev, dtype=dt)
        As[:, :, :M] = A.transpose(1, 2)
        a_bs = K * lda
    else:
        lda = pad(K)
        As = torch.zeros(batch, M, lda, device=dev, dtype=dt)
        As[:, :, :K] = A
        a_bs = M * lda
    if b_mn:
        ldb = pad(N)
        Bs = torch.zeros(batch, K, ldb, device=dev, dtype=dt)
        Bs[:, :, :N] = Bm.transpose(1, 2)
        b_bs = K * ldb
    else:
        ldb = pad(K)
        Bs = torch.zeros(batch, N, ldb, device=dev, dtype=dt)
        Bs[:, :, :K] = Bm
        b_bs = N * ldb
    odt = torch.float32 if out_f32 else ENC16
    ldc = (N + 7) // 8 * 8
    out = torch.full((batch, M, ldc), 7.0, device=dev, dtype=odt)
    bias_t = torch.randn(batch, N, device=dev) if bias else None
    res_t = torch.randn(batch, M, ldc, device=dev).to(odt) if res else None
    rows_t = torch.tensor(rows, device=dev, dtype=torch.int32) if rows is not None else None
    g = _lib.GemmArgs()
    g.kind, g.a_mn, g.b_mn, g.batch = kind, a_mn, b_mn, batch
    g.M, g.N, g.K, g.block_n = M, N, K, block_n
    g.A, g.B = As.data_ptr(), Bs.data_ptr()
    g.lda, g.a_bs, g.ldb, g.b_bs = lda, a_bs, ldb, b_bs
    g.out, g.ldc, g.out_bs = out.data_ptr(), ldc, M * ldc
    g.out_f32, g.act = out_f32, act
    if bias:
        g.bias, g.bias_bs = bias_t.data_ptr(), N
    if res:
        g.res, g.ldr, g.res_bs = res_t.data_ptr(), ldc, M * ldc
    if rows is not None:
        g.batch_rows = rows_t.data_ptr()
    g.alpha = 1.0
    rc = L.cadre_gemm(ctypes.byref(g), _lib.stream_ptr())
    if rc != 0:
        print(f"FAIL {name}: rc={rc} {L.cadre_last_error().decode()}", flush=True)
        return False
    torch.cuda.synchronize()
    Af, Bf = A.float(), Bm.float()
    ref = torch.bmm(Af.double(), Bf.double().transpose(1, 2)).float()
    if bias:
        ref = ref + bias_t[:, None, :]
    if res:
        ref = ref + res_t[:, :, :N].float()
    if act == 1:
        ref = ref.relu()
    if act == 2:
        ref = F.leaky_relu(ref, 0.01)
    got = out[:, :, :N].float()
    if rows is not None:
        for b, r in enumerate(rows):
            ref[b, r:] = 0
            # rows beyond the last processed tile keep the fill value; only compare processed tiles
            last = min(M, (r + 127) // 128 * 128)
            got[b, last:] = 0
    tol = 2e-3 if kind else (1e-2 if not out_f32 else 1e-4)
    return report(name, got, ref, tol)


def run_conv(B, H, W, Cin, Cout, k, stride, pad, act=1, res=False, name=""):
    x = torch.randn(B, Cin, H, W, device=dev).to(ENC16)
    w = (torch.randn(Cout, Cin, k, k, device=dev) / (Cin * k * k) ** 0.5).to(ENC16)
    bias = torch.randn(Cout, device=dev)
    Ho = (H + 2 * pad - k) // stride + 1
    Wo = (W + 2 * pad - k) // stride + 1
    x_nhwc = x.permute(0, 2, 3, 1).contiguous()
    w_k = w.permute(0, 2, 3, 1).contiguous().view(Cout, -1)
    r = torch.randn(B, Ho, Wo, Cout, device=dev).to(ENC16) if res else None
    out = torch.full((B, Ho, Wo, Cout), 7.0, device=dev, dtype=ENC16)
    rc = L.cadre_conv2d_nhwc(_lib.ptr(x_nhwc), B, H, W, Cin, _lib.ptr(w_k), Cout, k, k, stride, pad,
                             _lib.ptr(bias), _lib.ptr(r), 0, act, _lib.ptr(out), 0, _lib.stream_ptr())
    if rc != 0:
        print(f"FAIL {name}: rc={rc} {L.cadre_last_error().decode()}", flush=True)
        return False
    torch.cuda.synchronize()
    ref = F.conv2d(x.float(), w.float(), bias, stride=stride, padding=pad)
    if res:
        ref = ref + r.float().permute(0, 3, 1, 2)
    if act == 1:
        ref = ref.relu()
    return report(name, out.float().permute(0, 3, 1, 2), ref, 1e-2)


def run_flat(B, H, W, res=False, name=""):
    x = torch.randn(B, 64, H, W, device=dev).to(ENC16)
    w = (torch.randn(64, 64, 3, 3, device=dev) / 24.0).to(ENC16)
    bias = torch.randn(64, device=dev)
    xp = torch.zeros(B, H + 2, W + 2, 64, device=dev, dtype=ENC16)
    xp[:, 1:-1, 1:-1] = x.permute(0, 2, 3, 1)
    w_k = w.permute(0, 2, 3, 1).contiguous().view(64, -1)
    rp = None
    if res:
        r = torch.randn(B, 64, H, W, device=dev).to(ENC16)
        rp = torch.zeros_like(xp)
        rp[:, 1:-1, 1:-1] = r.permute(0, 2, 3, 1)
    out = torch.full((B, H + 2, W + 2, 64), 7.0, device=dev, dtype=ENC16)
    rc = L.cadre_conv3x3_flat64(_lib.ptr(xp), B, H, W, _lib.ptr(w_k), _lib.ptr(bias), _lib.ptr(rp), 1, _lib.ptr(out),
                                _lib.stream_ptr())
    if rc != 0:
        print(f"FAIL {name}: rc={rc} {L.cadre_last_error().decode()}", flush=True)
        return False
    torch.cuda.synchronize()
    ref = F.conv2d(x.float(), w.float(), bias, stride=1, padding=1)
    if res:
        ref = ref + r.float()
    ref = ref.relu()
    border = out.float().clone()
    border[:, 1:-1, 1:-1] = 0
    ok = report(name, out[:, 1:-1, 1:-1].float().permute(0, 3, 1, 2), ref, 1e-2)
    print(f"     border max |y| = {border.abs().max().item():.3e} (must be 0)", flush=True)
    return ok


def run_conv_inpad(B, H, W, Cin, Cout, k, stride, pad, name=""):
    x = torch.randn(B, Cin, H, W, device=dev).to(ENC16)
    w = (torch.randn(Cout, Cin, k, k, device=dev) / (Cin * k * k) ** 0.5).to(ENC16)
    bias = torch.randn(Cout, device=dev)
    Ho = (H + 2 * pad - k) // stride + 1
    Wo = (W + 2 * pad - k) // stride + 1
    xp = torch.zeros(B, H + 2, W + 2, Cin, device=dev, dtype=ENC16)
    xp[:, 1:-1, 1:-1] = x.permute(0, 2, 3, 1)
    w_k = w.permute(0, 2, 3, 1).contiguous().view(Cout, -1)
    out = torch.full((B, Ho, Wo, Cout), 7.0, device=dev, dtype=ENC16)
    rc = L.cadre_conv2d_nhwc(_lib.ptr(xp), B, H, W, Cin, _lib.ptr(w_k), Cout, k, k, stride, pad, _lib.ptr(bias), None, 0,
                             1, _lib.ptr(out), 1, _lib.stream_ptr())
    if rc != 0:
        print(f"FAIL {name}: rc={rc} {L.cadre_last_error().decode()}", flush=True)
        return False
    torch.cuda.synchronize()
    ref = F.conv2d(x.float(), w.float(), bias, stride=stride, padding=pad).relu()
    return report(name, out.float().permute(0, 3, 1, 2), ref, 1e-2)


def run_stem(B, name="stem"):
    x = torch.randn(B, 4, 144, 256, device=dev).to(ENC16)
    w = (torch.randn(64, 4, 7, 7, device=dev) / 14.0).to(ENC16)
    bias = torch.randn(64, device=dev)
    xp = torch.zeros(B, 150, 262, 4, device=dev, dtype=ENC16)
    xp[:, 3:147, 3:259, :] = x.permute(0, 2, 3, 1)
    # row-pair interleaved: [B][75][262][2][4]
    xp = xp.view(B, 75, 2, 262, 4).permute(0, 1, 3, 2, 4).contiguous()
    # weights [64][j 4][kw 8][r 2][c 4], zero for kh==7 / kw==7
    wk = torch.zeros(64, 8, 8, 4, device=dev, dtype=ENC16)   # [o][kh][kw][c]
    wk[:, :7, :7, :] = w.permute(0, 2, 3, 1)
    wk = wk.view(64, 4, 2, 8, 4).permute(0, 1, 3, 2, 4).contiguous().view(64, 256)
    out = torch.zeros(B, 38, 66, 64, device=dev, dtype=ENC16)    # zero-bordered pooled map (interior written)
    rc = L.cadre_stem_pool(_lib.ptr(xp), B, _lib.ptr(wk), _lib.ptr(bias), _lib.ptr(out), _lib.stream_ptr())
    if rc != 0:
        print(f"FAIL {name}: rc={rc} {L.cadre_last_error().decode()}", flush=True)
        return False
    torch.cuda.synchronize()
    ref = F.max_pool2d(F.conv2d(x.float(), w.float(), bias, stride=2, padding=3).relu(), 3, 2, 1)
    return report(name, out[:, 1:-1, 1:-1].float().permute(0, 3, 1, 2), ref, 1e-2)


def timed(fn, iters=20):
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(True), torch.cuda.Event(True)
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters


def main():
    group = sys.argv[1] if len(sys.argv) > 1 else "all"
    print(L.cadre_version().decode(), torch.cuda.get_device_name(0), group, flush=True)
    if group in ("all", "gemm"):
        gemm_cases()
    if group in ("all", "conv"):
        conv_cases()
    if group in ("all", "stem"):
        run_stem(2)
        run_stem(5, name="stem B=5")
    if group in ("all", "flat"):
        run_flat(1, 36, 64, name="flat3x3 B=1")
        run_flat(3, 36, 64, res=True, name="flat3x3 B=3 +res")
        run_flat(37, 36, 64, res=True, name="flat3x3 B=37 +res")
        run_conv_inpad(3, 36, 64, 64, 128, 3, 2, 1, name="conv3x3 s2 from padded input")
        run_conv_inpad(3, 36, 64, 64, 128, 1, 2, 0, name="conv1x1 s2 from padded input")
    if group in ("all", "perf"):
        perf_cases()


def gemm_cases():
    run_gemm(0, 0, 0, 128, 128, 64, name="bf16 KK 128x128x64")
    run_gemm(0, 0, 0, 256, 128, 256, name="bf16 KK 256x128x256")
    run_gemm(0, 0, 0, 300, 200, 104, name="bf16 KK tails 300x200x104")
    run_gemm(0, 0, 0, 256, 64, 512, name="bf16 KK N=64")
    run_gemm(0, 0, 0, 256, 256, 512, out_f32=0, act=1, bias=True, res=True, name="bf16 KK bf16-out bias+res+relu")
    run_gemm(0, 0, 1, 256, 256, 256, name="bf16 K/MN 256^3")
    run_gemm(0, 1, 1, 256, 256, 256, name="bf16 MN/MN 256^3")
    run_gemm(1, 0, 0, 128, 128, 32, name="tf32 KK 128x128x32")
    run_gemm(1, 0, 0, 200, 2120, 530, bias=True, name="tf32 KK 200x2120x530")
    run_gemm(1, 0, 1, 200, 530, 2120, name="tf32 K/MN dgrad 200x530x2120")
    run_gemm(1, 1, 1, 2120, 530, 200, name="tf32 MN/MN wgrad 2120x530x200")
    run_gemm(1, 0, 0, 300, 256, 530, batch=4, rows=[300, 130, 0, 77], name="tf32 KK batched rows")
    run_gemm(1, 0, 0, 128, 64, 128, name="tf32 KK N=64")


def conv_cases():
    run_conv(2, 36, 64, 64, 64, 3, 1, 1, name="conv3x3 s1 36x64 c64->64")
    run_conv(3, 36, 64, 64, 128, 3, 2, 1, name="conv3x3 s2 36x64 c64->128")
    run_conv(3, 36, 64, 64, 128, 1, 2, 0, act=0, name="conv1x1 s2 36x64 c64->128")
    run_conv(4, 18, 32, 128, 128, 3, 1, 1, res=True, name="conv3x3 s1 18x32 c128 +res")
    run_conv(9, 18, 32, 128, 256, 3, 2, 1, name="conv3x3 s2 18x32 c128->256")
    run_conv(9, 9, 16, 256, 256, 3, 1, 1, name="conv3x3 s1 9x16 c256")
    run_conv(17, 9, 16, 256, 512, 3, 2, 1, name="conv3x3 s2 9x16 c256->512")
    run_conv(17, 9, 16, 256, 512, 1, 2, 0, act=0, name="conv1x1 s2 9x16 c256->512")
    run_conv(20, 5, 8, 512, 512, 3, 1, 1, name="conv3x3 s1 5x8 c512")
    run_conv(20, 5, 8, 512, 128, 3, 1, 1, name="conv3x3 s1 5x8 c512->128")
    run_conv(20, 5, 8, 128, 512, 1, 1, 0, act=0, name="conv1x1 s1 5x8 c128->512")


def perf_cases():
    # throughput probes (kernel only)
    for (M, N, K) in [(4096, 4096, 4096), (8192, 8192, 8192)]:
        A = torch.randn(M, K, device=dev).to(ENC16)
        Bm = torch.randn(N, K, device=dev).to(ENC16)
        out = torch.empty(M, N, device=dev, dtype=ENC16)
        g = _lib.GemmArgs()
        g.kind, g.batch, g.M, g.N, g.K = 0, 1, M, N, K
        g.A, g.B, g.lda, g.ldb = A.data_ptr(), Bm.data_ptr(), K, K
        g.out, g.ldc, g.alpha = out.data_ptr(), N, 1.0
        sp = _lib.stream_ptr()
        ms = timed(lambda: L.cadre_gemm(ctypes.byref(g), sp))
        ms_t = timed(lambda: torch.matmul(A, Bm.t()))
        print(f"perf bf16 gemm {M}x{N}x{K}: {ms:.3f} ms = {2*M*N*K/ms/1e9:.1f} TFLOP/s (torch {ms_t:.3f} ms = "
              f"{2*M*N*K/ms_t/1e9:.1f})", flush=True)
    B = 256
    x = torch.randn(B, 36, 64, 64, device=dev).to(ENC16)
    w = torch.randn(64, 576, device=dev).to(ENC16)
    bias = torch.randn(64, device=dev)
    out = torch.empty(B, 36, 64, 64, device=dev, dtype=ENC16)
    sp = _lib.stream_ptr()
    ms = timed(lambda: L.cadre_conv2d_nhwc(_lib.ptr(x), B, 36, 64, 64, _lib.ptr(w), 64, 3, 3, 1, 1, _lib.ptr(bias),
                                           None, 0, 1, _lib.ptr(out), 0, sp))
    fl = 2 * B * 36 * 64 * 64 * 576
    print(f"perf conv3x3 layer1 B={B}: {ms:.3f} ms = {fl/ms/1e9:.1f} TFLOP/s", flush=True)
    x4 = torch.randn(B, 5, 8, 512, device=dev).to(ENC16)
    w4 = torch.randn(512, 4608, device=dev).to(ENC16)
    b4 = torch.randn(512, device=dev)
    o4 = torch.empty(B, 5, 8, 512, device=dev, dtype=ENC16)
    ms = timed(lambda: L.cadre_conv2d_nhwc(_lib.ptr(x4), B, 5, 8, 512, _lib.ptr(w4), 512, 3, 3, 1, 1, _lib.ptr(b4),
                                           None, 0, 1, _lib.ptr(o4), 0, sp))
    fl = 2 * B * 40 * 512 * 4608
    print(f"perf conv3x3 layer4 B={B}: {ms:.3f} ms = {fl/ms/1e9:.1f} TFLOP/s", flush=True)


if __name__ == "__main__":
    main()
