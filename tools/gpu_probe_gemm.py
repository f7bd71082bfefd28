"""GPU probe for the convolution, stem and flat kernels built on the tcgen05 tile kernel: prints one line per case
(never asserts), so one run shows every failing layout combination at once, plus a few throughput probes. Not part of
the test-suite: the GEMM instantiations are tested element by element in tests/test_ppo_gemm_gpu.py."""
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
