"""The encoder's tile kernels one operator at a time, at the forward plan's shapes and at their tile edges.

Every operand is generated in fp16, so the kernel and the reference see the same values, and the reference is the same
operation in float64 on the device. Outputs are compared element by element:

    |got - ref| <= u_out * |ref| + 2^-24 + c * S,     S = the same operation on |operands| (conv(|x|, |w|) + |b| ...)

u_out = 2^-11 is the fp16 output rounding (2^-24 for fp32 outputs); c * S covers the fp32 accumulation. c is set from
measurement with a margin of about 4x (`C_ACC`); it stays far below one filter tap's share of S, so a tap, a k-block, a
bias or a tile that goes missing fails the bound. Every output tensor sits between guard regions holding a sentinel,
which must come back unchanged, and bordered outputs must follow their contract (the flat kernels force the border to 0,
the stem and `out_pad` convolutions never write it). The last test replays the backbone through these entry points with
the plan's arguments and must reproduce the encoder's layer4 output bit for bit.
"""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import restate as R

pytestmark = pytest.mark.gpu

U16 = 2.0 ** -11          # fp16 round-to-nearest, relative
U32 = 2.0 ** -24          # fp32 round-to-nearest, relative
TINY = 2.0 ** -24         # absolute floor (fp16 subnormal spacing is 2^-24)
GUARD = 8192              # sentinel elements in front of and behind every output tensor
SENTINEL = -1234.0        # exact in fp16 and fp32
BORDER = -3.0             # pre-filled border of outputs whose border the kernel must not write

# fp32 accumulation term c of the bound, per kernel family: the measured worst c (B200) times about 4
C_ACC = {
    "stem+pool": 2.0 ** -21,                  # measured 9.2e-8
    "layer1 flat64": 2.0 ** -20,              # measured 1.7e-7
    "halo128": 2.0 ** -20,                    # measured 2.3e-7
    "implicit-GEMM conv": 2.0 ** -19,         # measured 4.2e-7
    "fused shortcut": 2.0 ** -19,             # measured 4.2e-7
    "fc1 (persistent GEMM)": 2.0 ** -19,      # measured 3.6e-7
    "fc2 (batched GEMM, fp32 out)": 2.0 ** -19,   # measured 3.8e-7
    "stage": 2.0 ** -19,                      # the implicit-GEMM / GEMM accumulation behind each stage
}
# attention stages carry fp16 attention weights: per-frame rel-L2 and worst element / frame rms, the measured worst
# (B200, B = 1 ... 1024) times about 4: PAM 2.8e-4 / 2.6e-3, CAM 9.2e-5 / 1.3e-3, latent 2.3e-4 / 7.8e-4
STAGE_REL = {"PAM": (1.2e-3, 1.2e-2), "CAM": (4e-4, 5e-3), "fc1 -> latent": (1e-3, 4e-3)}

_WORST = {}


@pytest.fixture(scope="module", autouse=True)
def _report_worst():
    yield
    for name in sorted(_WORST):
        print("  ".join([name] + [f"{k} {v:.3g}" for k, v in _WORST[name].items()]))


def _note(name, **vals):
    d = _WORST.setdefault(name, {})
    for k, v in vals.items():
        d[k] = max(d.get(k, 0.0), v)


def _L():
    from cadre_b200 import _lib
    return _lib, _lib.lib()


def _call(fn, *args):
    _lib, _ = _L()
    _lib.check(fn(*[_lib.ptr(a) if isinstance(a, torch.Tensor) else a for a in args], _lib.stream_ptr()))


def _gen(seed):
    return torch.Generator(device="cuda").manual_seed(seed)


def _randn(g, *shape, scale=1.0, dtype=torch.float16):
    return (torch.randn(*shape, device="cuda", generator=g) * scale).to(dtype)


class Guarded:
    """A tensor of `shape` inside one allocation, between two guard regions of SENTINEL."""

    def __init__(self, shape, fill, dtype=torch.float16):
        self.n = int(np.prod(shape))
        self.buf = torch.full((2 * GUARD + self.n,), SENTINEL, dtype=dtype, device="cuda")
        self.t = self.buf[GUARD:GUARD + self.n].view(shape)
        self.t.fill_(fill)

    def check(self):
        assert bool((self.buf[:GUARD] == SENTINEL).all()), "write in front of the output tensor"
        assert bool((self.buf[GUARD + self.n:] == SENTINEL).all()), "write behind the output tensor"


def _bordered(x_nhwc, border=0.0):
    B, H, W, C = x_nhwc.shape
    p = torch.full((B, H + 2, W + 2, C), border, dtype=x_nhwc.dtype, device=x_nhwc.device)
    p[:, 1:-1, 1:-1] = x_nhwc
    return p


def _border_is(t, value):
    """Every border pixel of a bordered NHWC tensor holds exactly `value` (bit for bit: +0.0 for 0)."""
    want = torch.tensor(value, dtype=t.dtype).view(torch.int16).item()
    m = torch.ones(t.shape[1], t.shape[2], dtype=torch.bool, device=t.device)
    m[1:-1, 1:-1] = False
    return bool((t.view(torch.int16)[:, m] == want).all())


def _nhwc(x):
    return x.permute(0, 2, 3, 1).contiguous()


def _khwc(w):
    return w.permute(0, 2, 3, 1).contiguous().view(w.shape[0], -1)


def _conv_ref(x, w, b, stride, pad):
    """NCHW float64 convolution of x, w (+ b), and the same on |x|, |w|, |b| (the scale S of the bound)."""
    x, w = x.double(), w.double()
    b = b.double() if b is not None else None
    return (F.conv2d(x, w, b, stride, pad),
            F.conv2d(x.abs(), w.abs(), b.abs() if b is not None else None, stride, pad))


def _check_bound(name, got, ref, S, c, u_out=U16):
    """|got - ref| <= u_out |ref| + 2^-24 + c S element by element; records the worst err / bound and the c needed."""
    got = got.double()
    assert bool(torch.isfinite(got).all()), f"{name}: non-finite output"
    err = (got - ref).abs()
    bound = u_out * ref.abs() + TINY + c * S
    ratio = (err / bound)
    worst = float(ratio.max())
    need = float(((err - u_out * ref.abs() - TINY) / S.clamp_min(1e-300)).max().clamp_min(0.0))
    _note(name, err_over_bound=worst, c_needed=need)
    if worst > 1.0:
        i = int(ratio.flatten().argmax())
        idx = np.unravel_index(i, tuple(ratio.shape))
        raise AssertionError(f"{name}: worst err/bound {worst:.3g} at {idx}: got {got.flatten()[i].item():.6g}, "
                             f"ref {ref.flatten()[i].item():.6g}, S {S.flatten()[i].item():.4g} (c needed {need:.3g})")


# ------------------------------------------------------------------------------------------------ shared encoder
@pytest.fixture(scope="module")
def enc():
    from cadre_b200.encoder import Encoder
    return Encoder(R.danet_fixture_state(0), "cuda:0", max_batch=640)


def _u8_frames(B, seed):
    """rgb with 0 and 255 in every frame; route maps cycling non-binary, all zero, all 255, binary."""
    g = torch.Generator().manual_seed(seed)
    rgb = torch.randint(0, 256, (B, 144, 256, 3), dtype=torch.uint8, generator=g)
    rgb[:, 0, 0], rgb[:, -1, -1] = 0, 255
    route = torch.empty(B, 256, 144, dtype=torch.uint8)
    for n in range(B):
        kind = n % 4
        if kind == 0:
            route[n] = torch.randint(0, 201, (256, 144), dtype=torch.uint8, generator=g)
        elif kind == 1:
            route[n] = 0
        elif kind == 2:
            route[n] = 255
        else:
            route[n] = (torch.rand(256, 144, generator=g) < 0.1).to(torch.uint8) * 255
    return rgb, route


def _pack_image(x):
    """fp16 NCHW [B,4,144,256] -> the stem's row-pair interleaved padded layout [B][75][262][2][4]."""
    B = x.shape[0]
    p = torch.zeros(B, 150, 262, 4, dtype=x.dtype, device=x.device)
    p[:, 3:147, 3:259] = x.permute(0, 2, 3, 1)
    return p.view(B, 75, 2, 262, 4).permute(0, 1, 3, 2, 4).contiguous()


def _unpack_image(p, B):
    return p.view(B, 75, 262, 2, 4).permute(0, 1, 3, 2, 4).reshape(B, 150, 262, 4)[:, 3:147, 3:259].permute(0, 3, 1, 2)


def _pack_stem_w(w):
    """[64,4,7,7] -> [64][256] = [cout][row pair 4][kw 8][row 2][c 4], zero where kh == 7 or kw == 7 (prepare_weights)."""
    wk = torch.zeros(64, 8, 8, 4, dtype=w.dtype, device=w.device)
    wk[:, :7, :7] = w.permute(0, 2, 3, 1)
    return wk.view(64, 4, 2, 8, 4).permute(0, 1, 3, 2, 4).contiguous().view(64, 256)


def _unpack_stem_w(wk):
    return wk.view(64, 4, 8, 2, 4).permute(0, 1, 3, 2, 4).reshape(64, 8, 8, 4)[:, :7, :7].permute(0, 3, 1, 2)


# ------------------------------------------------------------------------------------------------ 1. ingest
@pytest.mark.parametrize("B", [1, 3, 37])
def test_ingest_buffer_is_the_fp16_interleave_of_pre_process(enc, B):
    """preprocess_kernel (uint8) and pack_f32_kernel (fp32) write, bit for bit, the round-to-nearest fp16 image of
    pre_process_tensors at padded rows / columns 3..146 / 3..258 of P[n][row // 2][col][row % 2][c], zero elsewhere."""
    from cadre_b200.agent import pre_process_tensors
    rgb, route = _u8_frames(B, seed=B)
    x = pre_process_tensors(rgb, route)
    want = _pack_image(x.half()).view(-1).view(torch.int16)
    enc.forward_u8(rgb.cuda(), route.cuda())
    got = enc.debug_buffer(6, B).view(torch.int16).cpu()
    assert torch.equal(got, want)
    enc.forward_f32(x.cuda())
    assert torch.equal(enc.debug_buffer(6, B).view(torch.int16).cpu(), want)


# ------------------------------------------------------------------------------------------------ 2. stem + pool
def _run_stem_pool(xp, B, wk, bias):
    _, L = _L()
    out = Guarded((B, 38, 66, 64), BORDER)
    out.t[:, 1:-1, 1:-1] = 7.0
    _call(L.cadre_stem_pool, xp, B, wk, bias, out.t)
    torch.cuda.synchronize()
    out.check()
    assert _border_is(out.t, BORDER), "the stem wrote into the border of its output"
    return out.t[:, 1:-1, 1:-1].permute(0, 3, 1, 2)


def _stem_ref(x, w, b):
    ref, S = _conv_ref(x, w, b, 2, 3)
    return F.max_pool2d(ref.relu(), 3, 2, 1), F.max_pool2d(S, 3, 2, 1)


@pytest.mark.parametrize("B", [1, 2, 49, 50, 640])
def test_stem_pool_matches_fp64(B):
    """tc_stem_pool_kernel: conv7x7/s2/p3 + bias -> ReLU -> maxpool(3, 2, 1). 3 units per image: B = 50 gives 150 units
    on 148 CTAs, so two CTAs take a second unit."""
    g = _gen(200 + B)
    x = _randn(g, B, 4, 144, 256)
    w = _randn(g, 64, 4, 7, 7, scale=1 / 14.0)
    bias = _randn(g, 64, scale=0.5, dtype=torch.float32)
    got = _run_stem_pool(_pack_image(x), B, _pack_stem_w(w), bias)
    ref, S = _stem_ref(x, w, bias)
    _check_bound("stem+pool", got, ref, S, C_ACC["stem+pool"])


def test_stem_pool_with_encoder_weights_on_ingested_frames(enc):
    """The encoder's own packed stem weights on the image its ingest kernel wrote (buffer 6)."""
    B = 37
    rgb, route = _u8_frames(B, seed=300)
    enc.forward_u8(rgb.cuda(), route.cuda())
    xp = enc.debug_buffer(6, B)
    got = _run_stem_pool(xp, B, enc._t["stem_w"], enc._t["stem_b"])
    ref, S = _stem_ref(_unpack_image(xp, B), _unpack_stem_w(enc._t["stem_w"]), enc._t["stem_b"])
    _check_bound("stem+pool", got, ref, S, C_ACC["stem+pool"])


# ------------------------------------------------------------------------------------------------ 3. layer1
@pytest.mark.parametrize("H,W,B", [(36, 64, 1), (36, 64, 5), (36, 64, 8), (36, 64, 32), (36, 64, 640), (3, 5, 7)])
def test_layer1_flat64_matches_fp64_at_tile_edges(H, W, B):
    """tc_flat3x3_kernel over 128-pixel tiles of the flat bordered tensor: B = 1 / 5 end in a tail tile of 76 / 124
    pixels, B = 8 has 157 tiles (a second persistent round), B = 32 no tail, B = 640 is the plan's batch, and at 3x5
    every tile spans several images. Residual on / off, act 0 / 1; the border comes back as exactly 0. At W = 64 the
    result also agrees with the implicit-GEMM kernel (cadre_conv2d_nhwc, in_pad = 1)."""
    _lib, L = _L()
    g = _gen(1000 * H + B)
    x = _randn(g, B, 64, H, W)
    w = _randn(g, 64, 64, 3, 3, scale=1 / 24.0)
    bias = _randn(g, 64, scale=0.5, dtype=torch.float32)
    r = _randn(g, B, 64, H, W)
    xp, rp, w_k = _bordered(_nhwc(x)), _bordered(_nhwc(r)), _khwc(w)
    ref0, S0 = _conv_ref(x, w, bias, 1, 1)
    for res in (False, True):
        for act in (0, 1):
            out = Guarded((B, H + 2, W + 2, 64), 7.0)
            _call(L.cadre_conv3x3_flat64, xp, B, H, W, w_k, bias, rp if res else None, act, out.t)
            torch.cuda.synchronize()
            out.check()
            assert _border_is(out.t, 0.0), "border not forced to 0"
            ref, S = (ref0 + r.double(), S0 + r.double().abs()) if res else (ref0, S0)
            if act:
                ref = ref.relu()
            got = out.t[:, 1:-1, 1:-1].permute(0, 3, 1, 2)
            _check_bound("layer1 flat64", got, ref, S, C_ACC["layer1 flat64"])
            if W == 64:
                old = torch.full((B, H, W, 64), 7.0, device="cuda", dtype=torch.float16)
                _call(L.cadre_conv2d_nhwc, xp, B, H, W, 64, w_k, 64, 3, 3, 1, 1, bias, _nhwc(r) if res else None, 0,
                      act, old, 1)
                torch.cuda.synchronize()
                d = (got.double() - old.permute(0, 3, 1, 2).double()).abs()
                bound = 2 * (U16 * ref.abs() + TINY + C_ACC["layer1 flat64"] * S)
                assert bool((d <= bound).all()), f"flat64 and implicit GEMM differ: worst {float((d / bound).max()):.3g}"


# ------------------------------------------------------------------------------------------------ 4. implicit GEMM
# every cadre_conv2d_nhwc launch of the plan (encoder.cu encoder_trunk) and the unfused downsample convs:
# name: (Hin, Win, Cin, Cout, k, stride, pad, in_pad, out_pad, residual, res_after_act, act)
PLAN_CONVS = {
    "layer2.0.conv1": (36, 64, 64, 128, 3, 2, 1, 1, 1, False, 0, 1),
    "layer3.0.conv1": (18, 32, 128, 256, 3, 2, 1, 1, 0, False, 0, 1),
    "layer3.1.conv1": (9, 16, 256, 256, 3, 1, 1, 0, 0, False, 0, 1),
    "layer3.1.conv2": (9, 16, 256, 256, 3, 1, 1, 0, 0, True, 0, 1),
    "layer4.0.conv1": (9, 16, 256, 512, 3, 2, 1, 0, 0, False, 0, 1),
    "layer4.1.conv1": (5, 8, 512, 512, 3, 1, 1, 0, 0, False, 0, 1),
    "layer4.1.conv2": (5, 8, 512, 512, 3, 1, 1, 0, 0, True, 0, 1),
    "conv5a|5c": (5, 8, 512, 256, 3, 1, 1, 0, 0, False, 0, 1),
    "conv51": (5, 8, 128, 128, 3, 1, 1, 0, 0, False, 0, 1),
    "conv52+sum": (5, 8, 128, 128, 3, 1, 1, 0, 0, True, 1, 1),
    "layer2.0.downsample": (36, 64, 64, 128, 1, 2, 0, 1, 0, False, 0, 0),
    "layer3.0.downsample": (18, 32, 128, 256, 1, 2, 0, 0, 0, False, 0, 0),
    "layer4.0.downsample": (9, 16, 256, 512, 1, 2, 0, 0, 0, False, 0, 0),
}


@pytest.mark.parametrize("B", [1, 3, 17, 640])
@pytest.mark.parametrize("name", list(PLAN_CONVS))
def test_plan_conv_matches_fp64(name, B):
    """tc_persist_kernel with the plan's arguments. Wout = 16 / 8 with odd Hout gives tiles of TN = 8 / 16 images, so
    B = 17 leaves a tile with one valid image; B = 3 gives an odd number of m-tiles for the cta_group::2 pairs."""
    _lib, L = _L()
    Hin, Win, Cin, Cout, k, stride, pad, in_pad, out_pad, has_res, res_after_act, act = PLAN_CONVS[name]
    Ho, Wo = (Hin + 2 * pad - k) // stride + 1, (Win + 2 * pad - k) // stride + 1
    g = _gen(100 * list(PLAN_CONVS).index(name) + B)
    x = _randn(g, B, Cin, Hin, Win)
    w = _randn(g, Cout, Cin, k, k, scale=(Cin * k * k) ** -0.5)
    bias = _randn(g, Cout, scale=0.5, dtype=torch.float32)
    r = _randn(g, B, Ho, Wo, Cout) if has_res else None
    xin = _bordered(_nhwc(x)) if in_pad else _nhwc(x)
    if out_pad:
        out = Guarded((B, Ho + 2, Wo + 2, Cout), BORDER)
        out.t[:, 1:-1, 1:-1] = 7.0
        _call(L.cadre_conv2d_nhwc_bordered_out, xin, B, Hin, Win, Cin, _khwc(w), Cout, k, k, stride, pad, bias, act,
              out.t, in_pad)
        got = out.t[:, 1:-1, 1:-1]
    else:
        out = Guarded((B, Ho, Wo, Cout), 7.0)
        _call(L.cadre_conv2d_nhwc, xin, B, Hin, Win, Cin, _khwc(w), Cout, k, k, stride, pad, bias, r, res_after_act,
              act, out.t, in_pad)
        got = out.t
    torch.cuda.synchronize()
    out.check()
    if out_pad:
        assert _border_is(out.t, BORDER), "an out_pad convolution wrote into the border"
    ref, S = _conv_ref(x, w, bias, stride, pad)
    if has_res:
        rd = r.permute(0, 3, 1, 2).double()
        ref = (ref.relu() + rd) if res_after_act else (ref + rd).relu()
        S = S + rd.abs()
    elif act:
        ref = ref.relu()
    _check_bound("implicit-GEMM conv", got.permute(0, 3, 1, 2), ref, S, C_ACC["implicit-GEMM conv"])


# ------------------------------------------------------------------------------------------------ 5. fused shortcut
# the three plan variants: (Hin, Win, C, in_pad, out_pad, Hin2, Win2, Cin2, in2_pad)
SHORTCUTS = {
    "layer2.0": (18, 32, 128, 1, 1, 36, 64, 64, 1),   # bordered t0 -> bordered y0, in2 = layer1's bordered output
    "layer3.0": (9, 16, 256, 0, 0, 18, 32, 128, 1),   # plain t, in2 = the bordered layer2 output
    "layer4.0": (5, 8, 512, 0, 0, 9, 16, 256, 0),     # everything plain
}


@pytest.mark.parametrize("B", [1, 3, 17, 640])
@pytest.mark.parametrize("variant", list(SHORTCUTS))
def test_fused_shortcut_matches_fp64(variant, B):
    """relu(conv3x3(t) + conv1x1/s2(x) + (b2 + bd)) as one implicit GEMM whose last Cin2/64 k-blocks read x on its
    stride-2 sub-lattice (ConvArgs::in2)."""
    _lib, L = _L()
    H, W, C, in_pad, out_pad, H2, W2, C2, in2_pad = SHORTCUTS[variant]
    g = _gen(500 + 7 * B + C)
    t = _randn(g, B, C, H, W)
    x = _randn(g, B, C2, H2, W2)
    w2 = _randn(g, C, C, 3, 3, scale=(9 * C) ** -0.5)
    wd = _randn(g, C, C2, 1, 1, scale=C2 ** -0.5)
    b2 = _randn(g, C, scale=0.5, dtype=torch.float32)
    bd = _randn(g, C, scale=0.5, dtype=torch.float32)
    wf = torch.cat([_khwc(w2), _khwc(wd)], 1).contiguous()
    bf = b2 + bd
    tin = _bordered(_nhwc(t)) if in_pad else _nhwc(t)
    xin = _bordered(_nhwc(x)) if in2_pad else _nhwc(x)
    if out_pad:
        out = Guarded((B, H + 2, W + 2, C), BORDER)
        out.t[:, 1:-1, 1:-1] = 7.0
        got = out.t[:, 1:-1, 1:-1]
    else:
        out = Guarded((B, H, W, C), 7.0)
        got = out.t
    _call(L.cadre_conv2d_nhwc_shortcut, tin, B, H, W, C, wf, C, 3, 3, 1, bf, 1, out.t, in_pad, out_pad, xin, C2, H2, W2,
          in2_pad)
    torch.cuda.synchronize()
    out.check()
    if out_pad:
        assert _border_is(out.t, BORDER), "an out_pad convolution wrote into the border"
    ref, S = _conv_ref(t, w2, bf, 1, 1)
    ref_d, S_d = _conv_ref(x, wd, None, 2, 0)
    _check_bound("fused shortcut", got.permute(0, 3, 1, 2), (ref + ref_d).relu(), S + S_d, C_ACC["fused shortcut"])


# ------------------------------------------------------------------------------------------------ 6. linears
def _gemm_args(**kw):
    _lib, _ = _L()
    a = _lib.GemmArgs()
    a.alpha = 1.0
    for k, v in kw.items():
        setattr(a, k, v.data_ptr() if isinstance(v, torch.Tensor) else v)
    return a


@pytest.mark.parametrize("M", [1, 127, 128, 129, 640])
def test_fc1_and_fc2_match_fp64(M):
    """fc1: the persistent MODE_GEMM branch of launch_gemm (kind 0, N = 3072, K = 5120, LeakyReLU, fp16 out);
    fc2: the batched GEMM (batch 6, a_bs = 512, fp32 out). Rows >= M of the outputs stay untouched."""
    import ctypes
    _lib, L = _L()
    g = _gen(700 + M)
    A = _randn(g, M, 5120)
    W1 = _randn(g, 3072, 5120, scale=5120 ** -0.5)
    b1 = _randn(g, 3072, scale=0.5, dtype=torch.float32)
    h = Guarded((M + 128, 3072), 7.0)
    _lib.check(L.cadre_gemm(ctypes.byref(_gemm_args(kind=0, batch=1, M=M, N=3072, K=5120, A=A, lda=5120, B=W1, ldb=5120,
                                                    out=h.t, ldc=3072, out_f32=0, bias=b1, act=2)),
                            _lib.stream_ptr()))
    torch.cuda.synchronize()
    h.check()
    assert bool((h.t[M:] == 7.0).all()), "fc1 wrote rows >= M"
    pre = A.double() @ W1.double().t() + b1.double()
    ref = torch.where(pre > 0, pre, pre * float(np.float32(0.01)))    # the fp32 slope LeakyReLU(0.01) multiplies by
    S = A.double().abs() @ W1.double().abs().t() + b1.double().abs()
    _check_bound("fc1 (persistent GEMM)", h.t[:M], ref, S, C_ACC["fc1 (persistent GEMM)"])

    fc1 = h.t[:M].contiguous()
    W2 = _randn(g, 6, 256, 512, scale=512 ** -0.5)
    b2 = _randn(g, 6, 256, scale=0.5, dtype=torch.float32)
    q = Guarded((6, M, 256), 7.0, dtype=torch.float32)
    _lib.check(L.cadre_gemm(ctypes.byref(_gemm_args(kind=0, batch=6, M=M, N=256, K=512, A=fc1, lda=3072, a_bs=512,
                                                    B=W2, ldb=512, b_bs=256 * 512, out=q.t, ldc=256, out_bs=M * 256,
                                                    out_f32=1, bias=b2, bias_bs=256)),
                            _lib.stream_ptr()))
    torch.cuda.synchronize()
    q.check()
    a3 = fc1.double().view(M, 6, 512).transpose(0, 1)
    ref = torch.bmm(a3, W2.double().transpose(1, 2)) + b2.double()[:, None]
    S = torch.bmm(a3.abs(), W2.double().abs().transpose(1, 2)) + b2.double().abs()[:, None]
    _check_bound("fc2 (batched GEMM, fp32 out)", q.t, ref, S, C_ACC["fc2 (batched GEMM, fp32 out)"], u_out=U32)


# ------------------------------------------------------------------------------------------------ 7. attention tail
def _frame_rel(name, got, ref):
    """per-frame rel-L2 and worst |element error| / frame rms against the STAGE_REL bounds."""
    B = got.shape[0]
    d = (got.double() - ref).reshape(B, -1)
    rf = ref.reshape(B, -1)
    rms = rf.pow(2).mean(1).sqrt()
    rel = float((d.norm(dim=1) / rf.norm(dim=1)).max())
    el = float((d.abs().max(1).values / rms).max())
    _note("stage " + name, frame_rel_l2=rel, worst_elem_over_rms=el)
    assert rel < STAGE_REL[name][0] and el < STAGE_REL[name][1], f"{name}: per-frame rel-L2 {rel:.3g}, worst / rms {el:.3g}"


@pytest.mark.parametrize("B,max_batch", [(1, 640), (297, 640), (640, 640), (1024, 1024)])
def test_attention_tail_stages_from_the_forwards_own_inputs(enc, B, max_batch):
    """Each stage after layer4 from the CUDA's own fp16 input (the previous debug buffer), against the oracle on float64
    copies of the state dict: layer4 -> conv5a|5c -> PAM / CAM -> feat_sum -> fc1 -> latent. B = 297 runs PAM's frame
    loop (> 2 x 148 frames), B = 1024 CAM's (> 6 x 148). Stages with folded fp16 weights are bounded element-wise with
    c = 2^-11 (the weight rounding) + C_ACC (+ 2^-11 for feat_sum's fp16 sa_conv); PAM, CAM and the latent by STAGE_REL."""
    from cadre_b200.encoder import Encoder, prepare_weights
    sd = R.danet_fixture_state(0)
    e = enc if max_batch == 640 else Encoder(sd, "cuda:0", max_batch=max_batch)
    x = torch.rand(B, 4, 144, 256, device="cuda", generator=_gen(900 + B))
    lat = e.forward_f32(x).double()
    sd64 = {k: v.double().cuda() for k, v in sd.items()}
    fw = prepare_weights(sd, "cuda", torch.float64, check_range=False)   # folded weights, for the scale S

    def nchw(buf, c):
        return e.debug_buffer(buf, B).view(B, 5, 8, c).permute(0, 3, 1, 2).double()

    def folded(name, cin):
        return fw[name + "_w"].view(-1, 3, 3, cin).permute(0, 3, 1, 2), fw[name + "_b"]

    c_w = U16 + C_ACC["stage"]
    l4, h5, sa, sc, fs = nchw(0, 512), nchw(2, 256), nchw(3, 128), nchw(4, 128), nchw(1, 128)
    with torch.no_grad():
        ref = torch.cat([R._conv_bn_relu(l4, sd64, "da_head.conv5a"), R._conv_bn_relu(l4, sd64, "da_head.conv5c")], 1)
        _, S = _conv_ref(l4, *folded("head5", 512), 1, 1)
        _check_bound("stage layer4 -> conv5a|5c", h5, ref, S, c_w)

        _frame_rel("PAM", sa, R.pam(h5[:, :128], sd64))
        _frame_rel("CAM", sc, R.cam(h5[:, 128:], sd64))

        ref = R._conv_bn_relu(sa, sd64, "da_head.conv51") + R._conv_bn_relu(sc, sd64, "da_head.conv52")
        S = _conv_ref(sa, *folded("conv51", 128), 1, 1)[1] + _conv_ref(sc, *folded("conv52", 128), 1, 1)[1]
        _check_bound("stage PAM, CAM -> feat_sum", fs, ref, S, c_w + U16)

        da = F.conv2d(fs, sd64["da_head.conv8.1.weight"], sd64["da_head.conv8.1.bias"])
        hid, outs = [], []
        for task, conv in (("visual", "visual_conv"), ("bc", "bc_conv")):
            t = F.conv2d(da, sd64[conv + ".weight"], sd64[conv + ".bias"]).reshape(B, -1)
            for role in ("query", "key", "value"):
                p = f"inter_task_att.{task}_{role}_layer"
                hid.append(F.leaky_relu(F.linear(t, sd64[p + ".1.weight"], sd64[p + ".1.bias"]), 0.01))
                outs.append(p)
        fs_flat = e.debug_buffer(1, B).view(B, 5120).double()
        S = fs_flat.abs() @ fw["fc1_w"].abs().t() + fw["fc1_b"].abs()
        fc1 = e.debug_buffer(5, B).view(B, 3072).double()
        _check_bound("stage feat_sum -> fc1", fc1, torch.cat(hid, 1), S, c_w)

        qkv = [F.linear(fc1[:, 512 * i:512 * (i + 1)], sd64[p + ".3.weight"], sd64[p + ".3.bias"])
               for i, p in enumerate(outs)]
        av, ab = R.inter_task_attend(*qkv)
        _frame_rel("fc1 -> latent", lat, torch.cat([av, ab], 1))


# ------------------------------------------------------------------------------------------------ 8. replay
def _replay_backbone(t, xp, B):
    """encoder_trunk up to layer4 through the operator entry points, with the plan's arguments and weights (the
    shortcut weights appended along K and the biases summed, as encoder_create does)."""
    _, L = _L()

    def z(*shape):
        return torch.zeros(*shape, device="cuda", dtype=torch.float16)

    def w(i):
        return t[f"conv_w{i}"]

    def b(i):
        return t[f"conv_b{i}"]

    def fused(i):
        return torch.cat([w(i), w(i + 1)], 1).contiguous(), b(i) + b(i + 1)

    x = z(B, 38, 66, 64)
    _call(L.cadre_stem_pool, xp, B, t["stem_w"], t["stem_b"], x)
    for bi in range(2):                               # layer1: flat 3x3 kernel on bordered activations
        h, o = z(B, 38, 66, 64), z(B, 38, 66, 64)
        _call(L.cadre_conv3x3_flat64, x, B, 36, 64, w(2 * bi), b(2 * bi), None, 1, h)
        _call(L.cadre_conv3x3_flat64, h, B, 36, 64, w(2 * bi + 1), b(2 * bi + 1), x, 1, o)
        x = o
    t0, y0, t1, y1 = (z(B, 20, 34, 128) for _ in range(4))   # layer2 on bordered activations
    _call(L.cadre_conv2d_nhwc_bordered_out, x, B, 36, 64, 64, w(4), 128, 3, 3, 2, 1, b(4), 1, t0, 1)
    wf, bf = fused(5)
    _call(L.cadre_conv2d_nhwc_shortcut, t0, B, 18, 32, 128, wf, 128, 3, 3, 1, bf, 1, y0, 1, 1, x, 64, 36, 64, 1)
    _call(L.cadre_conv3x3_flat128, y0, B, 18, 32, w(7), b(7), None, 1, t1)
    _call(L.cadre_conv3x3_flat128, t1, B, 18, 32, w(8), b(8), y0, 1, y1)
    x, H, W, C, in_pad = y1, 18, 32, 128, 1
    for li, ci in ((3, 9), (4, 14)):                  # layers 3 and 4 on plain activations
        Co, Ho, Wo = 2 * C, (H - 1) // 2 + 1, (W - 1) // 2 + 1
        a, y = z(B, Ho, Wo, Co), z(B, Ho, Wo, Co)
        _call(L.cadre_conv2d_nhwc, x, B, H, W, C, w(ci), Co, 3, 3, 2, 1, b(ci), None, 0, 1, a, in_pad)
        wf, bf = fused(ci + 1)
        _call(L.cadre_conv2d_nhwc_shortcut, a, B, Ho, Wo, Co, wf, Co, 3, 3, 1, bf, 1, y, 0, 0, x, C, H, W, in_pad)
        a2, y2 = z(B, Ho, Wo, Co), z(B, Ho, Wo, Co)
        _call(L.cadre_conv2d_nhwc, y, B, Ho, Wo, Co, w(ci + 3), Co, 3, 3, 1, 1, b(ci + 3), None, 0, 1, a2, 0)
        _call(L.cadre_conv2d_nhwc, a2, B, Ho, Wo, Co, w(ci + 4), Co, 3, 3, 1, 1, b(ci + 4), y, 0, 1, y2, 0)
        x, H, W, C, in_pad = y2, Ho, Wo, Co, 0
    torch.cuda.synchronize()
    return x


@pytest.mark.parametrize("B", [3, 640])
def test_backbone_replay_through_operator_entry_points_is_bit_identical(enc, B):
    """Ties the operator tests above to the arguments the plan really passes: stem -> 4 x flat64 -> layer2 (bordered
    out, fused shortcut, 2 x flat128) -> layers 3 / 4, from the ingested image, equals the encoder's layer4 output bit
    for bit."""
    rgb, route = _u8_frames(B, seed=400 + B)
    enc.forward_u8(rgb.cuda(), route.cuda())
    l4 = enc.debug_buffer(0, B)
    got = _replay_backbone(enc._t, enc.debug_buffer(6, B), B)
    assert torch.equal(got.reshape(-1).view(torch.int16), l4.view(torch.int16))
