"""The tile GEMM of the PPO update, through the public `cadre_gemm` entry point, one instantiation and call site at a time.

1. Readouts. One operand is a 0/1 selection matrix with exactly one 1.0 per output row, so every output element is one
   element of the other operand after the kernel's operand conversion (TF32 rounding by the TFLOAT32 tensor maps, or
   none for fp16). The whole output allocation is compared bit for bit: every swizzle atom, MN-major chunk, descriptor,
   batch offset, M / N / K tail and the untouched guard and padding around the output.
2. The update's own call sites (csrc/ppo.cu ppo_forward / ppo_update) with their majors, shapes, leading dimensions,
   batch strides, bias, activation, mask, per-expert row counts and alpha, at the capacities of a tiny run, cfg 3 and
   cfg 5. The reference is the same operation in float64 on the device, on the operands as the kernel sees them
   (TF32-rounded by `tf32_round`, or fp16 exactly), element by element:

       |got - ref| <= u_out * |ref| + 2^-24 + c * S,     S = the same operation on |operands| (+ |bias| ...)

   u_out = 2^-24 for fp32 outputs (2^-11 for fp16). c covers the fp32 accumulation and is set from the measured worst
   value with a margin of about 4x (`C_ACC`). It stays far below what a defect costs: a missing k-block of 32 terms
   changes an element by about sqrt(32) / K of S's scale (> 1e-2 S at K = 530), a missing bias by |b| (S is O(10)
   with |b| ~ 0.5), a missing expert row leaves the sentinel behind, and TF32 truncation instead of rounding biases
   every product by about 2^-11 (> 2^-12 S summed over K).
3. Contracts: rows [count, min(M, ceil(count / 128) * 128)) are written as +0.0 and rows beyond are left alone (count
   0 writes nothing); NaN in A rows >= count, in the K rows >= ceil(count / BK) * BK of `rows_is_k` operands and in
   every padding column never reaches an output; the ReLU-backward mask zeroes exactly where !(mask > 0); a count
   above M writes nothing past row M; an undispatched combination is an error and launches nothing.
"""
import ctypes
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
U16 = 2.0 ** -11          # fp16 round-to-nearest, relative
U32 = 2.0 ** -24          # fp32 round-to-nearest, relative
TINY = 2.0 ** -24         # absolute floor
GUARD = 8192              # sentinel elements in front of and behind every output (at least 128 rows more behind)
SENTINEL = -1234.0        # exact in fp16 and fp32

# TF32 conversion of the TFLOAT32 tensor maps, measured on a B200 with the readouts below: round to nearest with
# ties to even, and fp32 subnormals are kept (not flushed to zero).
TF32_TIES_AWAY = False
TF32_FTZ = False

# fp32 accumulation term c of the bound, per call site: the measured worst c (B200, every cap and branch) times about 4
C_ACC = {
    "x-part": 2.0 ** -19,          # measured 3.6e-7
    "W1": 2.0 ** -19,              # measured 5.7e-7
    "W2": 2.0 ** -20,              # measured 2.9e-7
    "dZ1": 2.0 ** -20,             # measured 2.9e-7
    "dW2": 2.0 ** -18,             # measured 9.0e-7 (K = cap)
    "dW1": 2.0 ** -18,             # measured 9.4e-7 (K = cap)
    "dh_8": 2.0 ** -19,            # measured 3.6e-7
    "LSTM wgrad": 2.0 ** -17,      # measured 1.4e-6 (K = 9 cap, up to 28 800)
    "mask": 2.0 ** -20,            # measured 2.6e-7
    "epilogue fp16": 2.0 ** -21,   # measured 1.1e-7
    "count above M": 2.0 ** -19,   # measured 4.1e-7
}

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


def _gen(seed):
    return torch.Generator(device="cuda").manual_seed(seed)


def tf32_round(x):
    """fp32 -> the value a TFLOAT32 tensor map hands the tensor core: 10 stored mantissa bits, fp32's exponent range.
    Round to nearest (ties per TF32_TIES_AWAY), subnormals flushed when TF32_FTZ; inf / NaN pass through."""
    d = x.double()
    _, e = torch.frexp(d)                                    # d = m 2^e, 0.5 <= |m| < 1
    q = ((e.clamp_min(-125).long() - 11 + 1023) << 52).view(torch.float64)   # TF32 quantum 2^(e-11), >= 2^-136
    y = d / q
    r = torch.copysign(torch.floor(y.abs() + 0.5), y) if TF32_TIES_AWAY else torch.round(y)
    r = r * q
    if TF32_FTZ:
        r = torch.where(d.abs() < 2.0 ** -126, d * 0.0, r)
    return torch.where(torch.isfinite(d), r, d).float()


def tf32_specials():
    """fp32 bit patterns at the TF32 rounding decision: exact ties (low 13 bits 0x1000) with the kept bit even and
    odd, their neighbours, a tie that carries into the exponent, and subnormals; both signs."""
    v = []
    for e in (0x3F800000, 0x40400000, 0x3C000000, 0x00800000, 0x7E800000):
        for kept in (0, 0x2000):
            for low in (0x1000, 0x0FFF, 0x1001, 0x0000, 0x1FFF):
                v.append(e | 0x2A8000 | kept | low)
    v += [0x3FFFF000, 0x3F7FF000, 0x007FF000, 0x00000001, 0x00001000, 0x00003000, 0x00000FFF, 0x00400000, 0x007FFFFF]
    v = np.array(v, dtype=np.uint32)
    return np.concatenate([v, v | np.uint32(0x80000000)])


def _view(flat, off, batch, rows, cols, bs, ld, col_major=False):
    """logical [batch, rows, cols] view of flat storage: element (b, r, c) at off + b*bs + r*ld + c (or + c*ld + r)."""
    st = (bs, 1, ld) if col_major else (bs, ld, 1)
    return flat.as_strided((batch, rows, cols), st, flat.storage_offset() + off)


def _operand(batch, rows, K, mn, ld, bs, dtype, off=0):
    """Storage of an operand, logical [batch, rows(M|N), K], K-major or MN-major, NaN everywhere outside the logical
    tensor (padding columns, batch gaps, the other half of a shared buffer): the kernel must never read it."""
    stored_rows, width = (K, rows) if mn else (rows, K)
    assert width <= ld
    flat = torch.full((off + (batch - 1) * bs + stored_rows * ld,), float("nan"), dtype=dtype, device="cuda")
    return flat, _view(flat, off, batch, rows, K, bs, ld, col_major=mn)


class Out:
    """Output storage inside one allocation of SENTINEL with guard regions; `mark` records what may be written."""

    def __init__(self, batch, M, N, ldc, out_bs, dtype, off=0):
        self.guard = max(GUARD, 128 * ldc)
        span = off + (batch - 1) * out_bs + M * ldc
        self.buf = torch.full((2 * self.guard + span,), SENTINEL, dtype=dtype, device="cuda")
        self.t = _view(self.buf[self.guard:], off, batch, M, N, out_bs, ldc)
        self.may = torch.zeros(self.buf.shape, dtype=torch.bool, device="cuda")
        self.may_t = _view(self.may[self.guard:], off, batch, M, N, out_bs, ldc)

    def check_untouched(self):
        """Everything not marked is still SENTINEL: guards, padding columns, batch gaps, rows nobody may write."""
        bad = (~self.may) & (self.buf != SENTINEL)
        n = int(bad.sum())
        if n:
            i = int(bad.nonzero()[0]) - self.guard
            raise AssertionError(f"{n} elements written outside the output contract, first at offset {i}")


def _gemm(**kw):
    """cadre_gemm with alpha 1 and batch 1 unless given; returns (rc, message)."""
    _lib, L = _L()
    a = _lib.GemmArgs()
    a.alpha, a.batch = 1.0, 1
    for k, v in kw.items():
        setattr(a, k, v.data_ptr() if isinstance(v, torch.Tensor) else v)
    rc = L.cadre_gemm(ctypes.byref(a), _lib.stream_ptr())
    return rc, (L.cadre_last_error().decode() if rc else "")


def _run(**kw):
    rc, msg = _gemm(**kw)
    assert rc == 0, msg
    torch.cuda.synchronize()


def _check_bound(name, got, ref, S, c, u_out=U32):
    """|got - ref| <= u_out |ref| + 2^-24 + c S element by element; records the worst err / bound and the c needed."""
    got = got.double()
    assert bool(torch.isfinite(got).all()), f"{name}: non-finite output"
    err = (got - ref).abs()
    bound = u_out * ref.abs() + TINY + c * S
    ratio = err / bound
    worst = float(ratio.max()) if ratio.numel() else 0.0
    need = float(((err - u_out * ref.abs() - TINY) / S.clamp_min(1e-300)).max().clamp_min(0.0)) if err.numel() else 0.0
    _note(name, err_over_bound=worst, c_needed=need)
    if worst > 1.0:
        i = int(ratio.flatten().argmax())
        idx = np.unravel_index(i, tuple(ratio.shape))
        raise AssertionError(f"{name}: worst err/bound {worst:.3g} at {idx}: got {got.flatten()[i].item():.6g}, "
                             f"ref {ref.flatten()[i].item():.6g}, S {S.flatten()[i].item():.4g} (c needed {need:.3g})")


def _bits(t):
    return t.view(torch.int32) if t.dtype == torch.float32 else t.view(torch.int16)


# ------------------------------------------------------------------------------------------------ 1. readouts
# every CADRE_GEMM_CASE of launch_gemm: (kind, a_mn, b_mn, block_n, out_f32), plus the two persistent MODE_GEMM
# branches (kind 0, K-major, batch 1, fp16 out, N % 8 == 0: block 64 for N <= 64, 128 above)
TILE_CASES = {
    "fp16-KK-bn64-h": (0, 0, 0, 64, 0),
    "fp16-KK-bn128-h": (0, 0, 0, 128, 0),
    "fp16-KK-bn64-f": (0, 0, 0, 64, 1),
    "fp16-KK-bn128-f": (0, 0, 0, 128, 1),
    "fp16-K/MN-f": (0, 0, 1, 128, 1),
    "fp16-MN/MN-f": (0, 1, 1, 128, 1),
    "tf32-KK-bn64": (1, 0, 0, 64, 1),
    "tf32-KK-bn128": (1, 0, 0, 128, 1),
    "tf32-K/MN": (1, 0, 1, 128, 1),
    "tf32-MN/MN": (1, 1, 1, 128, 1),
    "persistent-bn64": (0, 0, 0, 0, 0),
    "persistent-bn128": (0, 0, 0, 0, 0),
}
READOUTS = [(c, w) for c in TILE_CASES for w in ("A", "B")]


def _readout_operand(g, shape, kind):
    """random operand values, none of them zero; TF32 operands carry every special of tf32_specials()."""
    x = torch.randn(*shape, device="cuda", generator=g) * 3.0
    if kind:
        x = x + torch.rand(*shape, device="cuda", generator=g) * 1e-3      # full 23-bit mantissas
        sp = torch.from_numpy(tf32_specials().view(np.float32)).cuda()
        flat = x.view(-1)
        pos = torch.randperm(flat.numel(), device="cuda", generator=g)[:4 * sp.numel()]
        flat[pos] = sp.repeat(4)
        return x
    x = x.half()
    return torch.where(x == 0, torch.ones_like(x), x)


@pytest.mark.parametrize("case,which", READOUTS, ids=[f"{c}-{w}" for c, w in READOUTS])
def test_readout_is_bit_exact(case, which):
    """out = A * B^T with B (or A) a selection matrix: out[b, m, n] = conv(A[b, m, sel_b[n]]) (or conv(B[b, n,
    sel_b[m]])), bit for bit, and nothing else of the output allocation changes. M = 300, N = 530, K = 530 leave a tail
    in every dimension; batch 3 with batch strides larger than the tensors."""
    kind, a_mn, b_mn, block_n, out_f32 = TILE_CASES[case]
    persistent = case.startswith("persistent")
    batch = 1 if persistent else 3
    M, K = 300, 530
    N = {"persistent-bn64": 56, "persistent-bn128": 520}.get(case, 530)
    dt = torch.float32 if kind else torch.float16
    odt = torch.float32 if out_f32 else torch.float16
    lda = 304 if a_mn else 536
    ldb = 536 if b_mn else 544
    ldc = {"persistent-bn64": 64, "persistent-bn128": 528}.get(case, 536)
    a_bs, b_bs, out_bs = (K if a_mn else M) * lda + 64, (K if b_mn else N) * ldb + 32, M * ldc + 128
    g = _gen(2 * list(TILE_CASES).index(case) + (which == "B"))
    A_flat, A = _operand(batch, M, K, a_mn, lda, a_bs, dt)
    B_flat, B = _operand(batch, N, K, b_mn, ldb, b_bs, dt)
    perm = [torch.randperm(K, device="cuda", generator=g) for _ in range(batch)]
    if which == "A":
        A.copy_(_readout_operand(g, (batch, M, K), kind))
        B.zero_()
        for b in range(batch):
            B[b, torch.arange(N, device="cuda"), perm[b][:N]] = 1.0
        src = tf32_round(A) if kind else A
        want = torch.stack([src[b][:, perm[b][:N]] for b in range(batch)])
    else:
        B.copy_(_readout_operand(g, (batch, N, K), kind))
        A.zero_()
        for b in range(batch):
            A[b, torch.arange(M, device="cuda"), perm[b][:M]] = 1.0
        src = tf32_round(B) if kind else B
        want = torch.stack([src[b][:, perm[b][:M]].t() for b in range(batch)])
    out = Out(batch, M, N, ldc, out_bs, odt)
    kw = {}
    if persistent:    # the persistent branch requires a bias vector: +0.0 leaves every readout value unchanged
        kw["bias"] = torch.zeros(N, device="cuda")
    _run(kind=kind, a_mn=a_mn, b_mn=b_mn, batch=batch, M=M, N=N, K=K, block_n=block_n, A=A_flat, lda=lda, a_bs=a_bs,
         B=B_flat, ldb=ldb, b_bs=b_bs, out=out.t, ldc=ldc, out_bs=out_bs, out_f32=out_f32, **kw)
    exp = out.buf.clone()
    _view(exp[out.guard:], 0, batch, M, N, out_bs, ldc).copy_(want.to(odt))
    got_b, exp_b = _bits(out.buf), _bits(exp)
    # a value that converts to zero may come back as either zero (the selection sum of +-0 products)
    same = (got_b == exp_b) | ((out.buf == 0) & (exp == 0))
    n_bad = int((~same).sum())
    if n_bad:
        i = int((~same).nonzero()[0])
        raise AssertionError(f"readout mismatch: {n_bad} elements differ, first at offset {i - out.guard}: got "
                             f"{int(got_b[i]) & 0xFFFFFFFF:#010x}, want {int(exp_b[i]) & 0xFFFFFFFF:#010x}")


def test_tf32_specials_read_out_as_the_rounding_helper_says():
    """The constructed ties, neighbours and subnormals, one per output element of a K-major TF32 readout: the kernel
    agrees with tf32_round, and tf32_round is not truncation (so the readouts above pin the rounding)."""
    sp = torch.from_numpy(tf32_specials().view(np.float32)).cuda()
    n = sp.numel()
    K = (n + 31) // 32 * 32
    A = torch.ones(128, K, device="cuda")
    A[0, :n] = sp
    I = torch.eye(K, device="cuda")
    out = torch.full((128, K), SENTINEL, device="cuda")
    _run(kind=1, M=128, N=K, K=K, A=A, lda=K, B=I, ldb=K, out=out, ldc=K, out_f32=1)
    got, want = out[0, :n], tf32_round(sp)
    same = (_bits(got) == _bits(want)) | ((got == 0) & (want == 0))
    assert bool(same.all()), [(f"{int(v):08x}", f"{int(r) & 0xFFFFFFFF:08x}")
                              for v, r, s in zip(tf32_specials(), _bits(got).tolist(), same.tolist()) if not s]
    trunc = (_bits(sp) & ~0x1FFF).view(torch.float32)
    assert not bool((_bits(want) == _bits(trunc)).all())


def test_tf32_truncation_is_detected():
    """CADRE_TF32_TRUNCATE=1 (plain FLOAT32 tensor maps: the tensor core truncates) makes the TF32 readout fail."""
    test_id = f"{os.path.abspath(__file__)}::test_readout_is_bit_exact[tf32-KK-bn128-A]"
    cmd = [sys.executable] + (["-s"] if sys.flags.no_user_site else []) + [
        "-m", "pytest", "-q", "-p", "no:cacheprovider", test_id]
    r = subprocess.run(cmd, cwd=ROOT, env=dict(os.environ, CADRE_TF32_TRUNCATE="1"), capture_output=True, text=True,
                       timeout=600)
    assert r.returncode == 1 and "readout mismatch" in r.stdout, r.stdout[-3000:] + r.stderr[-3000:]


# ------------------------------------------------------------------------------------------------ 2. call sites
E, F, LDF, G, HID = 8, 530, 532, 2120, 128
LDH16, LDG16 = 544, 2176
LSTM_BLK = 2 * G * LDF + 2 * G
CAPS = [128, 512, 3200]      # one 128-row tile; cfg 3; cfg 5


def _site(name, cap):
    """cadre_gemm arguments of one ppo.cu call site (offsets are element offsets into the buffer the pointer points
    into); `rows`: 'm' for batch_rows, 'k' for rows_is_k, with the per-expert count multiplied by `rmul`."""
    base, _, arg = name.partition("/")
    br = int(arg) if base in ("W2", "dZ1", "dW2") else 0
    bs256 = cap * 2 * HID
    if base == "x-part":       # XP9 = X W_ih^T + (b_ih + b_hh), fp16 operands, 9 time slots per row
        return dict(kind=0, a_mn=0, b_mn=0, batch=E, M=9 * cap, N=G, K=F, lda=LDH16, a_bs=9 * cap * LDH16, ldb=LDH16,
                    b_bs=G * LDH16, ldc=G, out_bs=9 * cap * G, bias_bs=G, rows="m", rmul=9)
    if base == "W1":           # Y1 = relu(h_8 W1^T + b1), actor and critic in one N = 256 GEMM
        return dict(kind=1, a_mn=0, b_mn=0, batch=E, M=cap, N=2 * HID, K=F, lda=LDF, a_bs=cap * LDF, ldb=LDF,
                    b_bs=2 * HID * LDF, ldc=2 * HID, out_bs=bs256, bias_bs=2 * HID, act=1, rows="m")
    if base == "W2":           # Y2 = relu(Y1 W2^T + b2) per branch, A = Y1 + 128 br
        return dict(kind=1, a_mn=0, b_mn=0, batch=E, M=cap, N=HID, K=HID, a_off=HID * br, lda=2 * HID, a_bs=bs256,
                    b_off=br * HID * HID, ldb=HID, b_bs=2 * HID * HID, out_off=HID * br, ldc=2 * HID, out_bs=bs256,
                    bias_off=HID * br, bias_bs=2 * HID, act=1, rows="m")
    if base == "dZ1":          # dZ1 = (dZ2 W2) * relu'(Y1)
        return dict(kind=1, a_mn=0, b_mn=1, batch=E, M=cap, N=HID, K=HID, a_off=HID * br, lda=2 * HID, a_bs=bs256,
                    b_off=br * HID * HID, ldb=HID, b_bs=2 * HID * HID, out_off=HID * br, ldc=2 * HID, out_bs=bs256,
                    mask_off=HID * br, ldm=2 * HID, mask_bs=bs256, rows="m")
    if base == "dW2":          # dW2 = dZ2^T Y1
        return dict(kind=1, a_mn=1, b_mn=1, batch=E, M=HID, N=HID, K=cap, a_off=HID * br, lda=2 * HID, a_bs=bs256,
                    b_off=HID * br, ldb=2 * HID, b_bs=bs256, out_off=br * HID * HID, ldc=HID, out_bs=2 * HID * HID,
                    rows="k")
    if base == "dW1":          # dW1 = dZ1^T h_8
        return dict(kind=1, a_mn=1, b_mn=1, batch=E, M=2 * HID, N=F, K=cap, lda=2 * HID, a_bs=bs256, ldb=LDF,
                    b_bs=cap * LDF, ldc=LDF, out_bs=2 * HID * LDF, rows="k")
    if base == "dh_8":         # dh_8 = dZ1 W1
        return dict(kind=1, a_mn=0, b_mn=1, batch=E, M=cap, N=F, K=2 * HID, lda=2 * HID, a_bs=bs256, ldb=LDF,
                    b_bs=2 * HID * LDF, ldc=LDF, out_bs=cap * LDF, rows="m")
    if base == "LSTM wgrad":   # dW_hh = dG^T H (fp16, K = 9 rows per sample), one grad group of `arg` experts
        return dict(kind=0, a_mn=1, b_mn=1, batch=int(arg), M=G, N=F, K=9 * cap, lda=LDG16, a_bs=9 * cap * LDG16,
                    ldb=LDH16, b_bs=9 * cap * LDH16, out_off=G * LDF, ldc=LDF, out_bs=LSTM_BLK, alpha=2.0 ** -10,
                    rows="k", rmul=9)
    raise KeyError(name)


SITES = ["x-part", "W1", "W2/0", "W2/1", "dZ1/0", "dZ1/1", "dW2/0", "dW2/1", "dW1", "dh_8",
         "LSTM wgrad/8", "LSTM wgrad/4", "LSTM wgrad/2", "LSTM wgrad/1"]


def _counts(cap, bk, rot, n):
    """n per-expert row counts from {0, 1, BK-1, BK, BK+1, 127, 128, 129, cap} (those <= cap), rotated by `rot`."""
    vals = []
    for v in (0, 1, bk - 1, bk, bk + 1, 127, 128, 129, cap):
        if v <= cap and v not in vals:
            vals.append(v)
    vals = vals[rot % len(vals):] + vals[:rot % len(vals)]
    return [vals[i % len(vals)] for i in range(n)]


def _conv(x, kind):
    return tf32_round(x).double() if kind else x.double()


def _gemm_check(name, s, counts, seed, mask_values=None):
    """Run one call site with synthetic operands that follow the caller contract, and check it against float64."""
    kind, batch, M, N, K = s["kind"], s["batch"], s["M"], s["N"], s["K"]
    rows, rmul = s.get("rows"), s.get("rmul", 1)
    bk = 32 if kind else 64
    dt = torch.float32 if kind else torch.float16
    g = _gen(seed)
    A_flat, A = _operand(batch, M, K, s["a_mn"], s["lda"], s["a_bs"], dt, s.get("a_off", 0))
    B_flat, B = _operand(batch, N, K, s["b_mn"], s["ldb"], s["b_bs"], dt, s.get("b_off", 0))
    A.copy_(torch.randn(batch, M, K, device="cuda", generator=g).to(dt))
    B.copy_((torch.randn(batch, N, K, device="cuda", generator=g) * K ** -0.5).to(dt))
    cnt = [c * rmul for c in counts] if rows else None
    for b in range(batch):
        if rows == "m":            # rows >= count: whatever the buffer holds; NaN must not reach an output
            A[b, cnt[b]:] = float("nan")
        elif rows == "k":          # K rows up to the next BK multiple are zero (caller contract), beyond never read
            kz = min(K, -(-cnt[b] // bk) * bk)
            A[b, :, cnt[b]:kz] = 0.0
            B[b, :, cnt[b]:kz] = 0.0
            A[b, :, kz:] = float("nan")
            B[b, :, kz:] = float("nan")
    kw = dict(kind=kind, a_mn=s["a_mn"], b_mn=s["b_mn"], batch=batch, M=M, N=N, K=K, block_n=s.get("block_n", 128),
              A=A_flat[s.get("a_off", 0):], lda=s["lda"], a_bs=s["a_bs"], B=B_flat[s.get("b_off", 0):], ldb=s["ldb"],
              b_bs=s["b_bs"], ldc=s["ldc"], out_bs=s["out_bs"], out_f32=1, act=s.get("act", 0),
              alpha=s.get("alpha", 1.0))
    bias = mask = None
    if "bias_bs" in s:
        bflat = torch.full((s.get("bias_off", 0) + (batch - 1) * s["bias_bs"] + N,), float("nan"), device="cuda")
        bias = _view(bflat, s.get("bias_off", 0), batch, 1, N, s["bias_bs"], N)[:, 0]
        bias.copy_(torch.randn(batch, N, device="cuda", generator=g) * 0.5)
        kw.update(bias=bflat[s.get("bias_off", 0):], bias_bs=s["bias_bs"])
    if "ldm" in s:
        mflat, mask = _operand(batch, M, N, 0, s["ldm"], s["mask_bs"], torch.float32, s.get("mask_off", 0))
        if mask_values is None:    # a post-ReLU activation: zeros and positives
            mask.copy_(torch.randn(batch, M, N, device="cuda", generator=g).relu())
        else:
            mv = torch.tensor(mask_values, device="cuda", dtype=torch.float32)
            mask.copy_(mv[torch.randint(0, len(mask_values), (batch, M, N), device="cuda", generator=g)])
        kw.update(mask=mflat[s.get("mask_off", 0):], ldm=s["ldm"], mask_bs=s["mask_bs"])
    if rows:
        rows_t = torch.tensor(cnt, dtype=torch.int32, device="cuda")
        kw.update(batch_rows=rows_t, rows_is_k=int(rows == "k"))
    out = Out(batch, M, N, s["ldc"], s["out_bs"], torch.float32, s.get("out_off", 0))
    kw["out"] = out.t
    _run(**kw)
    alpha = s.get("alpha", 1.0)
    for b in range(batch):
        rr = min(cnt[b], M) if rows == "m" else M
        kk = min(cnt[b], K) if rows == "k" else K
        a, bm = _conv(A[b, :rr, :kk], kind), _conv(B[b, :, :kk], kind)
        ref, S = alpha * (a @ bm.t()), alpha * (a.abs() @ bm.abs().t())
        if bias is not None:
            ref, S = ref + bias[b].double(), S + bias[b].double().abs()
        if s.get("act") == 1:
            ref = ref.clamp_min(0.0)
        got = out.t[b, :rr]
        if mask is not None:
            keep = mask[b, :rr] > 0
            assert bool((_bits(got)[~keep] == 0).all()), f"{name}: masked elements are not +0.0"
            ref = torch.where(keep, ref, torch.zeros_like(ref))
        _check_bound(name, got, ref, S, C_ACC[name.split("/")[0]])
        out.may_t[b, :rr] = True
        if rows == "m":            # the rest of the last tile is written as +0.0
            zend = min(M, -(-cnt[b] // 128) * 128)
            assert bool((_bits(out.t[b, rr:zend]) == 0).all()), f"{name}: rows [count, tile end) are not +0.0"
            out.may_t[b, rr:zend] = True
        if rows == "k" and cnt[b] == 0 and bias is None:
            assert bool((_bits(out.t[b]) == 0).all()), f"{name}: count 0 must give an exact +0.0 output"
    out.check_untouched()


@pytest.mark.parametrize("cap", CAPS)
@pytest.mark.parametrize("site", SITES)
def test_call_site_matches_fp64(site, cap):
    s = _site(site, cap)
    bk = 32 if s["kind"] else 64
    rot = SITES.index(site)
    counts = _counts(cap, bk, rot, E)
    if site.startswith("LSTM wgrad"):      # the last grad group: experts [E - batch, E)
        counts = counts[E - s["batch"]:]
    _gemm_check(site, s, counts, seed=100 * rot + cap)


# ------------------------------------------------------------------------------------------------ 3. contracts
MASK_VALUES = [0.0, -0.0, -1.5, -2.0 ** -149, 2.0 ** -149, 2.0 ** -126, 1e-30, 1.0, 3.0, float("nan")]


@pytest.mark.parametrize("N,ldc,ldm", [(128, 256, 256), (130, 132, 132), (130, 131, 132)],
                         ids=["fast", "N-tail", "general"])
def test_relu_backward_mask_zeroes_exactly_where_not_positive(N, ldc, ldm):
    """The dZ1 instantiation (TF32 K/MN) with mask values +0, -0, negatives, subnormal and tiny positives and NaN:
    outputs are +0.0 exactly where !(mask > 0) and match fp64 elsewhere, on the float4 path (N % 4 == 0), with an N
    tail (the last column group on the general path) and with every column on the general path (ldc odd)."""
    s = dict(kind=1, a_mn=0, b_mn=1, batch=3, M=300, N=N, K=128, lda=128, a_bs=300 * 128 + 32, ldb=132,
             b_bs=128 * 132, ldc=ldc, out_bs=300 * ldc + 4, ldm=ldm, mask_bs=300 * ldm + 8, rows="m")
    _gemm_check("mask", s, [300, 129, 1], seed=N + ldc, mask_values=MASK_VALUES)


@pytest.mark.parametrize("N,ldc,ldm", [(256, 256, 256), (130, 132, 132)], ids=["fast", "N-tail"])
def test_count_above_M_writes_nothing_past_M(N, ldc, ldm):
    """batch_rows = 310 for M = 300 (not a multiple of 128): rows [300, 384) of the last tile are past the output and
    must stay untouched (the guard behind the output holds 128 rows, so nothing lands outside the allocation). The
    fp32 mask sits in front of 128 spare rows as well."""
    g = _gen(5 + N)
    mflat = torch.ones(2 * 300 * ldm + 128 * ldm, device="cuda")     # 128 spare rows of 1.0 behind the mask
    mask = _view(mflat, 0, 2, 300, N, 300 * ldm, ldm)
    mask.copy_(torch.randn(2, 300, N, device="cuda", generator=g))
    A_flat, A = _operand(2, 300, 530, 0, 532, 300 * 532, torch.float32)
    B_flat, B = _operand(2, N, 530, 0, 532, N * 532, torch.float32)
    A.copy_(torch.randn(2, 300, 530, device="cuda", generator=g))
    B.copy_(torch.randn(2, N, 530, device="cuda", generator=g) * 530 ** -0.5)
    bias = torch.randn(2, N, device="cuda", generator=g) * 0.5
    out = Out(2, 300, N, ldc, 300 * ldc, torch.float32)
    rows = torch.tensor([300, 310], dtype=torch.int32, device="cuda")
    _run(kind=1, batch=2, M=300, N=N, K=530, block_n=128, A=A_flat, lda=532, a_bs=300 * 532, B=B_flat, ldb=532,
         b_bs=N * 532, out=out.t, ldc=ldc, out_bs=300 * ldc, out_f32=1, bias=bias, bias_bs=N, mask=mflat, ldm=ldm,
         mask_bs=300 * ldm, batch_rows=rows)
    for b in range(2):
        a, bm = tf32_round(A[b]).double(), tf32_round(B[b]).double()
        ref = a @ bm.t() + bias[b].double()
        S = a.abs() @ bm.abs().t() + bias[b].double().abs()
        keep = mask[b] > 0
        ref = torch.where(keep, ref, torch.zeros_like(ref))
        _check_bound("count above M", out.t[b], ref, S, C_ACC["count above M"])
    out.may_t[:] = True
    out.check_untouched()


@pytest.mark.parametrize("variant", ["res-before-relu", "res-after-relu", "leaky"])
def test_fp16_output_epilogue_residual_and_leaky_relu(variant):
    """The non-persistent fp16-output path (batch 2, N = 530) with what no PPO call uses but the C ABI offers: a
    residual added before or after the ReLU, and LeakyReLU(0.01)."""
    batch, M, N, K, ld = 2, 300, 530, 530, 536
    g = _gen(11 + len(variant))
    A_flat, A = _operand(batch, M, K, 0, ld, M * ld + 64, torch.float16)
    B_flat, B = _operand(batch, N, K, 0, ld, N * ld, torch.float16)
    A.copy_(torch.randn(batch, M, K, device="cuda", generator=g).half())
    B.copy_((torch.randn(batch, N, K, device="cuda", generator=g) * K ** -0.5).half())
    bias = torch.randn(batch, N, device="cuda", generator=g) * 0.5
    out = Out(batch, M, N, ld, M * ld + 8, torch.float16)
    kw = dict(kind=0, batch=batch, M=M, N=N, K=K, A=A_flat, lda=ld, a_bs=M * ld + 64, B=B_flat, ldb=ld, b_bs=N * ld,
              out=out.t, ldc=ld, out_bs=M * ld + 8, out_f32=0, bias=bias, bias_bs=N, act=2 if variant == "leaky" else 1)
    res = None
    if variant != "leaky":
        r_flat, res = _operand(batch, M, N, 0, 540, M * 540, torch.float16)
        res.copy_(torch.randn(batch, M, N, device="cuda", generator=g).half())
        kw.update(res=r_flat, ldr=540, res_bs=M * 540, res_after_act=int(variant == "res-after-relu"))
    _run(**kw)
    for b in range(batch):
        a, bm = A[b].double(), B[b].double()
        pre = a @ bm.t() + bias[b].double()
        S = a.abs() @ bm.abs().t() + bias[b].double().abs()
        if variant == "leaky":
            ref = torch.where(pre > 0, pre, pre * float(np.float32(0.01)))
        else:
            r = res[b].double()
            ref = (pre.relu() + r) if variant == "res-after-relu" else (pre + r).relu()
            S = S + r.abs()
        _check_bound("epilogue fp16", out.t[b], ref, S, C_ACC["epilogue fp16"], u_out=U16)
    out.may_t[:] = True
    out.check_untouched()


@pytest.mark.parametrize("kind,a_mn,b_mn,out_f32", [(1, 1, 0, 1), (1, 0, 0, 0), (0, 1, 0, 1)],
                         ids=["tf32-MN/K", "tf32-fp32-out-missing", "fp16-MN/K"])
def test_undispatched_combination_is_an_error_and_launches_nothing(kind, a_mn, b_mn, out_f32):
    dt = torch.float32 if kind else torch.float16
    A = torch.ones(256, 256, device="cuda", dtype=dt)
    B = torch.ones(256, 256, device="cuda", dtype=dt)
    out = Out(1, 256, 256, 256, 0, torch.float32 if out_f32 else torch.float16)
    rc, msg = _gemm(kind=kind, a_mn=a_mn, b_mn=b_mn, M=256, N=256, K=256, A=A, lda=256, B=B, ldb=256, out=out.t,
                    ldc=256, out_f32=out_f32)
    torch.cuda.synchronize()
    assert rc != 0 and "launch_gemm: unsupported" in msg, msg
    out.check_untouched()
