"""CPU check of the TF32 rounding model that tests/test_ppo_gemm_gpu.py uses as its reference for the tile GEMM."""
import importlib.util
import os

import numpy as np
import torch


def _gpu_module():
    path = os.path.join(os.path.dirname(os.path.abspath(__file__)), "test_ppo_gemm_gpu.py")
    spec = importlib.util.spec_from_file_location("_ppo_gemm_gpu_helpers", path)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def _tf32_bits(u, ties_away, ftz):
    """fp32 bits -> TF32 bits in fp32 storage, on the integer representation: drop the low 13 mantissa bits and round
    the kept part up on more than half, or on exactly half (0x1000) when ties go away from zero or the kept part is odd.
    A carry runs into the exponent (0x7F7FF000 -> inf); inf and NaN stay; subnormals go to signed zero under ftz."""
    u = np.asarray(u, dtype=np.uint32)
    sign, mag = u & np.uint32(0x80000000), u & np.uint32(0x7FFFFFFF)
    low, kept = mag & np.uint32(0x1FFF), mag & np.uint32(0x7FFFE000)
    odd = (kept >> np.uint32(13)) & np.uint32(1)
    up = (low > 0x1000) | ((low == 0x1000) & (bool(ties_away) | (odd == 1)))
    r = kept + np.where(up, np.uint32(0x2000), np.uint32(0))
    if ftz:
        r = np.where(mag < 0x00800000, np.uint32(0), r)
    r = np.where(mag >= 0x7F800000, mag, r)
    return (sign | r).astype(np.uint32)


def test_tf32_round_matches_a_bit_level_model():
    """tf32_round (float64 quantum arithmetic) against the integer model above, for the rounding the GPU tests
    measured and for the other three tie / subnormal choices, on the constructed ties, neighbours and subnormals of
    the readouts and on random bit patterns of every exponent."""
    m = _gpu_module()
    rs = np.random.RandomState(0)
    vals = np.concatenate([m.tf32_specials(), rs.randint(0, 2 ** 32, 200000, dtype=np.uint64).astype(np.uint32),
                           np.array([0, 0x80000000, 0x7F7FF000, 0x7F7FEFFF, 0x7F800000, 0xFF800000, 0x7FC00000],
                                    dtype=np.uint32)])
    measured = (m.TF32_TIES_AWAY, m.TF32_FTZ)
    try:
        for ties_away in (False, True):
            for ftz in (False, True):
                m.TF32_TIES_AWAY, m.TF32_FTZ = ties_away, ftz
                got = m.tf32_round(torch.from_numpy(vals.view(np.float32))).numpy().view(np.uint32)
                want = _tf32_bits(vals, ties_away, ftz)
                nan = np.isnan(vals.view(np.float32))
                assert np.array_equal(np.isnan(got.view(np.float32)), nan)
                bad = np.nonzero((got != want) & ~nan)[0]
                assert bad.size == 0, (ties_away, ftz, [(f"{vals[i]:08x}", f"{got[i]:08x}", f"{want[i]:08x}")
                                                        for i in bad[:8]])
    finally:
        m.TF32_TIES_AWAY, m.TF32_FTZ = measured
    # the constructed values separate the two tie rules and flushing from keeping subnormals
    sp = m.tf32_specials()
    assert not np.array_equal(_tf32_bits(sp, False, False), _tf32_bits(sp, True, False))
    assert not np.array_equal(_tf32_bits(sp, False, False), _tf32_bits(sp, False, True))
