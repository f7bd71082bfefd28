"""CPU checks of the device-side rollout path: a numpy restatement of the counter-based categorical sampler
(Philox4x32-10 + the u / inverse-CDF rule of include/cadre_b200.h) against known-answer vectors, the ctypes mirror of
cadre_rollout_pool, and argument errors of the new entry points (error code + message, no crash, without a device)."""
import ctypes

import numpy as np
import pytest

PHILOX_M0, PHILOX_M1 = np.uint64(0xD2511F53), np.uint64(0xCD9E8D57)
PHILOX_W0, PHILOX_W1 = np.uint64(0x9E3779B9), np.uint64(0xBB67AE85)
MASK32 = np.uint64(0xFFFFFFFF)


def philox4x32_10(ctr, key):
    """Philox4x32-10 (Salmon et al., SC'11; Random123 / curand_Philox4x32_10) on arrays: ctr uint [..., 4],
    key uint [..., 2] -> uint32 [..., 4]."""
    c = [np.asarray(ctr, dtype=np.uint64)[..., i] & MASK32 for i in range(4)]
    k0 = np.asarray(key, dtype=np.uint64)[..., 0] & MASK32
    k1 = np.asarray(key, dtype=np.uint64)[..., 1] & MASK32
    for r in range(10):
        if r:
            k0, k1 = (k0 + PHILOX_W0) & MASK32, (k1 + PHILOX_W1) & MASK32
        p0, p1 = PHILOX_M0 * c[0], PHILOX_M1 * c[2]       # < 2^64: exact in uint64
        hi0, lo0 = p0 >> np.uint64(32), p0 & MASK32
        hi1, lo1 = p1 >> np.uint64(32), p1 & MASK32
        c = [hi1 ^ c[1] ^ k0, lo1, hi0 ^ c[3] ^ k1, lo0]
    return np.stack(c, -1).astype(np.uint32)


def sampler_uniform(seed, tick, env_ids, word):
    """u of the draw of environments env_ids (array) at `tick`, output word `word`: float32."""
    env_ids = np.asarray(env_ids, dtype=np.uint64)
    n = env_ids.shape[0]
    ctr = np.stack([np.full(n, tick & 0xFFFFFFFF, np.uint64), np.full(n, tick >> 32, np.uint64), env_ids,
                    np.zeros(n, np.uint64)], -1)
    key = np.tile(np.array([seed & 0xFFFFFFFF, seed >> 32], dtype=np.uint64), (n, 1))
    x = philox4x32_10(ctr, key)[:, word]
    return ((x >> np.uint32(8)).astype(np.float32) * np.float32(2.0 ** -24)).astype(np.float32)


def sampler_draw(lp, A, u):
    """The inverse-CDF rule in float32 with the kernel's order of operations: a = min{j : c_j > u c_{A-1}}, else
    max{j : p_j > 0}."""
    p = np.exp(np.asarray(lp[:A], dtype=np.float32)).astype(np.float32)
    c = np.float32(0)
    cs = []
    for j in range(A):
        c = np.float32(c + p[j])
        cs.append(c)
    t = np.float32(np.float32(u) * cs[-1])
    for j in range(A):
        if cs[j] > t:
            return j
    nz = np.nonzero(p > 0)[0]
    return int(nz[-1]) if nz.size else 0


@pytest.mark.parametrize("ctr,key,expect", [
    ((0, 0, 0, 0), (0, 0), (0x6627e8d5, 0xe169c58d, 0xbc57ac4c, 0x9b00dbd8)),
    ((0xffffffff,) * 4, (0xffffffff,) * 2, (0x408f276d, 0x41c83b0e, 0xa20bc7c6, 0x6d5451fd)),
    ((0x243f6a88, 0x85a308d3, 0x13198a2e, 0x03707344), (0xa4093822, 0x299f31d0),
     (0xd16cfe09, 0x94fdcceb, 0x5001e420, 0x24126ea1)),
])
def test_philox_known_answers(ctr, key, expect):
    got = philox4x32_10(np.array([ctr], dtype=np.uint64), np.array([key], dtype=np.uint64))[0]
    assert [int(v) for v in got] == list(expect)


def test_sampler_uniform_and_inverse_cdf_rule():
    # u: 24 bits, in [0, 1), exact in fp32; the counter layout puts tick in words 0-1 and the env id in word 2
    u = sampler_uniform(0, 0, [0], 0)
    x0 = 0x6627e8d5
    assert u.dtype == np.float32 and u[0] == np.float32((x0 >> 8) * 2.0 ** -24)
    x = philox4x32_10(np.array([[7, 0, 3, 0]], np.uint64), np.array([[5, 0]], np.uint64))[0]
    assert sampler_uniform(5, 7, [3], 1)[0] == np.float32((int(x[1]) >> 8) * 2.0 ** -24)
    x = philox4x32_10(np.array([[1, 2, 9, 0]], np.uint64), np.array([[3, 4]], np.uint64))[0]
    assert sampler_uniform((4 << 32) | 3, (2 << 32) | 1, [9], 0)[0] == np.float32((int(x[0]) >> 8) * 2.0 ** -24)
    us = sampler_uniform(5, 7, np.arange(4096), 0)
    assert us.min() >= 0 and us.max() < 1 and len(np.unique(us)) > 4000
    # the rule: boundaries, zero-probability actions and the fallback
    lp = np.array([np.log(0.25), -np.inf, np.log(0.5), np.log(0.25)], dtype=np.float32)
    assert sampler_draw(lp, 4, 0.0) == 0
    assert sampler_draw(lp, 4, 0.2499) == 0
    assert sampler_draw(lp, 4, 0.25) == 2            # c_0 = 0.25 is not > 0.25; the p = 0 action is skipped
    assert sampler_draw(lp, 4, 0.75) == 3
    assert sampler_draw(lp, 4, 1 - 2 ** -24) == 3
    assert sampler_draw(np.array([0.0, -np.inf, -np.inf], np.float32), 3, 0.999) == 0
    assert sampler_draw(np.array([-200.0, 0.0, -200.0], np.float32), 3, 0.0) == 1


def test_rollout_pool_mirror_matches_header_size():
    from cadre_b200 import ppo
    assert ctypes.sizeof(ppo.RolloutPoolC) == 9 * 8 + 5 * 4 + 4      # nine pointers, five int32, tail padding
    assert [f[0] for f in ppo.RolloutPoolC._fields_][-5:] == ["storages", "num_steps", "seq_length", "feature_dims",
                                                               "hidden_size"]


def _pool(T=16, n=4):
    from cadre_b200 import ppo
    r = ppo.RolloutPoolC()
    for name in ("obs", "action", "action_log_probs", "value_preds", "rewards", "masks", "command", "hn", "cn"):
        setattr(r, name, 0x1000)
    r.storages, r.num_steps, r.seq_length, r.feature_dims, r.hidden_size = n, T, 8, 530, 530
    return r


def test_new_entry_points_validate_their_arguments():
    """Without touching a device: bad sizes, a NULL handle and a cursor outside [0, num_steps] come back as an error
    code and a message."""
    import __graft_entry__
    __graft_entry__.build()
    from cadre_b200 import _lib
    lib = _lib.lib()
    p = ctypes.c_void_p(0x1000)
    u64 = ctypes.c_uint64

    def sample(ld, rows, A, word=0):
        return lib.cadre_categorical_sample(p, ld, rows, A, u64(0), u64(0), p, word, p, p, None, None)

    for ld, rows, A, word, msg in ((36, 8, 0, 0, b"A must"), (36, 8, 34, 0, b"A must"), (36, 0, 3, 0, b"rows"),
                                   (36, -1, 3, 0, b"rows"), (2, 8, 3, 0, b"ld"), (36, 8, 3, 4, b"word")):
        assert sample(ld, rows, A, word) != 0
        assert msg in lib.cadre_last_error(), lib.cadre_last_error()
    assert lib.cadre_categorical_sample(None, 36, 8, 3, u64(0), u64(0), p, 0, p, p, None, None) != 0
    assert b"pointers" in lib.cadre_last_error()

    T = 16
    pool = _pool(T)
    refs = (ctypes.c_void_p * 9)()
    idx = (ctypes.c_int32 * 4)(0, 1, 0, 1)

    def act(handle, slot, pool_ref):
        return lib.cadre_ppo_act(handle, refs, idx, p, p, pool_ref, slot, u64(0), u64(0), p, p, p, p, None)

    for slot in (-1, T + 1):
        assert act(None, slot, ctypes.byref(pool)) != 0
        assert b"slot" in lib.cadre_last_error()
        assert lib.cadre_rollout_env_results(ctypes.byref(pool), slot, p, p, None) != 0
        assert b"slot" in lib.cadre_last_error()
    for slot in (0, T):
        assert act(None, slot, ctypes.byref(pool)) != 0
        assert b"handle" in lib.cadre_last_error()
    assert act(None, 0, None) != 0 and b"pool" in lib.cadre_last_error()
    bad = _pool(T, n=0)
    assert act(None, 0, ctypes.byref(bad)) != 0 and b"sizes" in lib.cadre_last_error()
    assert lib.cadre_ppo_bootstrap(None, refs, idx, p, p, u64(0), p, None) != 0
    assert b"handle" in lib.cadre_last_error()
    assert lib.cadre_rollout_env_results(ctypes.byref(pool), 0, None, p, None) != 0
    assert b"pointers" in lib.cadre_last_error()


def test_device_rollout_needs_batched_acting():
    from cadre_b200.train import train
    with pytest.raises(ValueError, match="batched_acting"):
        train(0, None, None, None, None, None, batched_acting=False, device_rollout=True)

