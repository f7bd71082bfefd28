"""CPU checks of the PPO update diagnostics and rollout statistics: float64 restatements of both (used by
test_diagnostics_gpu.py as the reference), the new C entry points' declarations and exports, and argument errors."""
import ctypes
import os

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


# ------------------------------------------------------------------------------------------------ restatements
def update_diagnostics(cur_lp, old_lp, cur_v, old_v, clip=0.1):
    """The diagnostics of one head's minibatch in float64, from the quantities of ppo_agent/agent.py:184-193 (cur_lp /
    cur_v of the current policy, old_lp / old_v stored in the rollout): [approx KL = mean(expm1(d) - d), mean(-d),
    fraction of rows with |ratio - 1| > clip, fraction of rows with |v - old_v| > clip], d = cur_lp - old_lp."""
    f = lambda x: np.asarray(x, dtype=np.float64).reshape(-1)   # noqa: E731
    cur_lp, old_lp, cur_v, old_v = f(cur_lp), f(old_lp), f(cur_v), f(old_v)
    d = cur_lp - old_lp
    ratio = np.exp(d)
    return np.array([np.mean(np.expm1(d) - d), np.mean(-d), np.mean(np.abs(ratio - 1.0) > clip),
                     np.mean(np.abs(cur_v - old_v) > clip)])


def near_clip_rows(cur_lp, old_lp, clip=0.1, eps=1e-4):
    """Rows whose |ratio - 1| lies within eps of clip: the strict comparison may go either way there."""
    d = np.asarray(cur_lp, np.float64).reshape(-1) - np.asarray(old_lp, np.float64).reshape(-1)
    return int(np.sum(np.abs(np.abs(np.exp(d) - 1.0) - clip) <= eps))


def rollout_stats(returns, values):
    """cadre_rollout_stats in numpy float64: returns / values [E, T+1] (steps t < T) -> [E, 6] = explained variance
    (NaN where Var(R) = 0), mean and std of R - V, mean and std of R, mean of V; population variances."""
    R = np.asarray(returns, np.float64)[:, :-1]
    V = np.asarray(values, np.float64)[:, :-1]
    A = R - V
    mr, ma = R.mean(1, keepdims=True), A.mean(1, keepdims=True)
    var_r = ((R - mr) ** 2).mean(1)
    var_a = ((A - ma) ** 2).mean(1)
    with np.errstate(divide="ignore", invalid="ignore"):
        ev = np.where(var_r == 0, np.nan, 1.0 - var_a / np.where(var_r == 0, 1.0, var_r))
    return np.stack([ev, ma[:, 0], np.sqrt(var_a), mr[:, 0], np.sqrt(var_r), V.mean(1)], 1)


# ------------------------------------------------------------------------------------------------ tests
def test_rollout_stats_restatement_matches_direct_float64():
    rs = np.random.RandomState(3)
    E, T = 6, 50
    ret = rs.randn(E, T + 1).astype(np.float32) * 3 + 1
    val = (ret + rs.randn(E, T + 1).astype(np.float32)).astype(np.float32)
    ret[4, :T] = 2.5                                            # constant returns: Var(R) = 0
    got = rollout_stats(ret, val)
    for e in range(E):
        y, p = ret[e, :T].astype(np.float64), val[e, :T].astype(np.float64)
        var_y = np.var(y)                                       # SB3 common/utils.py explained_variance
        ev = np.nan if var_y == 0 else 1 - np.var(y - p) / var_y
        want = [ev, np.mean(y - p), np.std(y - p), np.mean(y), np.std(y), np.mean(p)]
        np.testing.assert_allclose(got[e], want, rtol=1e-12, atol=1e-12, equal_nan=True)
    assert np.isnan(got[4, 0]) and np.isfinite(np.delete(got, 4, 0)).all()
    assert got[4, 4] == 0.0


def test_update_diagnostics_restatement_hand_values():
    lp = np.log(np.array([0.5, 0.5, 0.5, 0.5]))
    old = lp - np.array([0.0, 0.2, 0.05, -0.2])                 # d = 0, 0.2, 0.05, -0.2
    v, old_v = np.zeros(4), np.array([0.0, 0.2, -0.05, -0.1])
    got = update_diagnostics(lp, old, v, old_v)
    d = np.array([0.0, 0.2, 0.05, -0.2])
    assert got[0] == pytest.approx(np.mean(np.exp(d) - 1 - d), rel=1e-12)
    assert got[1] == pytest.approx(-np.mean(d), rel=1e-12)
    assert got[2] == 0.5                                        # exp(0.2) - 1 = 0.221, 1 - exp(-0.2) = 0.181
    assert got[3] == 0.25                                       # strict: |-0.1| is not > 0.1
    assert near_clip_rows(lp, old) == 0 and near_clip_rows([np.log(1.1)], [0.0]) == 1


def test_new_symbols_are_declared_and_exported():
    import __graft_entry__
    __graft_entry__.build()
    from cadre_b200 import _lib
    header = open(os.path.join(ROOT, "include", "cadre_b200.h")).read()
    assert "int cadre_ppo_set_diagnostics(void* handle, float* diag_out, float* norms_out);" in header
    assert "int cadre_rollout_stats(const float* returns, const float* values, int E, int T, float* out, void* stream);" \
        in header
    lib = _lib.lib()
    for name in ("cadre_ppo_set_diagnostics", "cadre_rollout_stats"):
        assert hasattr(lib, name), name


def test_new_entry_points_validate_their_arguments():
    import __graft_entry__
    __graft_entry__.build()
    from cadre_b200 import _lib, ppo
    lib = _lib.lib()
    p = ctypes.c_void_p(0x1000)
    assert lib.cadre_ppo_set_diagnostics(None, p, p) != 0 and b"handle" in lib.cadre_last_error()
    assert lib.cadre_rollout_stats(None, p, 4, 8, p, None) != 0 and b"pointers" in lib.cadre_last_error()
    assert lib.cadre_rollout_stats(p, p, 4, 8, None, None) != 0 and b"pointers" in lib.cadre_last_error()
    for E, T in ((0, 8), (-1, 8), (4, 0)):
        assert lib.cadre_rollout_stats(p, p, E, T, p, None) != 0 and b"sizes" in lib.cadre_last_error()
    with pytest.raises(_lib.CadreError):
        ppo.rollout_stats(torch.zeros(4, 9), torch.zeros(4, 9))      # host tensors: no CPU fallback
