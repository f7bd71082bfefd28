"""CPU checks of target-KL early stopping: a float64 restatement of the stop rule (used by test_target_kl_gpu.py as the
reference), the new C entry points' declarations and exports, and argument errors."""
import ctypes
import math
import os

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


# ------------------------------------------------------------------------------------------------ restatement
def stop_rule(approx_kl, target_kl):
    """SB3's rule on a phase in float64. approx_kl [steps, workers of all ranks, 2]: each worker's and head's
    approximate KL of every update step. The KL of step n is the sum over the heads of the mean over the workers; the
    first step whose KL exceeds 1.5 * target_kl stops the phase and is not applied. Returns (kl [steps], stopped_at or
    None, steps applied)."""
    kl = np.asarray(approx_kl, np.float64).mean(1).sum(1)
    over = np.flatnonzero(kl > 1.5 * float(target_kl))
    stopped_at = int(over[0]) if over.size else None
    return kl, stopped_at, (stopped_at if stopped_at is not None else kl.shape[0])


def record_step(kl, margin=1e-3, lowest=1, prefer="last"):
    """A step k >= lowest whose KL exceeds every earlier KL by at least `margin` (relative), and a target_kl whose
    1.5 * target_kl is the geometric midpoint of KL_k and that earlier maximum: the phase then stops exactly at k.
    Returns (k, target_kl) or None."""
    kl = np.asarray(kl, np.float64)
    ks = [k for k in range(max(1, lowest), kl.shape[0]) if kl[:k].max() > 0 and kl[k] > kl[:k].max() * (1 + margin)]
    if not ks:
        return None
    k = ks[-1] if prefer == "last" else ks[0]
    return k, math.sqrt(kl[k] * kl[:k].max()) / 1.5


# ------------------------------------------------------------------------------------------------ tests
def test_stop_rule_on_constructed_histories():
    steps, W = 8, 3
    a = np.full((steps, W, 2), 1e-3)
    kl, stop, applied = stop_rule(a, 0.01)                        # KL 2e-3 everywhere, threshold 1.5e-2
    assert np.allclose(kl, 2e-3) and stop is None and applied == steps
    a[3] = 0.02                                                   # step 3: KL 0.04 > 0.015; later steps too
    a[5] = 0.05
    kl, stop, applied = stop_rule(a, 0.01)
    assert stop == 3 and applied == 3 and kl[3] == pytest.approx(0.04, rel=1e-12)
    a[0] = 0.05                                                   # the first step can stop the phase: nothing applied
    assert stop_rule(a, 0.01)[1:] == (0, 0)


def test_stop_rule_sums_heads_and_averages_workers():
    a = np.zeros((4, 2, 2))
    a[2, :, 0] = a[2, :, 1] = 0.008                               # each head below 0.015, their sum 0.016 above
    assert stop_rule(a, 0.01)[1] == 2
    b = np.zeros((4, 4, 2))
    b[1, 0, :] = 0.02                                             # one worker over, the mean over 4 workers not
    kl, stop, _ = stop_rule(b, 0.01)
    assert stop is None
    assert kl[1] == pytest.approx(2 * 0.02 / 4, rel=1e-12)
    c = np.zeros((3, 1, 2))
    c[1, 0] = [0.0075, 0.0075]                                    # exactly 1.5 * target_kl: not a stop (strict >)
    assert stop_rule(c, 0.01)[1] is None


def test_record_step_threshold_stops_there():
    kl = np.array([1e-8, 2e-4, 1e-4, 5e-4, 4.9e-4, 5.0001e-4, 9e-4, 8e-4])
    k, t = record_step(kl)
    assert k == 6 and 5e-4 < 1.5 * t < 9e-4
    assert stop_rule(np.stack([kl, 0 * kl], 1)[:, None, :], t)[1] == 6
    k0, t0 = record_step(kl, prefer="first")
    assert k0 == 1 and stop_rule(np.stack([kl, 0 * kl], 1)[:, None, :], t0)[1] == 1
    assert record_step(kl, lowest=7) is None                      # no record after step 6
    assert record_step(np.array([3e-3, 2e-3, 1e-3])) is None


def test_new_symbols_are_declared_and_exported():
    import __graft_entry__
    __graft_entry__.build()
    from cadre_b200 import _lib
    header = open(os.path.join(ROOT, "include", "cadre_b200.h")).read()
    for decl in ("int cadre_ppo_set_target_kl(void* handle, float target_kl, int total_workers, float* kl_sum_dev);",
                 "int cadre_ppo_kl_begin(void* handle, void* stream);",
                 "int cadre_ppo_kl_gate(void* handle, void* stream);",
                 "int cadre_ppo_early_stop(void* handle, int32_t* state_host, float* kl_host, int kl_count, void* stream);"):
        assert decl in header, decl
    lib = _lib.lib()
    for name in ("cadre_ppo_set_target_kl", "cadre_ppo_kl_begin", "cadre_ppo_kl_gate", "cadre_ppo_early_stop"):
        assert hasattr(lib, name), name


def test_new_entry_points_validate_their_arguments():
    import __graft_entry__
    __graft_entry__.build()
    from cadre_b200 import _lib
    lib = _lib.lib()
    p = ctypes.c_void_p(0x1000)
    f = ctypes.c_float
    for bad in (-0.01, math.nan, math.inf, -math.inf):
        assert lib.cadre_ppo_set_target_kl(None, f(bad), 4, p) != 0 and b"target_kl" in lib.cadre_last_error(), bad
    assert lib.cadre_ppo_set_target_kl(None, f(0.02), 4, p) != 0 and b"handle" in lib.cadre_last_error()
    assert lib.cadre_ppo_set_target_kl(None, f(0.0), 0, None) != 0 and b"handle" in lib.cadre_last_error()
    assert lib.cadre_ppo_kl_begin(None, None) != 0 and b"handle" in lib.cadre_last_error()
    assert lib.cadre_ppo_kl_gate(None, None) != 0 and b"handle" in lib.cadre_last_error()
    st = (ctypes.c_int32 * 5)()
    assert lib.cadre_ppo_early_stop(None, st, None, 0, None) != 0 and b"NULL" in lib.cadre_last_error()
    assert lib.cadre_ppo_early_stop(p, None, None, 0, None) != 0 and b"NULL" in lib.cadre_last_error()
    assert lib.cadre_ppo_early_stop(p, st, None, 4, None) != 0 and b"kl_count" in lib.cadre_last_error()
    assert lib.cadre_ppo_early_stop(p, st, p, 4097, None) != 0 and b"kl_count" in lib.cadre_last_error()


@pytest.mark.parametrize("bad", [0, 0.0, -0.02, math.nan, math.inf, -math.inf, 1e-50, 1e39, True, "0.02", [0.02]])
def test_learner_rejects_bad_target_kl(bad):
    """Checked before anything touches a device: a bad value fails the same way with or without a GPU."""
    import __graft_entry__
    __graft_entry__.build()
    from cadre_b200._lib import CadreError
    from cadre_b200.learner import Learner, check_target_kl
    with pytest.raises(CadreError, match="target_kl"):
        check_target_kl(bad)
    with pytest.raises(CadreError, match="target_kl"):
        Learner(1, 4, None, "cpu", target_kl=bad)


def test_learner_accepts_target_kl():
    import __graft_entry__
    __graft_entry__.build()
    from cadre_b200.learner import check_target_kl
    assert check_target_kl(None) is None
    assert check_target_kl(0.02) == 0.02 and check_target_kl(np.float32(0.5)) == 0.5 and check_target_kl(3) == 3.0


def test_chief_assigns_the_learner_step_count():
    """utils.chief advances `optimizer.step_count` itself (`+= 1`) before its Adam step: the Learner's step count must
    stay assignable. A stub engine records the step chief passes, so no device is needed."""
    import torch
    from types import SimpleNamespace
    from cadre_b200 import utils
    from cadre_b200.learner import Learner
    steps = []
    learner = Learner.__new__(Learner)
    learner._phase, learner._step_count, learner.lr = None, 0, 3e-4
    learner.engine = SimpleNamespace(adam_step=lambda p, g, m, v, step, max_norm, lr: steps.append(step))
    learner.params, learner.grads, learner.exp_avg, learner.exp_avg_sq = (torch.zeros(8) for _ in range(4))
    shared = SimpleNamespace(grads=torch.arange(8.0), reset=lambda: None)
    counter, light = utils.Counter(), utils.TrafficLight()
    assert not utils.chief(1, light, counter, None, shared, learner)
    for n in (1, 2):
        counter.increment()
        assert utils.chief(1, light, counter, None, shared, learner)
        assert learner.step_count == n and steps == list(range(1, n + 1))
    assert torch.equal(learner.grads, shared.grads)
