"""CPU checks of ensemble evaluation: a numpy restatement of the control reduction of cadre_ensemble_control against
CadreAgent.avg_action (bit for bit), the sampler's counter word 3 (the snapshot index), argument errors of the two new
entry points without a device, and the episode accounting of eval.evaluate_envs with fake environments."""
import ctypes
from types import SimpleNamespace

import numpy as np
import pytest

from test_rollout_cpu import philox4x32_10, sampler_uniform


def _tables():
    from cadre_b200.config import load_config
    cfg = load_config().agent_cfg
    steer = np.array([cfg.STEER_CONTROL[i] for i in range(33)], dtype=np.float64)
    throttle = np.array([cfg.THROTTLE_CONTROL[i] for i in range(3)], dtype=np.float64).reshape(-1)
    return cfg, steer, throttle


def ensemble_uniform(seed, tick, env_ids, k, word):
    """u of snapshot k's draw: Philox counter (tick lo, tick hi, env id, k), output word `word`; float32."""
    env_ids = np.asarray(env_ids, dtype=np.uint64)
    n = env_ids.shape[0]
    ctr = np.stack([np.full(n, tick & 0xFFFFFFFF, np.uint64), np.full(n, tick >> 32, np.uint64), env_ids,
                    np.full(n, k, np.uint64)], -1)
    key = np.tile(np.array([seed & 0xFFFFFFFF, seed >> 32], dtype=np.uint64), (n, 1))
    x = philox4x32_10(ctr, key)[:, word]
    return ((x >> np.uint32(8)).astype(np.float32) * np.float32(2.0 ** -24)).astype(np.float32)


def control_reduction(actions, steer_table, throttle_table):
    """The kernel's reduction of one environment's actions int [K, 2]: float64 sums in snapshot order, / K, and with
    K > 1 a mean brake below 0.5 released."""
    K = len(actions)
    s = t = b = np.float64(0.0)
    for a_s, a_t in actions:
        s = s + steer_table[a_s]
        t = t + throttle_table[2 * a_t]
        b = b + throttle_table[2 * a_t + 1]
    n = np.float64(K)
    s, t, b = s / n, t / n, b / n
    if K > 1 and b < 0.5:
        b = np.float64(0.0)
    return np.array([s, t, b], dtype=np.float64)


def _avg_action(cfg, actions):
    """CadreAgent.avg_action on a namespace holding the two tables, actions int [K, 2]."""
    from cadre_b200.agent import CadreAgent
    ns = SimpleNamespace(STEER_CONTROL=cfg.STEER_CONTROL, THROTTLE_CONTROL=cfg.THROTTLE_CONTROL)
    ns.convert_action = lambda a: CadreAgent.convert_action(ns, a)
    return np.array(CadreAgent.avg_action(ns, [[np.int64(a_s), np.int64(a_t)] for a_s, a_t in actions]),
                    dtype=np.float64)


def _bits(x):
    return np.ascontiguousarray(x, dtype=np.float64).view(np.uint64)


@pytest.mark.parametrize("K", list(range(1, 10)) + [16, 33, 64])
def test_control_reduction_matches_avg_action_bit_for_bit(K):
    cfg, steer, throttle = _tables()
    rs = np.random.RandomState(K)
    for trial in range(200):
        actions = np.stack([rs.randint(0, 33, K), rs.randint(0, 3, K)], 1)
        if trial % 4 == 0:                      # mostly braking: means around and above 0.5
            actions[:, 1] = np.where(rs.rand(K) < 0.7, 1, rs.randint(0, 3, K))
        ref = _avg_action(cfg, actions)
        got = control_reduction(actions, steer, throttle)
        assert np.array_equal(_bits(got), _bits(ref)), (K, actions.tolist(), got, ref)


@pytest.mark.parametrize("K", [2, 4, 8, 16, 64])
def test_control_reduction_at_a_mean_brake_of_one_half(K):
    """Exactly half the snapshots brake: the mean is 0.5, which is not below 0.5, so the brake stays."""
    cfg, steer, throttle = _tables()
    rs = np.random.RandomState(100 + K)
    actions = np.stack([rs.randint(0, 33, K), np.array([1] * (K // 2) + [2] * (K - K // 2))], 1)
    got = control_reduction(actions, steer, throttle)
    assert got[2] == 0.5
    assert np.array_equal(_bits(got), _bits(_avg_action(cfg, actions)))
    actions[0, 1] = 0                          # one brake fewer: below 0.5, released
    got = control_reduction(actions, steer, throttle)
    assert got[2] == 0.0 and np.array_equal(_bits(got), _bits(_avg_action(cfg, actions)))
    one = control_reduction(actions[:1], steer, throttle)   # a single snapshot never releases its brake
    assert np.array_equal(_bits(one), _bits(_avg_action(cfg, actions[:1])))


def test_snapshot_index_is_counter_word_three():
    ids = np.arange(257)
    for seed, tick in ((0, 0), (5, 7), ((4 << 32) | 3, (2 << 32) | 1)):
        for word in range(4):
            assert np.array_equal(ensemble_uniform(seed, tick, ids, 0, word).view(np.uint32),
                                  sampler_uniform(seed, tick, ids, word).view(np.uint32))
            for k in (1, 63):
                other = ensemble_uniform(seed, tick, ids, k, word)
                assert (other != sampler_uniform(seed, tick, ids, word)).mean() > 0.9
    x = philox4x32_10(np.array([[7, 0, 3, 5]], np.uint64), np.array([[9, 0]], np.uint64))[0]
    assert ensemble_uniform(9, 7, [3], 5, 1)[0] == np.float32((int(x[1]) >> 8) * 2.0 ** -24)


def test_ensemble_entry_points_validate_their_arguments():
    """Without touching a device: every bad argument comes back as an error code and a message, before any launch."""
    import __graft_entry__
    __graft_entry__.build()
    from cadre_b200 import _lib
    lib = _lib.lib()
    p = ctypes.c_void_p(0x1000)
    u64 = ctypes.c_uint64

    def control(row=p, K=3, E=4, greedy=0, ids=p, steer=p, thr=p, ctl=p, act=p):
        return lib.cadre_ensemble_control(row, K, E, u64(0), u64(0), ids, greedy, steer, thr, ctl, act, None)

    cases = [(dict(K=0), b"K must"), (dict(K=65), b"K must"), (dict(K=-1), b"K must"), (dict(E=0), b"E must"),
             (dict(E=-3), b"E must"), (dict(greedy=2), b"greedy"), (dict(greedy=-1), b"greedy")]
    cases += [(dict({name: None}), b"pointers") for name in ("row", "ids", "steer", "thr", "ctl", "act")]
    for kw, msg in cases:
        assert control(**kw) != 0, kw
        assert msg in lib.cadre_last_error(), (kw, lib.cadre_last_error())

    refs = (ctypes.c_void_p * 9)()
    idx = (ctypes.c_int32 * 4)(0, 1, 0, 1)

    def act(handle=None, refs=refs, idx=idx, params=None, K=3, row=p, greedy=0, ids=p, steer=p, thr=p, ctl=p,
            act=p):
        if params is None:
            params = (ctypes.c_void_p * 3)(0x1000, 0x2000, 0x3000)
        return lib.cadre_ppo_ensemble_act(handle, refs, idx, params, K, row, u64(0), u64(0), ids, greedy, steer, thr,
                                          ctl, act, None)

    cases = [(dict(K=0), b"K must"), (dict(K=65), b"K must"), (dict(greedy=2), b"greedy"),
             (dict(params=(ctypes.c_void_p * 3)(0x1000, None, 0x3000)), b"params_host[k] is NULL"),
             (dict(refs=None), b"ppo_ensemble_act pointers"), (dict(idx=None), b"ppo_ensemble_act pointers"),
             (dict(handle=None), b"handle")]
    cases += [(dict(params=ctypes.cast(None, ctypes.POINTER(ctypes.c_void_p))), b"ppo_ensemble_act pointers")]
    cases += [(dict({name: None}), b"ensemble pointers") for name in ("row", "ids", "steer", "thr", "ctl", "act")]
    for kw, msg in cases:
        assert act(**kw) != 0, kw
        assert msg in lib.cadre_last_error(), (kw, lib.cadre_last_error())


class _FakeEnv:
    """Episodes of fixed lengths; records every call."""

    def __init__(self, lengths):
        self.lengths, self.episode, self.t, self.calls = list(lengths), -1, 0, []

    def reset(self):
        self.episode += 1
        self.t = 0
        self.calls.append("reset")
        return {"ep": self.episode, "t": 0}

    def step(self, control):
        self.t += 1
        self.calls.append("step")
        done = self.t >= self.lengths[self.episode % len(self.lengths)]
        return {"ep": self.episode, "t": self.t}, [1.0, 0.5], done, {}


class _FakeEnsemble:
    def __init__(self, envs):
        self.envs, self.acted, self.resets = envs, [], []

    def reset(self, e):
        assert self.envs[e].calls[-1] == "reset"        # right after that environment's reset
        self.resets.append((e, self.envs[e].episode))

    def act(self, ticks, envs):
        assert len(ticks) == len(envs) and len(set(envs)) == len(envs)
        for t, e in zip(ticks, envs):                   # each env's current tick
            assert t == {"ep": self.envs[e].episode, "t": self.envs[e].t}
        self.acted.append(list(envs))
        return np.array([[0.1 * e, 0.5, 0.0] for e in envs], dtype=np.float64)


@pytest.mark.parametrize("max_steps", [None, 3, 1, 0])
def test_evaluate_envs_episode_accounting(max_steps):
    from cadre_b200.eval import evaluate_envs
    lengths = [[2, 5], [7], [1, 1, 4], [3, 9, 2]]
    envs = [_FakeEnv(l) for l in lengths]
    ens = _FakeEnsemble(envs)
    eval_episode = 3
    cap = max_steps if max_steps is not None else 10 ** 9
    res = evaluate_envs(ens, envs, eval_episode, max_steps=max_steps)
    assert len(res) == len(envs)
    for e, env in enumerate(envs):
        assert len(res[e]) == eval_episode
        want = [min(lengths[e][i % len(lengths[e])], cap) for i in range(eval_episode)]
        assert [r["steps"] for r in res[e]] == want
        assert env.calls.count("reset") == eval_episode and env.calls.count("step") == sum(want)
        assert [r["return"] for r in res[e]] == [[1.0 * n, 0.5 * n] for n in want]
        assert all(r["controls"] == [[0.1 * e, 0.5, 0.0]] * r["steps"] for r in res[e])
        assert [ep for ee, ep in ens.resets if ee == e] == list(range(eval_episode))
        # acted on in exactly the ticks it was stepped in, never after its last episode
        assert sum(e in a for a in ens.acted) == sum(want)
        last = max([i for i, a in enumerate(ens.acted) if e in a], default=-1)
        assert all(e not in a for a in ens.acted[last + 1:])
    assert len(ens.acted) == max(sum(min(lengths[e][i % len(lengths[e])], cap) for i in range(eval_episode))
                                 for e in range(len(envs)))


def test_evaluate_envs_without_episodes():
    from cadre_b200.eval import evaluate_envs
    envs = [_FakeEnv([2]) for _ in range(2)]
    ens = _FakeEnsemble(envs)
    assert evaluate_envs(ens, envs, 0) == [[], []]
    assert ens.acted == [] and all(env.calls == [] for env in envs)
