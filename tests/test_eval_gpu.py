"""Ensemble evaluation on the B200: cadre_ensemble_control on hand-made rows (draws, greedy ties, controls bit for bit,
distribution per snapshot), cadre_ppo_ensemble_act against PpoEngine.evaluate / cadre_ppo_act / avg_action, and
eval.evaluate_envs end to end over SyntheticEnvs with snapshots written by save_snapshot."""
from types import SimpleNamespace

import numpy as np
import pytest
import torch

from oracle import restate as R
from test_eval_cpu import _avg_action, _bits, _tables, control_reduction, ensemble_uniform
from test_rollout_gpu import _f64_inverse_cdf, _row_kinds

pytestmark = pytest.mark.gpu

DEV = "cuda:0"


def _device_tables():
    cfg, steer, throttle = _tables()
    return cfg, torch.from_numpy(steer).to(DEV), torch.from_numpy(throttle).to(DEV)


def _rows(K, E, rs, ties=False):
    """fp32 [K, 2, E, 36] rows in evaluate's format: log-probs at columns 3.. (NaN past A), from the row kinds of the
    sampler tests (steer) and random / tied throttle rows."""
    kinds = _row_kinds(rs)
    steer_kinds = [row for _, A, row in kinds if A == 33]
    rows = torch.full((K, 2, E, 36), float("nan"))
    rows[:, :, :, :3] = 0.0
    for k in range(K):
        for e in range(E):
            rows[k, 0, e, 3:36] = steer_kinds[(k * E + e) % len(steer_kinds)][:33]
            t = torch.log_softmax(torch.as_tensor(rs.randn(3) * 2, dtype=torch.float32), -1)
            if ties and (k + e) % 3 == 0:
                t[rs.randint(3)] = t.max()
            rows[k, 1, e, 3:6] = t
            if ties and (k + e) % 2 == 0:      # exact ties of the steer maximum
                lp = rows[k, 0, e, 3:36]
                lp[rs.choice(33, 3, replace=False)] = torch.nan_to_num(lp, nan=-1e30).max()
    return rows


@pytest.mark.parametrize("K", [1, 3, 64])
def test_ensemble_control_draws_and_controls(K):
    from cadre_b200 import ppo
    cfg, steer, throttle = _device_tables()
    rs = np.random.RandomState(K)
    E, seed = 37, 0x1234_5678_9abc
    rows = _rows(K, E, rs)
    rows_d = rows.to(DEV)
    env_ids = np.arange(E) * 3 + 5
    ids = torch.tensor(env_ids, dtype=torch.int32, device=DEV)
    rows_np = rows.numpy()
    total = near_total = 0
    for tick in (0, 1, 9, (1 << 32) + 2):
        controls, actions = ppo.ensemble_control(rows_d, seed, tick, ids, steer, throttle)
        controls, actions = controls.cpu().numpy(), actions.cpu().numpy()
        assert actions.shape == (K, E, 2) and controls.shape == (E, 3)
        for k in range(K):
            for h, A in ((0, 33), (1, 3)):
                a = actions[k, :, h]
                assert a.min() >= 0 and a.max() < A
                lp = rows_np[k, h, :, 3:3 + A]
                assert (np.exp(lp[np.arange(E), a]) > 0).all(), "a zero-probability action was drawn"
                u = ensemble_uniform(seed, tick, env_ids, k, h)
                ref, near = _f64_inverse_cdf(lp, A, u)
                assert not ((a != ref) & ~near).any(), (k, h, tick)
                total += E
                near_total += int(near.sum())
                if k == 0:   # snapshot 0 draws what the rollout sampler draws
                    r0, _ = ppo.categorical_sample(rows_d[0, h, :, 3:].contiguous(), A, seed, tick, ids, h)
                    assert np.array_equal(r0.cpu().numpy(), a)
        for e in range(E):
            want = control_reduction(actions[:, e], _tables()[1], _tables()[2])
            assert np.array_equal(_bits(controls[e]), _bits(want))
            assert np.array_equal(_bits(controls[e]), _bits(_avg_action(cfg, actions[:, e])))
    assert near_total < 1e-2 * total, (near_total, total)


@pytest.mark.parametrize("K", [1, 5, 64])
def test_ensemble_control_greedy_takes_the_first_maximum(K):
    from cadre_b200 import ppo
    cfg, steer, throttle = _device_tables()
    rs = np.random.RandomState(10 + K)
    E = 23
    rows = _rows(K, E, rs, ties=True)
    ids = torch.arange(E, dtype=torch.int32, device=DEV)
    c1, a1 = ppo.ensemble_control(rows.to(DEV), 3, 0, ids, steer, throttle, greedy=True)
    c2, a2 = ppo.ensemble_control(rows.to(DEV), 4, 7, ids, steer, throttle, greedy=True)
    assert torch.equal(a1, a2) and torch.equal(c1, c2)          # no dependence on seed or tick
    a1, c1 = a1.cpu().numpy(), c1.cpu().numpy()
    ties = 0
    for k in range(K):
        for h, A in ((0, 33), (1, 3)):
            lp = rows[k, h, :, 3:3 + A]
            assert np.array_equal(a1[k, :, h], torch.argmax(lp, -1).numpy())
            ties += int(((lp == lp.max(-1, keepdim=True).values).sum(-1) > 1).sum())
    assert ties > 0
    for e in range(E):
        assert np.array_equal(_bits(c1[e]), _bits(_avg_action(cfg, a1[:, e])))


def test_ensemble_control_distribution_per_snapshot():
    from cadre_b200 import ppo
    _, steer, throttle = _device_tables()
    kinds = _row_kinds(np.random.RandomState(0))
    K, n = 3, 60_000
    rows = torch.full((K, 2, n, 36), float("nan"))
    rows[:, :, :, :3] = 0.0
    steer_row, thr_row = kinds[4][2], kinds[5][2]      # sum_ne_1 (33 actions), throttle (3 actions)
    rows[:, 0, :, 3:36] = steer_row[:33]
    rows[:, 1, :, 3:6] = thr_row[:3]
    ids = torch.arange(n, dtype=torch.int32, device=DEV)
    _, actions = ppo.ensemble_control(rows.to(DEV), 42, 3, ids, steer, throttle)
    actions = actions.cpu()
    for k in range(K):
        for h, (A, row) in enumerate(((33, steer_row), (3, thr_row))):
            counts = torch.bincount(actions[k, :, h], minlength=A).double()
            p = torch.exp(row[:A].double())
            p = p / p.sum()
            exp = p * n
            big = exp >= 5
            chi = (((counts[big] - exp[big]) ** 2) / exp[big]).sum().item()
            dof = int(big.sum().item())
            assert chi < dof + 6 * (2 * dof) ** 0.5 + 10, (k, h, chi, dof)
    # the snapshots draw independently: two snapshots agree about as often as two independent draws would
    p = torch.exp(steer_row[:33].double())
    p = p / p.sum()
    agree = (actions[0, :, 0] == actions[1, :, 0]).double().mean().item()
    assert abs(agree - (p * p).sum().item()) < 0.02, agree


def _windows(E, commands, rs):
    z = lambda *s, dtype=torch.float32: torch.zeros(*s, dtype=dtype, device=DEV)  # noqa: E731
    obs = torch.tensor(rs.randn(E, 8, 530).astype(np.float32), device=DEV)
    cmd = torch.tensor(np.asarray(commands, np.int32).reshape(E, 1), device=DEV)
    st = [SimpleNamespace(obs=obs, action=z(E, 1, dtype=torch.int64), value_preds=z(E, 1), returns=z(E, 1),
                          action_log_probs=z(E, 1), hn=z(E, 530), cn=z(E, 530), command=cmd) for _ in range(2)]
    return [tuple(st)], [(z(E, 1), z(E, 1))], [[list(range(E)), list(range(E))]]


@pytest.mark.parametrize("E,routing", [(1, "all"), (5, "all"), (64, "all"), (5, "one"), (64, "one")])
def test_ppo_ensemble_act(E, routing):
    from cadre_b200 import ppo
    from cadre_b200.learner import RolloutPool
    from cadre_b200.models import FlatParams
    cfg, steer, throttle = _device_tables()
    rs = np.random.RandomState(E)
    commands = [e % 4 for e in range(E)] if routing == "all" else [2] * E
    sts, advs, idx = _windows(E, commands, rs)
    params = [FlatParams(DEV, R.ppo_fixture_state(s)).params for s in (0, 1, 2)]
    assert not torch.equal(params[0], params[1]) and not torch.equal(params[1], params[2])
    eng = ppo.PpoEngine(1, E, device=DEV)
    ids = torch.tensor(rs.permutation(1000)[:E], dtype=torch.int32, device=DEV)
    seed = 99
    for K in (3, 1):
        rows = torch.zeros(K, 2, E, ppo.ROW_OUT, device=DEV)
        controls = torch.empty(E, 3, dtype=torch.float64, device=DEV)
        actions = torch.empty(K, E, 2, dtype=torch.int64, device=DEV)
        for tick in (0, 5):
            eng.ensemble_act(sts, advs, idx, params[:K], rows, seed, tick, ids, False, steer, throttle, controls,
                             actions)
            launches = eng.launches
            for k in range(K):
                ref = eng.evaluate(sts, advs, idx, params[k])
                assert torch.equal(rows[k], ref), (K, k, (rows[k] - ref).abs().max().item())
            assert launches == K * eng.launches + 1         # K x (forward + head_eval) + the ensemble kernel
            a, c = actions.cpu().numpy(), controls.cpu().numpy()
            for e in range(E):
                assert np.array_equal(_bits(c[e]), _bits(_avg_action(cfg, a[:, e])))
            if K == 1:   # a one-snapshot ensemble acts like the rollout path (cadre_ppo_act, BatchedActor.act_into)
                pool = RolloutPool(E, dict(num_steps=4, mini_batch_num=1, feature_dims=530, seq_length=8,
                                           hidden_size=530, use_gae=True, gamma=0.99, tau=0.95), DEV)
                hidden = (torch.zeros(1, 530, device=DEV), torch.zeros(1, 530, device=DEV))
                act = torch.empty(E, 2, dtype=torch.int64, device=DEV)
                rows_a = torch.zeros(2, E, ppo.ROW_OUT, device=DEV)
                eng.act(sts, advs, idx, params[0], rows_a, pool.c_ref(), 0, seed, tick, ids, hidden, act)
                assert torch.equal(act, actions[0])
                assert torch.equal(rows_a, rows[0])
    greedy_c = torch.empty_like(controls)
    greedy_a = torch.empty(3, E, 2, dtype=torch.int64, device=DEV)
    rows = torch.zeros(3, 2, E, ppo.ROW_OUT, device=DEV)
    eng.ensemble_act(sts, advs, idx, params, rows, seed, 0, ids, True, steer, throttle, greedy_c, greedy_a)
    for k in range(3):
        for h, A in ((0, 33), (1, 3)):
            assert torch.equal(greedy_a[k, :, h], torch.argmax(rows[k, h, :, 3:3 + A], -1))


def test_ppo_ensemble_act_rejects_a_multi_worker_engine():
    from cadre_b200 import ppo
    from cadre_b200._lib import CadreError
    _, steer, throttle = _device_tables()
    eng = ppo.PpoEngine(2, 2, device=DEV)
    sts, advs, _ = _windows(2, [0, 1], np.random.RandomState(0))
    p = torch.zeros(ppo.ppo_params.TOTAL, device=DEV)
    with pytest.raises(CadreError, match="workers = 1"):
        eng.ensemble_act(sts * 2, advs * 2, [[[0, 1], [0, 1]]] * 2, [p], torch.zeros(1, 2, 4, 36, device=DEV), 0, 0,
                         torch.zeros(4, dtype=torch.int32, device=DEV), False, steer, throttle,
                         torch.zeros(4, 3, dtype=torch.float64, device=DEV),
                         torch.zeros(1, 4, 2, dtype=torch.int64, device=DEV))


@pytest.fixture(scope="module")
def agent():
    from cadre_b200.agent import CadreAgent
    from cadre_b200.config import load_config
    cfg = load_config()
    return CadreAgent(**cfg.agent_cfg, danet_state=R.danet_fixture_state(0), ppo_state=R.ppo_fixture_state(0),
                      max_encoder_batch=8)


def _run_eval(agent, params, record):
    from cadre_b200.eval import DeviceEnsemble, evaluate_envs
    from cadre_b200.synthetic_env import SyntheticEnv
    E = 4
    envs = [SyntheticEnv(dict(rank=e, seq_length=8, done_prob=0.15)) for e in range(E)]
    ens = DeviceEnsemble(agent, params, E, seed=21, env_ids=[10, 11, 12, 13])
    log = []
    act = ens.act

    def recording_act(ticks, envs_):
        out = act(ticks, envs_)
        log.append((list(envs_), ticks if record else None,
                    [ens.actor.feats[e].clone() for e in envs_] if record else None, ens.last_actions.copy(), out))
        return out
    ens.act = recording_act
    res = evaluate_envs(ens, envs, 2, max_steps=20)
    return res, log, ens


def test_evaluate_envs_end_to_end(agent, tmp_path):
    import os
    from cadre_b200.eval import load_snapshot_params
    from cadre_b200.config import load_config
    from cadre_b200.models import init_state
    cfg = load_config()
    keep = agent.owner.params.clone()
    os.makedirs(tmp_path / "models")
    try:
        sources = []
        for ep, s in ((100, 1), (200, 2), (300, 3)):
            agent.owner.load_state(init_state(s))
            sources.append(agent.owner.params.clone())
            agent.save_snapshot(str(tmp_path / "models" / f"ppo_model_{ep}.pt"))
    finally:
        agent.owner.params.copy_(keep)
    params = load_snapshot_params(cfg.agent_cfg.model_cfg, str(tmp_path), [100, 200, 300])
    assert len(params) == 3 and all(torch.equal(p, s) for p, s in zip(params, sources))
    assert not torch.equal(params[0], params[1])

    res1, log1, ens1 = _run_eval(agent, params, record=True)
    res2, log2, ens2 = _run_eval(agent, params, record=False)
    assert res1 == res2                                  # every step count, return and control, bit for bit
    assert len(log1) == len(log2) and ens1.frames_encoded == ens2.frames_encoded
    for (envs1, _, _, a1, c1), (envs2, _, _, a2, c2) in zip(log1, log2):
        assert envs1 == envs2 and np.array_equal(a1, a2) and np.array_equal(c1.view(np.uint64), c2.view(np.uint64))
    # episodes end at different ticks, so environments leave the batch at different ticks
    assert all(len(r) == 2 for r in res1)
    assert len({sum(ep["steps"] for ep in r) for r in res1}) > 1
    assert any(len(envs) < 4 for envs, *_ in log1)
    steps = sum(ep["steps"] for r in res1 for ep in r)
    episodes = sum(len(r) for r in res1)
    assert sum(len(envs) for envs, *_ in log1) == steps
    assert ens1.frames_encoded == 8 * episodes + (steps - episodes)     # 8 per reset, then 1 per env and tick
    for envs, ticks, feats, actions, controls in log1:
        for i, e in enumerate(envs):
            assert torch.equal(feats[i], agent.get_latent_feature(ticks[i]))
            assert np.array_equal(_bits(controls[i]), _bits(_avg_action(agent, actions[:, e])))


def test_eval_main_prints_one_line_per_episode(tmp_path):
    """python -m cadre_b200.eval: a 3-snapshot ensemble over env_cfg.num_processes SyntheticEnvs."""
    import os
    import subprocess
    import sys
    from cadre_b200.config import load_config
    from cadre_b200.models import FlatParams, ModelDict, init_state, save_model_dict
    os.makedirs(tmp_path / "models")
    torch.save({"autoencoder": R.danet_fixture_state(0)}, str(tmp_path / "enc.pt"))
    for ep, s in ((100, 1), (200, 2), (300, 3)):
        save_model_dict(ModelDict(FlatParams("cpu", init_state(s))), str(tmp_path / "models" / f"ppo_model_{ep}.pt"))
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    env = dict(os.environ, CADRE_ENCODER_CKPT=str(tmp_path / "enc.pt"), CADRE_CHECKPOINT_DIR=str(tmp_path),
               CADRE_LOAD_EPISODE="100,200,300", CADRE_EVAL_EPISODE="2", CADRE_MAX_STEPS="12")
    r = subprocess.run([sys.executable, "-m", "cadre_b200.eval"], cwd=root, env=env, capture_output=True, text=True,
                       timeout=600)
    assert r.returncode == 0, r.stdout + r.stderr
    lines = [ln for ln in r.stdout.splitlines() if " episode " in ln and ln.startswith("env ")]
    E = load_config().env_cfg.num_processes
    assert len(lines) == 2 * E, r.stdout
    assert "ensemble of 3 snapshots" in r.stdout
