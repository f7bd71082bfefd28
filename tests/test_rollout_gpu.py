"""Device-side rollout path on the B200: the counter-based categorical sampler (exact draws against the numpy
restatement, distribution, keying), cadre_ppo_act writing a whole tick into the RolloutPool (bit-identical to the
existing act_batch + RolloutStorage.insert path), the batched bootstrap, and train(device_rollout=True)."""
import numpy as np
import pytest
import torch

from oracle import restate as R
from test_rollout_cpu import sampler_uniform

pytestmark = pytest.mark.gpu

DEV = "cuda:0"


def _lp_row(logits):
    return torch.log_softmax(torch.as_tensor(logits, dtype=torch.float32), -1)


def _row_kinds(rs):
    """Hand-made rows of normalised logits [36]: (name, A, row)."""
    kinds = []
    kinds.append(("uniform33", 33, torch.full((33,), float(np.log(np.float32(1.0 / 33))))))
    p = np.full(33, 1e-6 / 32)
    p[rs.randint(33)] = 1 - 1e-6
    kinds.append(("pmax", 33, torch.log(torch.tensor(p, dtype=torch.float64)).float()))
    two = torch.full((33,), float("-inf"))
    i, j = rs.choice(33, 2, replace=False)
    two[i] = two[j] = float(np.log(0.5))
    kinds.append(("two_hot", 33, two))
    under = _lp_row(rs.randn(33) * 2)
    under[rs.choice(33, 12, replace=False)] = -200.0        # exp(-200) underflows to 0 in fp32
    kinds.append(("underflow", 33, under))
    kinds.append(("sum_ne_1", 33, _lp_row(rs.randn(33) * 3)))   # fp32 log_softmax: sum of expf is not 1
    kinds.append(("throttle_nan", 3, _lp_row(rs.randn(3))))
    rows = []
    for name, A, lp in kinds:
        row = torch.full((36,), float("nan"))
        row[:A] = lp[:A]
        rows.append((name, A, row))
    return rows


def _f64_inverse_cdf(lp, A, u):
    """float64 reference of the draws of rows lp [n, >=A] at uniforms u [n]: (action, near a CDF boundary)."""
    p = np.exp(lp[:, :A].astype(np.float64))
    c = np.cumsum(p, 1)
    t = u.astype(np.float64) * c[:, -1]
    a = (c <= t[:, None]).sum(1)
    a = np.minimum(a, A - 1)
    near = (np.abs(c - t[:, None]) / c[:, -1:] < 1e-6).any(1)
    return a, near


def test_sampler_exact_draws():
    from cadre_b200 import ppo
    rs = np.random.RandomState(0)
    kinds = _row_kinds(rs)
    n_rows, ticks, seed = 4096, 64, 0x1234_5678_9abc
    kind_of = np.arange(n_rows) % len(kinds)
    total = near_total = 0
    for A in (33, 3):
        sel = np.nonzero([kinds[k][1] == A for k in kind_of])[0]
        lp = torch.stack([kinds[k][2] for k in kind_of[sel]])                # [n, 36], NaN past A
        lp_d = lp.to(DEV)
        ids = torch.tensor(sel, dtype=torch.int32, device=DEV)
        lp_np = lp.numpy()
        for tick in range(ticks):
            u_d = torch.empty(len(sel), device=DEV)
            a, lpo = ppo.categorical_sample(lp_d, A, seed, tick, ids, tick % 2, u_out=u_d)
            a, lpo, u = a.cpu().numpy(), lpo.cpu().numpy(), u_d.cpu().numpy()
            u_ref = sampler_uniform(seed, tick, sel, tick % 2)
            assert np.array_equal(u.view(np.uint32), u_ref.view(np.uint32))
            assert a.min() >= 0 and a.max() < A
            p_a = np.exp(lp_np[np.arange(len(sel)), a].astype(np.float32))
            assert (p_a > 0).all(), "a zero-probability action was drawn"
            assert np.array_equal(lpo.view(np.uint32), lp_np[np.arange(len(sel)), a].view(np.uint32))
            ref, near = _f64_inverse_cdf(lp_np, A, u_ref)
            bad = (a != ref) & ~near
            assert not bad.any(), (A, tick, np.nonzero(bad)[0][:5])
            total += len(sel)
            near_total += int(near.sum())
    assert near_total < 1e-3 * total, (near_total, total)


@pytest.mark.parametrize("kind", range(6))
def test_sampler_distribution(kind):
    from cadre_b200 import ppo
    name, A, row = _row_kinds(np.random.RandomState(0))[kind]
    n = 120_000
    lp = row.unsqueeze(0).expand(n, 36).contiguous().to(DEV)
    ids = torch.arange(n, dtype=torch.int32, device=DEV)
    a, _ = ppo.categorical_sample(lp, A, 42, 3, ids, 0)
    counts = torch.bincount(a.cpu(), minlength=A).double()
    p = torch.exp(row[:A].double())
    p = p / p.sum()
    exp = p * n
    big = exp >= 5
    chi = (((counts[big] - exp[big]) ** 2) / exp[big]).sum().item()
    dof = int(big.sum().item())
    e_small, c_small = exp[~big].sum().item(), counts[~big].sum().item()
    if e_small >= 5:            # the folded small bins are one more chi-square bin
        chi += (c_small - e_small) ** 2 / e_small
        dof += 1
    else:                       # too few expected draws for a chi-square term: a Poisson tail bound instead
        assert c_small <= e_small + 6 * e_small ** 0.5 + 6, (name, c_small, e_small)
    assert chi < dof + 6 * (2 * dof) ** 0.5 + 10, (name, chi, dof)
    assert counts[p == 0].sum().item() == 0


def test_sampler_keying():
    """An environment's draw depends on (seed, env id, tick) only: batch of 1, of 64, permuted, split over two actors."""
    from cadre_b200 import ppo
    rows = 64
    row = _row_kinds(np.random.RandomState(0))[0][2]
    lp = row.unsqueeze(0).expand(rows, 36).contiguous().to(DEV)
    ids = torch.arange(rows, dtype=torch.int32, device=DEV)
    perm = torch.randperm(rows, generator=torch.Generator().manual_seed(1)).to(DEV)
    for tick in (0, 1, 7, (1 << 32) + 5):
        for word in (0, 1):
            full, _ = ppo.categorical_sample(lp, 33, 9, tick, ids, word)
            one = torch.cat([ppo.categorical_sample(lp[:1], 33, 9, tick, ids[e:e + 1], word)[0] for e in range(rows)])
            pa, _ = ppo.categorical_sample(lp, 33, 9, tick, ids[perm].contiguous(), word)
            lo, _ = ppo.categorical_sample(lp[:32], 33, 9, tick, ids[:32].contiguous(), word)
            hi, _ = ppo.categorical_sample(lp[32:], 33, 9, tick, ids[32:].contiguous(), word)
            assert torch.equal(one, full) and torch.equal(pa, full[perm]) and torch.equal(torch.cat([lo, hi]), full)
    n = 4096
    lp = row.unsqueeze(0).expand(n, 36).contiguous().to(DEV)
    ids = torch.arange(n, dtype=torch.int32, device=DEV)
    base, _ = ppo.categorical_sample(lp, 33, 9, 4, ids, 0)
    for seed, tick, word in ((10, 4, 0), (9, 5, 0), (9, 4, 1), (9 + (1 << 32), 4, 0), (9, 4 + (1 << 32), 0)):
        other, _ = ppo.categorical_sample(lp, 33, seed, tick, ids, word)
        assert (other != base).double().mean().item() >= 0.9, (seed, tick, word)


@pytest.fixture(scope="module")
def agent():
    from cadre_b200.agent import CadreAgent
    from cadre_b200.config import load_config
    cfg = load_config()
    return CadreAgent(**cfg.agent_cfg, danet_state=R.danet_fixture_state(0), ppo_state=R.ppo_fixture_state(0),
                      max_encoder_batch=8)


W_PAR, T_PAR, TICKS_PAR = 3, 16, 40      # 40 ticks: the cursor wraps past slot T twice


def _envs(W):
    from cadre_b200.synthetic_env import SyntheticEnv
    return [SyntheticEnv(dict(rank=w, seq_length=8, done_prob=0.25, action_done_prob=0.2)) for w in range(W)]


def _pool(W, T):
    from cadre_b200.learner import RolloutPool
    return RolloutPool(W, dict(num_steps=T, mini_batch_num=2, feature_dims=530, seq_length=8, hidden_size=530,
                               use_gae=True, gamma=0.99, tau=0.95), DEV)


@pytest.fixture(scope="module")
def device_run(agent):
    """W_PAR workers for TICKS_PAR ticks through act_into / write_env_results; records actions and done flags."""
    from cadre_b200 import ppo
    from cadre_b200.actor import BatchedActor
    envs, pool = _envs(W_PAR), _pool(W_PAR, T_PAR)
    actor = BatchedActor(agent, W_PAR, seed=77, env_ids=[5, 6, 7])
    obs = [e.reset() for e in envs]
    done = [False] * W_PAR
    log = []
    resets = 0
    for tick in range(TICKS_PAR):
        slot = pool.storages[0][0].step
        a = actor.act_into(obs, pool)
        assert a.shape == (W_PAR, 2) and a.dtype == np.int64
        for h, A in ((0, 33), (1, 3)):      # the act kernel draws what the standalone sampler draws from its rows
            ref, _ = ppo.categorical_sample(actor._rows[h, :, 3:].contiguous(), A, 77, tick, actor._env_ids_d, h)
            assert np.array_equal(ref.cpu().numpy(), a[:, h])
        rewards, masks = np.zeros((W_PAR, 2), np.float32), np.zeros((W_PAR, 2), np.float32)
        for w, env in enumerate(envs):
            obs[w], r, done[w], info = env.step(agent.convert_action(a[w]))
            rewards[w] = r
            masks[w] = [0.0 if d else 1.0 for d in info["action_done"]]
            if done[w]:
                obs[w] = env.reset()
                actor.reset(w)
                resets += 1
        pool.write_env_results(slot, rewards, masks)
        log.append((slot, a, list(done)))
    assert resets > 0 and actor.ticks == TICKS_PAR
    torch.cuda.synchronize()
    return pool, log, actor


def test_act_into_pool_is_bit_identical_to_insert_path(agent, device_run):
    from cadre_b200.actor import BatchedActor
    pool_d, log, _ = device_run
    envs, pool = _envs(W_PAR), _pool(W_PAR, T_PAR)
    actor = BatchedActor(agent, W_PAR)
    obs = [e.reset() for e in envs]
    for slot, a, _ in log:
        assert pool.storages[0][0].step == slot
        feats, _, _, values = actor.act_batch(obs)
        for h in range(2):                      # log-probs of the device path's actions
            actor._st[h].action.copy_(torch.from_numpy(a[:, h:h + 1]))
        out = actor._engine.evaluate([tuple(actor._st)], [actor._adv], actor._idx, agent.owner.params)
        assert torch.equal(out[:, :, 0].t(), values)
        for w, env in enumerate(envs):
            command = obs[w]["command"]
            obs[w], r, done, info = env.step(agent.convert_action(a[w]))
            for h in range(2):
                mask = torch.tensor([[0.0] if info["action_done"][h] else [1.0]])
                pool.storages[w][h].insert(feats[w].clone(), torch.tensor(a[w, h]), out[h, w, 1], values[w, h], r[h],
                                           mask, agent.hidden_state, command)
            if done:
                obs[w] = env.reset()
                actor.reset(w)
    torch.cuda.synchronize()
    for name in ("obs", "action", "action_log_probs", "value_preds", "command", "hn", "cn", "rewards", "masks"):
        d, r = pool_d.batched[name], pool.batched[name]
        assert torch.equal(d, r), (name, (d != r).sum().item())
    assert pool.batched["action"].max().item() > 2                  # steer draws were written, not only zeros
    assert (pool.batched["masks"] == 0).any() and (pool.batched["obs"][:, T_PAR] != 0).any()
    for w in range(W_PAR):
        for h in range(2):
            assert pool_d.storages[w][h].step == pool.storages[w][h].step == TICKS_PAR % (T_PAR + 1)


def test_bootstrap_into_matches_get_value(agent, device_run):
    pool, _, actor = device_run
    for done in ([False, False, False], [True, False, True], [False, True, False]):
        nv = actor.bootstrap_into(pool, done).clone().view(W_PAR, 2).cpu()
        exact = True
        for w in range(W_PAR):
            vs, vt = agent.get_value(done[w], pool.storages[w][0].get_last(), pool.storages[w][1].get_last())
            ref = torch.tensor([float(vs.reshape(-1)[0]), float(vt.reshape(-1)[0])])
            if done[w]:
                assert nv[w].tolist() == [0.0, 0.0]
            else:
                assert (nv[w] - ref).abs().max().item() < 1e-6, (w, nv[w], ref)
                exact = exact and torch.equal(nv[w], ref)
        print(f"bootstrap done={done}: bit-exact with get_value: {exact}")
    # compute_returns(None) reads pool.next_value
    actor.bootstrap_into(pool, [False, True, False])
    pool.compute_returns(None)
    assert torch.isfinite(pool.batched["returns"]).all()


def test_train_loop_with_device_rollout():
    from cadre_b200.config import load_config
    from cadre_b200.train import train
    params = []
    for _ in range(2):
        cfg = load_config()
        cfg.rollout_cfg.num_steps = 8
        cfg.rollout_cfg.mini_batch_num = 2
        cfg.train_cfg.log_interval = 1000
        cfg.env_cfg["done_prob"] = 0.1
        ppo0 = R.ppo_fixture_state(0)
        learner, hist = train(0, cfg.train_cfg, cfg.agent_cfg, cfg.env_cfg, cfg.rollout_cfg, R.danet_fixture_state(0),
                              ppo_state=ppo0, workers=2, max_episode=2, device_rollout=True, log=lambda *a: None)
        assert len(hist) == 2 and all(np.isfinite(v) for ep in hist for v in ep)
        assert learner.step_count == 2 * cfg.train_cfg.ppo_epoch * 2
        new = learner.state()
        moved = (new["steer_lstm_0"]["rnn.weight_ih"].cpu() - ppo0["steer_lstm_0"]["rnn.weight_ih"]).abs().max().item()
        assert 0 < moved < 0.1
        params.append(learner.params.clone())
    assert torch.equal(params[0], params[1])
