"""PPO update diagnostics and rollout statistics on the GPU: exact answers on constructed ratios / values, agreement
with the float64 restatement on the oracle's forward rows, bit-identical training with diagnostics on, staged
histories against single steps, the two-rank norm history, rollout statistics against numpy, and the training loop."""
import os
import socket
import sys
from types import SimpleNamespace

import numpy as np
import pytest
import torch
import torch.multiprocessing as mp

from oracle import restate as R
from test_diagnostics_cpu import near_clip_rows, rollout_stats as rollout_stats_f64, update_diagnostics
from test_ppo_gpu import ROUTING_PLANS, _config_inputs, _oracle_rows, _plan_seed

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CLIP = R.CLIP


def _diag_update(eng, x, flat):
    """One update with diagnostics on: [W, 2, 4] float64 (the destination starts at -7 so a missing write shows)."""
    d = torch.full((x.W, 2, 4), -7.0, device=DEV)
    eng.set_diagnostics(d, None)
    eng.update(x.storages, x.advs, x.idx, flat, torch.zeros_like(flat))
    eng.set_diagnostics(None, None)
    eng.check()
    return d.cpu().numpy().astype(np.float64)


# ------------------------------------------------------------------------------------------------ 1. constructed
@pytest.mark.parametrize("plan", ["uniform", "one_expert", "skewed"])
def test_constructed_ratios_give_exact_answers(plan):
    """old_lp / old_v set from the engine's own `evaluate` rows: no row is clipped; then chosen rows get d = +0.2
    (ratio 1.22, clipped) or +0.05 (ratio 1.05, not), and old_v = v -+ 0.2 (clipped) or -+ 0.05 (not): the clip
    fractions are exactly count * (1 / mb) and the KL terms the float64 means over the stored values. The routing plans
    put all rows of a head into one expert (three empty experts per head) or skew them."""
    from cadre_b200 import ppo, ppo_params as P
    W, mb, T = 4, 100, 200
    if plan != "uniform":
        assert ROUTING_PLANS[plan][:2] == (W, mb)
    x = _config_inputs(W, mb, T, 3100 if plan == "uniform" else _plan_seed(plan), None if plan == "uniform" else plan)
    flat = P.pack_state(R.ppo_fixture_state(0), DEV)
    eng = ppo.PpoEngine(W, mb, device=DEV)
    ev = eng.evaluate(x.storages, x.advs, x.idx, flat)
    v, lp = ev[:, :, 0].reshape(2, W, mb), ev[:, :, 1].reshape(2, W, mb)
    idx = torch.as_tensor(x.idx, dtype=torch.long, device=DEV)
    inv_mb = np.float32(1) / np.float32(mb)

    def store(d_lp, d_v):
        """old_lp = lp - d_lp, old_v = v - d_v on the minibatch rows; returns the stored (old_lp, old_v) [W, 2, mb]"""
        old = np.zeros((2, W, 2, mb))
        for w in range(W):
            for h in range(2):
                st = x.storages[w][h]
                st.action_log_probs[idx[w, h], 0] = lp[h, w] - torch.tensor(d_lp[w, h], dtype=torch.float32, device=DEV)
                st.value_preds[idx[w, h], 0] = v[h, w] - torch.tensor(d_v[w, h], dtype=torch.float32, device=DEV)
                old[0, w, h] = st.action_log_probs[idx[w, h], 0].double().cpu().numpy()
                old[1, w, h] = st.value_preds[idx[w, h], 0].double().cpu().numpy()
        return old

    zero = np.zeros((W, 2, mb))
    store(zero, zero)
    d = _diag_update(eng, x, flat)
    assert (d[..., 2] == 0).all() and (d[..., 3] == 0).all(), d
    assert np.abs(d[..., :2]).max() <= 1e-5, d[..., :2]
    print(f"{plan}: old_lp = evaluate's log-probs: |kl_k3| max {np.abs(d[..., 0]).max():.3e}, |kl_k1| max "
          f"{np.abs(d[..., 1]).max():.3e} ({'exactly 0' if not d[..., :2].any() else 'not exactly 0'})")

    i = np.arange(mb)
    d_lp, d_v = np.zeros((W, 2, mb)), np.zeros((W, 2, mb))
    for w in range(W):
        for h in range(2):
            g = (i + 3 * w + h) % 5
            d_lp[w, h] = np.where(g == 0, 0.2, np.where(g == 1, 0.05, 0.0))
            gv = (i + w + 2 * h) % 4
            sign = np.where(i % 2 == 0, 1.0, -1.0)
            d_v[w, h] = sign * np.where(gv == 0, 0.2, np.where(gv == 1, 0.05, 0.0))
    old = store(d_lp, d_v)
    d = _diag_update(eng, x, flat)
    lp64, v64 = lp.double().cpu().numpy(), v.double().cpu().numpy()
    for w in range(W):
        for h in range(2):
            dd = lp64[h, w] - old[0, w, h]
            assert d[w, h, 2] == np.float32(np.float32((d_lp[w, h] == 0.2).sum()) * inv_mb), (w, h, d[w, h])
            assert d[w, h, 3] == np.float32(np.float32((np.abs(d_v[w, h]) == 0.2).sum()) * inv_mb), (w, h, d[w, h])
            assert abs(d[w, h, 1] - np.mean(-dd)) <= 2e-5, (w, h, d[w, h, 1], np.mean(-dd))
            assert abs(d[w, h, 0] - np.mean(np.expm1(dd) - dd)) <= 2e-5, (w, h, d[w, h, 0])
            assert np.abs(v64[h, w] - old[1, w, h] - d_v[w, h]).max() < 1e-6     # the value shifts as stored


# ------------------------------------------------------------------------------------------------ 2. oracle
@pytest.mark.parametrize("W,mb,T,seed0", [(4, 100, 200, 300), (8, 400, 800, 700)])
def test_diagnostics_match_oracle(W, mb, T, seed0):
    """cfg 3 and cfg 5 on the seeded fixtures: KL terms within 1e-4 + 1e-3 rel of the float64 restatement on the
    oracle's rows; a clip fraction may differ only by rows that lie at the clip boundary within the forward's error
    (ratio: |ratio - 1| within 1e-4 of clip; value: |v - old_v| within twice the worst value error of the rows)."""
    from cadre_b200 import ppo, ppo_params as P
    torch.set_num_threads(min(16, os.cpu_count() or 1))
    x = _config_inputs(W, mb, T, seed0)
    sd = R.ppo_fixture_state(0)
    flat = P.pack_state(sd, DEV)
    eng = ppo.PpoEngine(W, mb, device=DEV)
    d = _diag_update(eng, x, flat)
    ev = eng.evaluate(x.storages, x.advs, x.idx, flat).double().cpu().numpy()
    u = SimpleNamespace(x=x, sd=sd)
    for h in range(2):
        rows = _oracle_rows(u, h).double().numpy()                       # [W * mb]: value, log-prob, entropy
        v_err = np.abs(ev[h, :, 0] - rows[:, 0]).max()
        for w in range(W):
            st, ix = x.cpu[w][0][h], torch.as_tensor(x.idx[w, h], dtype=torch.long)
            old_lp = st["action_log_probs"][ix, 0].double().numpy()
            old_v = st["value_preds"][ix, 0].double().numpy()
            r = rows[w * mb:(w + 1) * mb]
            ref = update_diagnostics(r[:, 1], old_lp, r[:, 0], old_v, CLIP)
            for k in (0, 1):
                assert abs(d[w, h, k] - ref[k]) <= 1e-4 + 1e-3 * abs(ref[k]), (w, h, k, d[w, h, k], ref[k])
            n_lp = near_clip_rows(r[:, 1], old_lp, CLIP, 1e-4)
            n_v = int(np.sum(np.abs(np.abs(r[:, 0] - old_v) - CLIP) <= 2 * v_err + 1e-6))
            assert abs(d[w, h, 2] - ref[2]) <= n_lp / mb + 1e-6, (w, h, d[w, h, 2], ref[2], n_lp)
            assert abs(d[w, h, 3] - ref[3]) <= n_v / mb + 1e-6, (w, h, d[w, h, 3], ref[3], n_v)
        print(f"W={W} mb={mb} {R.HEADS[h]}: kl_k3 {d[:, h, 0].mean():.4e}, clip frac {d[:, h, 2].mean():.3f}, "
              f"value clip frac {d[:, h, 3].mean():.3f}, worst value error {v_err:.2e}")


# ------------------------------------------------------------------------------------------------ 3. / 4. learner
def _filled_pool(W, T, seed, dev=DEV):
    from cadre_b200.learner import RolloutPool
    pool = RolloutPool(W, dict(num_steps=T, mini_batch_num=2, feature_dims=530, seq_length=8, use_gae=True,
                               gamma=0.99, tau=0.95), dev)
    rs = np.random.RandomState(seed)
    for w in range(W):
        for h, A in enumerate((R.STEER_ACTIONS, R.THROTTLE_ACTIONS)):
            c = R.synthetic_storage(rs, T=T, actions=A)
            for k in ("obs", "rewards", "value_preds", "action_log_probs", "action", "masks", "command"):
                getattr(pool.storages[w][h], k).copy_(c[k])
    pool.compute_returns(torch.from_numpy(rs.randn(W, 2).astype(np.float32)))
    return pool


SEEDS = [40, 41, 42, 43]


def _learner(diagnostics):
    from cadre_b200.learner import Learner
    return Learner(4, 100, R.ppo_fixture_state(0), DEV, seeds=SEEDS, diagnostics=diagnostics)


def _record_steps(learner):
    """Snapshot losses, gradient, Adam moments and parameters after every update step of the learner."""
    snaps = []
    step = learner._exchange_and_step

    def wrapped(s):
        step(s)
        snaps.append([t.clone() for t in (learner.losses, learner.grads, learner.exp_avg, learner.exp_avg_sq,
                                          learner.params)])
    learner._exchange_and_step = wrapped
    return snaps


def test_diagnostics_leave_training_bit_identical():
    """One learn() phase (4 epochs x 2 minibatches) with diagnostics off, on, and on again: every step's losses,
    gradient, exp_avg, exp_avg_sq and parameters are bit-identical, and so are the two runs' diagnostics."""
    pool = _filled_pool(4, 200, 11)
    runs = []
    for diag in (False, True, True):
        learner = _learner(diag)
        snaps = _record_steps(learner)
        assert learner.learn(pool, 4) == 8
        torch.cuda.synchronize()
        learner.check()
        runs.append((snaps, learner.diagnostics() if diag else None))
    names = ("losses", "grads", "exp_avg", "exp_avg_sq", "params")
    for k in range(8):
        for j, name in enumerate(names):
            assert torch.equal(runs[0][0][k][j], runs[1][0][k][j]), (k, name)
            assert torch.equal(runs[0][0][k][j], runs[2][0][k][j]), (k, name)
    d1, d2 = runs[1][1], runs[2][1]
    for key in ("approx_kl", "kl_k1", "clip_frac", "value_clip_frac", "grad_norm", "grad_clipped"):
        assert d1[key].shape[0] == 8 and np.array_equal(d1[key], d2[key]), key
    assert d1["approx_kl"].shape == (8, 4, 2) and d1["grad_norm"].shape == (8, 16)
    assert all(np.isfinite(d1[k]).all() for k in ("approx_kl", "kl_k1", "clip_frac", "value_clip_frac", "grad_norm"))
    assert (d1["approx_kl"] >= 0).all() and ((d1["clip_frac"] >= 0) & (d1["clip_frac"] <= 1)).all()


def test_staged_history_matches_single_steps():
    """The staged histories of a learn() phase against a fresh learner that runs the same indices one update_step at a
    time: each step's per-row block and grad_norm row are bit-identical, and grad_norm equals module_norms() read
    after that step."""
    from cadre_b200 import ppo
    pool = _filled_pool(4, 200, 12)
    a, b = _learner(True), _learner(True)
    n = a.learn(pool, 4)
    da = a.diagnostics()
    idx_all = np.concatenate([b.sample_epoch_indices(pool.storages) for _ in range(4)], 0)
    assert idx_all.shape[0] == n == 8
    for k in range(n):
        b.update_step(pool.storages, idx_all[k])
        db = b.diagnostics()
        norms = b.engine.module_norms()
        for key in ppo.DIAG_TERMS + ("grad_norm",):
            assert db[key].shape[0] == 1 and np.array_equal(da[key][k], db[key][0]), (k, key)
        assert np.array_equal(np.array([norms[m] for m in db["modules"]], np.float32), db["grad_norm"][0]), k
        assert np.array_equal(db["grad_clipped"][0], db["grad_norm"][0] > b.max_grad_norm)
    assert torch.equal(a.params, b.params)


def _rank(rank, world, port, out_dir, exchange):
    sys.path.insert(0, ROOT)
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), CADRE_ALLREDUCE=exchange,
                      CADRE_NO_ALLREDUCE_OVERLAP="0", CADRE_GRAD_GROUPS="2")
    import torch.distributed as dist
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    from cadre_b200.learner import Learner
    dev = f"cuda:{rank}"
    learner = Learner(2, 100, R.ppo_fixture_state(0), dev, seeds=[500 + 2 * rank + w for w in range(2)],
                      diagnostics=True)
    assert learner.exchange == exchange
    pool = _filled_pool(2, 200, 900 + rank, dev)
    learner.learn(pool, 2)
    learner.check()
    torch.save(learner.diagnostics(), os.path.join(out_dir, f"rank{rank}.pt"))
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.parametrize("exchange", ["nccl", "switch"])
def test_two_rank_grad_norm_history_is_identical(tmp_path, exchange):
    """Two ranks, pipelined gradient ranges (two expert groups, each clipped + stepped after its own all-reduce): the
    norms are taken after the all-reduce, so both ranks record the same grad_norm history bit for bit."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    mp.spawn(_rank, args=(2, port, str(tmp_path), exchange), nprocs=2, join=True)
    res = [torch.load(str(tmp_path / f"rank{r}.pt"), weights_only=False) for r in range(2)]
    assert res[0]["grad_norm"].shape == (4, 16) and np.isfinite(res[0]["grad_norm"]).all()
    assert np.array_equal(res[0]["grad_norm"], res[1]["grad_norm"])


# ------------------------------------------------------------------------------------------------ 5. rollout stats
@pytest.mark.parametrize("T", [200, 800])
def test_pool_rollout_stats_match_numpy(T):
    """RolloutPool.rollout_stats after compute_returns, with episode ends (masks 0) and done workers (next value 0),
    against numpy float64 on the same returns / values; a storage with constant returns gives NaN explained variance."""
    from cadre_b200 import ppo
    from cadre_b200.learner import RolloutPool
    W = 8
    pool = RolloutPool(W, dict(num_steps=T, mini_batch_num=2, feature_dims=530, seq_length=8, use_gae=True,
                               gamma=0.99, tau=0.95), DEV)
    g = torch.Generator().manual_seed(T)
    b = pool.batched
    b["rewards"].copy_(torch.rand(2 * W, T + 1, 1, generator=g))
    b["value_preds"].copy_(torch.randn(2 * W, T + 1, 1, generator=g))
    b["masks"].copy_((torch.rand(2 * W, T + 1, 1, generator=g) > 0.05).float())
    nv = torch.randn(W, 2, generator=g)
    nv[1] = 0.0                                                        # a done worker
    pool.compute_returns(nv)
    got = pool.rollout_stats()
    ref = rollout_stats_f64(b["returns"][..., 0].cpu().numpy(), b["value_preds"][..., 0].cpu().numpy())
    for k, name in enumerate(ppo.ROLLOUT_STATS):
        assert got[name].shape == (W, 2) and got[name].dtype == np.float32
        np.testing.assert_allclose(got[name].reshape(-1), ref[:, k], rtol=1e-5, atol=1e-5 * max(1.0, np.abs(ref[:, k]).max()),
                                   err_msg=name)
    b["returns"][3, :T] = 1.25                                         # storage 3 (worker 1, throttle): constant
    got = pool.rollout_stats()
    assert np.isnan(got["explained_variance"][1, 1]) and got["return_std"][1, 1] == 0.0
    assert np.isfinite(np.delete(got["explained_variance"].reshape(-1), 3)).all()


def test_rollout_stats_128_sequences_T800():
    """cfg 5's shape (64 environments x 2 heads, T = 800) straight through ppo.gae + ppo.rollout_stats."""
    from cadre_b200 import ppo
    E, T = 128, 800
    g = torch.Generator(device=DEV).manual_seed(5)
    r = torch.rand(E, T + 1, device=DEV, generator=g)
    v = torch.randn(E, T + 1, device=DEV, generator=g) * 2 + 0.5
    m = (torch.rand(E, T + 1, device=DEV, generator=g) > 0.02).float()
    ret, adv = torch.zeros(E, T + 1, device=DEV), torch.zeros(E, T, device=DEV)
    ppo.gae(r, v, m, torch.randn(E, device=DEV, generator=g), ret, adv)
    got = ppo.rollout_stats(ret, v).cpu().numpy().astype(np.float64)
    ref = rollout_stats_f64(ret.cpu().numpy(), v.cpu().numpy())
    np.testing.assert_allclose(got, ref, rtol=1e-5, atol=1e-6)
    assert np.isfinite(got).all()


# ------------------------------------------------------------------------------------------------ 6. training loop
def test_train_loop_with_diagnostics():
    """train(diagnostics=True, device_rollout=True) for two episodes: finite diagnostics in every history entry, one
    extra log line per episode, and parameters bit-identical to the same run with diagnostics off."""
    from cadre_b200.config import load_config
    from cadre_b200.train import train
    params, hists, logs = [], [], []
    for diag in (False, True):
        cfg = load_config()
        cfg.rollout_cfg.num_steps = 8
        cfg.rollout_cfg.mini_batch_num = 2
        cfg.train_cfg.log_interval = 1
        cfg.env_cfg["done_prob"] = 0.1
        lines = []
        learner, hist = train(0, cfg.train_cfg, cfg.agent_cfg, cfg.env_cfg, cfg.rollout_cfg, R.danet_fixture_state(0),
                              ppo_state=R.ppo_fixture_state(0), workers=2, max_episode=2, device_rollout=True,
                              log=lines.append, diagnostics=diag)
        params.append(learner.params.clone())
        hists.append(hist)
        logs.append(lines)
    assert torch.equal(params[0], params[1])
    assert [h[:3] for h in hists[1]] == hists[0] and all(len(h) == 3 for h in hists[0])
    steps = 2 * load_config().train_cfg.ppo_epoch
    for entry in hists[1]:
        d = entry[3]
        assert d["approx_kl"].shape == (steps, 2, 2) and d["grad_norm"].shape == (steps, 16)
        for key in ("approx_kl", "kl_k1", "clip_frac", "value_clip_frac", "grad_norm", "explained_variance",
                    "adv_mean", "adv_std", "return_mean", "return_std", "value_mean"):
            assert np.isfinite(d[key]).all(), key
    assert logs[1][0::2] == logs[0] and len(logs[1]) == 4 and "approx kl" in logs[1][1]
    print(logs[1][1])
