"""Target-KL early stopping on the GPU: off is untouched (bit-identical against a threshold that never triggers), a stop
at step k equals a phase of k steps (also past a 64-step staging chunk), a skipped step routes no rows, the decision is
global across two ranks, and the training loop logs the stop."""
import os
import socket
import sys

import numpy as np
import pytest
import torch
import torch.multiprocessing as mp

from oracle import restate as R
from test_diagnostics_gpu import _filled_pool
from test_target_kl_cpu import record_step, stop_rule

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
STATE = ("params", "exp_avg", "exp_avg_sq")


def _learner(W, mb, seeds, dev=DEV, **kw):
    from cadre_b200.learner import Learner
    return Learner(W, mb, R.ppo_fixture_state(0), dev, seeds=seeds, **kw)


def _on_policy_pool(W, T, seed, dev=DEV):
    """A filled pool whose stored log-probs are the fixture policy's own (the engine's evaluate): the KL of a phase
    starts near 0 and grows as the policy moves, so a threshold can be placed between steps."""
    from cadre_b200 import ppo_params as P
    pool = _filled_pool(W, T, seed, dev)
    return _relabel(pool, P.pack_state(R.ppo_fixture_state(0), dev), dev)


def _relabel(pool, params, dev=DEV):
    """Store the log-probs of the policy `params` in the pool, as a fresh rollout of it would."""
    from cadre_b200 import ppo
    W, T = pool.workers, pool.num_steps
    eng = ppo.PpoEngine(W, T, device=dev)
    idx = np.tile(np.arange(T, dtype=np.int32), (W, 2, 1))
    advs = [(s.advantages, t.advantages) for s, t in pool.storages]
    ev = eng.evaluate(pool.storages, advs, idx, params)
    for w in range(W):
        for h in range(2):
            pool.storages[w][h].action_log_probs[:T, 0] = ev[h, w * T:(w + 1) * T, 1]
    torch.cuda.synchronize(dev)
    return pool


def _phase_kl(W, mb, pool, seeds, ppo_epoch, lr=3e-4):
    """KL of every step of one phase with target_kl off (from the diagnostics) and the per-step losses."""
    learner = _learner(W, mb, seeds, diagnostics=True, lr=lr)
    losses = []
    step = learner._exchange_and_step

    def wrapped(s):
        step(s)
        losses.append(learner.losses.clone())
    learner._exchange_and_step = wrapped
    learner.learn(pool, ppo_epoch)
    d = learner.diagnostics()
    return stop_rule(d["approx_kl"], 1.0)[0], losses, d


def _draws(learner, pool, ppo_epoch):
    return np.concatenate([learner.sample_epoch_indices(pool.storages) for _ in range(ppo_epoch)], 0)


def _assert_same_state(a, b, what):
    for name in STATE:
        assert torch.equal(getattr(a, name), getattr(b, name)), (what, name)
    assert a.step_count == b.step_count, (what, a.step_count, b.step_count)


# ------------------------------------------------------------------------------------------------ 1. off is untouched
@pytest.mark.parametrize("W,mb,T", [(4, 100, 200), (8, 400, 800)])
def test_target_kl_that_never_triggers_leaves_training_bit_identical(W, mb, T):
    """One learn() phase with target_kl=None and with target_kl=1e9: every step's losses, gradient, Adam moments and
    parameters, the engine's launch count, the final Adam step and both scaled_losses are bit-identical; the gated
    learner reports every step applied."""
    pool = _filled_pool(W, T, 21)
    seeds = [40 + w for w in range(W)]
    runs = []
    for tkl in (None, 1e9):
        learner = _learner(W, mb, seeds, target_kl=tkl)
        snaps = []
        step = learner._exchange_and_step

        def wrapped(s, learner=learner, step=step, snaps=snaps):
            step(s)
            snaps.append([t.clone() for t in (learner.grads, learner.exp_avg, learner.exp_avg_sq, learner.params)])
        learner._exchange_and_step = wrapped
        assert learner.learn(pool, 4) == 8
        learner.check()
        losses = [learner._loss_hist[n].clone() for n in range(8)] if tkl else None
        runs.append((learner, snaps, losses))
    (off, s_off, _), (on, s_on, l_on) = runs
    for n in range(8):
        for j, name in enumerate(("grads", "exp_avg", "exp_avg_sq", "params")):
            assert torch.equal(s_off[n][j], s_on[n][j]), (n, name)
    es = on.early_stop()
    assert es["steps"] == 8 and es["applied"] == 8 and es["stopped_at"] is None and np.isfinite(es["kl"]).all()
    assert torch.equal(off.losses, l_on[7])
    assert on.engine.launches == off.engine.launches
    assert on.step_count == off.step_count == 8
    assert torch.equal(off.scaled_losses(), on.scaled_losses())
    assert torch.equal(off.scaled_losses(mean=True), on.scaled_losses(mean=True))
    assert on.grads.shape == off.grads.shape


# ------------------------------------------------------------------------------------------------ 2. / 3. stop at k
def _stop_equals_short_phase(W, mb, T, ppo_epoch, lowest, lrs, prefer="last"):
    """A phase stopped at a step k >= lowest (the first learning rate of `lrs` whose ungated phase has a KL record
    there) checked against the ungated phase."""
    seeds = [60 + w for w in range(W)]
    pool = _on_policy_pool(W, T, 31)
    for lr in lrs:
        kl, losses, d_off = _phase_kl(W, mb, pool, seeds, ppo_epoch, lr)
        rec = record_step(kl, lowest=lowest, prefer=prefer)
        if rec is not None:
            break
    steps = kl.shape[0]
    assert rec is not None, f"no step >= {lowest} sets a KL record by 1e-3: {kl}"
    k, tkl = rec
    b = _learner(W, mb, seeds, diagnostics=True, lr=lr, target_kl=tkl)
    assert b.learn(pool, ppo_epoch) == steps
    b.check()
    es = b.early_stop()
    assert es["stopped_at"] == k and es["applied"] == k and es["steps"] == steps, (es, k, kl)
    assert np.isfinite(es["kl"][:k + 1]).all() and np.isnan(es["kl"][k + 1:]).all()
    np.testing.assert_allclose(es["kl"][:k + 1], kl[:k + 1], rtol=1e-5)
    assert es["kl"][k] > 1.5 * np.float32(tkl) >= es["kl"][:k].max()
    # losses: the mean over steps 0..k (the one that stopped included) and the last of them, bit for bit
    s = torch.zeros_like(losses[0])
    for n in range(k + 1):
        s += losses[n]
    coeffs = torch.tensor([b.value_coeff, b.clip_coeff, b.ent_coeff])
    assert torch.equal(b.scaled_losses(mean=True), (s / (k + 1)).sum(1).cpu() * coeffs)
    assert torch.equal(b.scaled_losses(), losses[k].sum(1).cpu() * coeffs)
    # diagnostics: rows 0..k those of the ungated phase, later rows NaN
    d = b.diagnostics()
    assert d["stopped_at"] == k and (d["applied"] == (np.arange(steps) < k)).all()
    for key in ("approx_kl", "clip_frac", "grad_norm"):
        assert np.array_equal(d[key][:k + 1], d_off[key][:k + 1]), key
        assert np.isnan(d[key][k + 1:]).all(), key
    return pool, seeds, b, k, steps, lr


def _check_against_replay(W, mb, ppo_epoch, lr, pool, seeds, b, k):
    """b (gated, after one phase stopped at k) against a learner that ran the first k slices with update_step; then a
    second phase on both and one more update_step on both."""
    c = _learner(W, mb, seeds, lr=lr)
    idx = _draws(c, pool, ppo_epoch)
    for n in range(k):
        c.update_step(pool.storages, idx[n])
    _assert_same_state(b, c, "phase 1")
    assert b.step_count == k
    _relabel(pool, b.params)           # a new rollout of the current policy: the second phase starts below the threshold
    b.learn(pool, ppo_epoch)
    k2 = b.early_stop()["applied"]
    idx2 = _draws(c, pool, ppo_epoch)
    for n in range(k2):
        c.update_step(pool.storages, idx2[n])
    _assert_same_state(b, c, "phase 2")
    extra = _draws(c, pool, 1)[0]
    b.update_step(pool.storages, extra)
    c.update_step(pool.storages, extra)
    _assert_same_state(b, c, "update_step")
    b.check()
    return k2


def test_stop_at_step_k_equals_a_phase_of_k_steps():
    """cfg 3 shapes, 8 steps: stop at the last step that sets a KL record; params, moments and the Adam step equal k
    update_steps on the same slices, through a second phase and one more update_step."""
    pool, seeds, b, k, steps, lr = _stop_equals_short_phase(4, 100, 200, 4, 1, [3e-4])
    k2 = _check_against_replay(4, 100, 4, lr, pool, seeds, b, k)
    print(f"stop at {k} of {steps}; second phase applied {k2}")


def test_stop_past_a_staging_chunk():
    """80 steps in one phase (two staging chunks of 64 + 16): the stop comes at a step past 64, and the chunk boundary
    neither clears it nor restarts the Adam step."""
    pool, seeds, b, k, steps, lr = _stop_equals_short_phase(2, 100, 200, 40, 65, [3e-4, 1e-4])
    assert steps == 80 and k >= 65
    k2 = _check_against_replay(2, 100, 40, lr, pool, seeds, b, k)
    print(f"stop at {k} of {steps} (lr {lr}); second phase applied {k2}")


# ------------------------------------------------------------------------------------------------ 4. all experts empty
def test_skipped_step_routes_no_rows():
    """After a stop early in the phase the last step is skipped: its update routes no rows to any of the eight experts,
    so the whole gradient is exactly 0, its losses are 0 and the recurrence kernels report no timeout. The next phase
    then matches a fresh learner given the same parameters, moments, Adam step and RNG streams."""
    W, mb = 4, 100
    pool, seeds, b, k, steps, _ = _stop_equals_short_phase(W, mb, 200, 4, 1, [3e-4], prefer="first")
    assert k <= steps - 2
    assert not b.grads.any() and b.grads.numel() == b.params.numel()
    assert not b._loss_hist[k + 1:].any()
    b.check()
    f = _learner(W, mb, seeds, target_kl=b.target_kl)
    for name in STATE:
        getattr(f, name).copy_(getattr(b, name))
    f._step_count = b.step_count
    f._rng_states = [s.clone() for s in b._rng_states]
    for x in (b, f):
        x.learn(pool, 4)
    assert b.early_stop()["applied"] == f.early_stop()["applied"]
    _assert_same_state(b, f, "next phase")
    assert torch.equal(b.scaled_losses(mean=True), f.scaled_losses(mean=True))


def test_engine_rejects_bad_target_kl_arguments():
    from cadre_b200 import _lib, ppo
    eng = ppo.PpoEngine(4, 16, device=DEV)
    kl = torch.zeros(4, device=DEV)
    with pytest.raises(_lib.CadreError, match="total_workers"):
        eng.set_target_kl(0.01, 3, kl)
    with pytest.raises(_lib.CadreError, match="kl_sum_dev"):
        eng.set_target_kl(0.01, 4, None)
    with pytest.raises(_lib.CadreError, match="not set"):
        eng.kl_gate()
    eng.set_target_kl(0.01, 8, kl)
    eng.set_target_kl(None)
    with pytest.raises(_lib.CadreError, match="not set"):
        eng.kl_gate()


def test_chief_steps_a_learner():
    """utils.chief (which does `optimizer.step_count += 1`) on a real Learner, with target_kl off and after a phase
    that stopped at its first step: the step count continues from the steps applied, and the parameters equal the
    engine's own clip + Adam at that step."""
    from types import SimpleNamespace
    from cadre_b200 import utils
    pool = _filled_pool(2, 200, 5)          # random stored log-probs: a tiny target_kl stops at step 0
    for tkl in (None, 1e-30):
        a = _learner(2, 100, [1, 2], target_kl=tkl)
        if tkl is not None:
            a.learn(pool, 1)
            assert a.early_stop()["stopped_at"] == 0
        assert a.step_count == 0
        ref = _learner(2, 100, [1, 2])
        for name in STATE:
            getattr(ref, name).copy_(getattr(a, name))
        g = torch.randn(a.params.numel(), generator=torch.Generator().manual_seed(3)).to(DEV)
        shared = SimpleNamespace(grads=g, reset=lambda: None)
        counter, light = utils.Counter(), utils.TrafficLight()
        counter.increment()
        assert utils.chief(1, light, counter, None, shared, a)
        ref.engine.adam_step(ref.params, g, ref.exp_avg, ref.exp_avg_sq, 1, 250.0, ref.lr)
        assert a.step_count == 1, tkl
        for name in STATE:
            assert torch.equal(getattr(a, name), getattr(ref, name)), (tkl, name)


# ------------------------------------------------------------------------------------------------ 5. two ranks
def _rank(rank, world, port, out_dir, backend, exchange, groups):
    sys.path.insert(0, ROOT)
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), CADRE_ALLREDUCE=exchange,
                      CADRE_NO_ALLREDUCE_OVERLAP="0", CADRE_GRAD_GROUPS=groups)
    import torch.distributed as dist
    dev = f"cuda:{rank % torch.cuda.device_count()}"
    torch.cuda.set_device(dev)
    if backend == "nccl":
        dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device(dev))
    else:
        dist.init_process_group(backend, rank=rank, world_size=world)
    W, mb, epochs = 2, 100, 4
    seeds = [500 + 2 * rank + w for w in range(W)]
    pool = _on_policy_pool(W, 200, 900 + rank, dev)

    def make(**kw):
        learner = _learner(W, mb, seeds, dev, **kw)
        assert learner.exchange == exchange
        return learner
    off = make(diagnostics=True)
    off.learn(pool, epochs)
    local = torch.from_numpy(off.diagnostics()["approx_kl"])                  # [steps, W, 2]
    local = local.to(dev) if backend == "nccl" else local
    every = [torch.zeros_like(local) for _ in range(world)]
    dist.all_gather(every, local)
    every = np.concatenate([t.cpu().numpy() for t in every], 1)               # [steps, world * W, 2]
    glob = stop_rule(every, 1.0)[0]
    locs = [stop_rule(every[:, r * W:(r + 1) * W], 1.0)[0] for r in range(world)]
    out = dict(glob=glob, locs=locs)
    rec = record_step(glob)
    if rec is not None:
        out["k"], tkl = rec
        on = make(target_kl=tkl)
        on.learn(pool, epochs)
        on.check()
        out["stop"] = on.early_stop()
        out["stop_params"] = on.params.cpu()
    # a threshold above every global KL of the phase but below the largest local KL of the rank with the larger one
    r_hi = int(np.argmax([l.max() for l in locs]))
    if locs[r_hi].max() > glob.max() * 1.001:
        out["local_rank"] = r_hi
        tkl = np.sqrt(locs[r_hi].max() * glob.max()) / 1.5
        quiet = make(target_kl=tkl)
        quiet.learn(pool, epochs)
        quiet.check()
        out["quiet"] = quiet.early_stop()
        out["quiet_params"] = quiet.params.cpu()
        out["off_params"] = off.params.cpu()
    torch.save(out, os.path.join(out_dir, f"rank{rank}.pt"))
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.parametrize("backend,exchange,groups", [("nccl", "nccl", "2"), ("nccl", "switch", "1"),
                                                    ("nccl", "switch", "2"), ("gloo", "nccl", "1"),
                                                    ("gloo", "nccl", "2")])
def test_two_ranks_stop_together(tmp_path, backend, exchange, groups):
    """Two ranks, different rollouts: both stop at the step the GLOBAL KL picks, with bit-identical replicas and
    early_stop() results; a threshold that one rank's local KL crosses but the global KL never does stops no rank.
    The KL sums ride in the single gradient range (groups "1"), or in a 16-byte exchange of their own before range 0
    (groups "2"). exchange "nccl" is the torch.distributed.all_reduce path: with the gloo backend both ranks share one
    GPU, so the learner's multi-rank ordering (tail exchange, gate after range 0's sum) runs on a one-GPU machine too."""
    if backend == "nccl" and torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    mp.spawn(_rank, args=(2, port, str(tmp_path), backend, exchange, groups), nprocs=2, join=True)
    res = [torch.load(str(tmp_path / f"rank{r}.pt"), weights_only=False) for r in range(2)]
    assert np.array_equal(res[0]["glob"], res[1]["glob"])
    assert "k" in res[0], f"no global KL record: {res[0]['glob']}"
    for r in range(2):
        es = res[r]["stop"]
        assert es["stopped_at"] == res[0]["k"] and es["applied"] == res[0]["k"], (r, es)
        np.testing.assert_array_equal(es["kl"], res[0]["stop"]["kl"])
    assert torch.equal(res[0]["stop_params"], res[1]["stop_params"])
    assert "local_rank" in res[0], "no rank's local KL exceeds the global maximum"
    for r in range(2):
        assert res[r]["quiet"]["stopped_at"] is None and res[r]["quiet"]["applied"] == res[r]["quiet"]["steps"], r
        assert torch.equal(res[r]["quiet_params"], res[r]["off_params"]), r
    assert torch.equal(res[0]["quiet_params"], res[1]["quiet_params"])


# ------------------------------------------------------------------------------------------------ 6. training loop
def test_train_loop_logs_early_stop():
    """train(device_rollout=True) with train_cfg.target_kl small enough to stop: the early-stop line is logged, history
    keeps its shape, and a second run gives bit-identical parameters and the same log."""
    from cadre_b200.config import load_config
    from cadre_b200.train import train
    params, hists, logs = [], [], []
    for _ in range(2):
        cfg = load_config()
        cfg.rollout_cfg.num_steps = 8
        cfg.rollout_cfg.mini_batch_num = 2
        cfg.train_cfg.log_interval = 1
        cfg.train_cfg.target_kl = 1e-6
        cfg.env_cfg["done_prob"] = 0.1
        lines = []
        learner, hist = train(0, cfg.train_cfg, cfg.agent_cfg, cfg.env_cfg, cfg.rollout_cfg, R.danet_fixture_state(0),
                              ppo_state=R.ppo_fixture_state(0), workers=2, max_episode=2, device_rollout=True,
                              log=lines.append)
        params.append(learner.params.clone())
        hists.append(hist)
        logs.append(lines)
    assert torch.equal(params[0], params[1]) and logs[0] == logs[1] and hists[0] == hists[1]
    assert len(hists[0]) == 2 and all(len(h) == 3 for h in hists[0])
    stops = [line for line in logs[0] if "early stop at update step" in line]
    assert stops and all("> 1.5 x 1.0e-06" in line for line in stops), logs[0]
    print(stops[0])
