"""Training checkpoints on the CPU: SyntheticEnv state round trip, durable saves and the choice of checkpoint to resume
from (a save that fails part-way is skipped), the config check (structural fields reject, hyperparameters are logged),
the encoder fingerprint and the replica check across two gloo ranks."""
import os
import socket
import sys
from types import SimpleNamespace

import numpy as np
import pytest
import torch
import torch.multiprocessing as mp

from cadre_b200 import checkpoint as C
from cadre_b200._lib import CadreError
from cadre_b200.config import load_config
from cadre_b200.synthetic_env import SyntheticEnv
from oracle import restate as R

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(env, n):
    out = []
    for _ in range(n):
        tick, reward, done, info = env.step([0.0, 0.5, 0.0])
        out.append((tick, reward.numpy().copy(), done, info["action_done"]))
        if done:
            out.append((env.reset(), None, None, None))
    return out


def _same(a, b):
    assert len(a) == len(b)
    for (ta, ra, da, ia), (tb, rb, db, ib) in zip(a, b):
        for k in ("rgb", "route_fig", "measurements"):
            assert np.array_equal(ta[k], tb[k]), k
        assert ta["command"] == tb["command"] and da == db and ia == ib
        assert (ra is None and rb is None) or np.array_equal(ra, rb)


@pytest.mark.parametrize("steps_before", [0, 5])
def test_synthetic_env_state_round_trip(steps_before):
    """set_state on a differently seeded env, then both envs give the same frames, rewards, dones and commands (with
    episode ends inside the compared window)."""
    a = SyntheticEnv(dict(seed=3, rank=1, done_prob=0.2, width=32, height=16))
    a.reset()
    _run(a, steps_before)
    state = a.get_state()
    b = SyntheticEnv(dict(seed=99, rank=0, done_prob=0.2, width=32, height=16))
    b.reset()
    b.set_state(state)
    ref = _run(a, 30)
    assert any(d for _, _, d, _ in ref if d)
    _same(ref, _run(b, 30))


def _stub_learner(seed=0, n=1000):
    """What checkpoint.save reads of a Learner, on the host, world size 1."""
    g = torch.Generator().manual_seed(seed)
    t = [torch.randn(n, generator=g) for _ in range(3)]
    rng = [torch.get_rng_state()]
    return SimpleNamespace(world=1, pg=None, params=t[0], exp_avg=t[1], exp_avg_sq=t[2], step_count=7,
                           state_dict=lambda: dict(params=t[0].clone(), exp_avg=t[1].clone(), exp_avg_sq=t[2].clone(),
                                                   step_count=7, param_count=n, rng_states=list(rng)))


def test_save_load_round_trip(tmp_path):
    lrn = _stub_learner()
    path = C.save(str(tmp_path), 3, 0, lrn, dict(a=1), dict(history=[[1.0, 2.0, 3.0]], pool="pool"))
    assert path == os.path.join(str(tmp_path), "ep_3") and C.is_complete(path)
    assert sorted(os.listdir(path)) == ["COMPLETE", "learner.pt", "rank_0.pt"]
    shared, mine = C.load(path, 0, dict(a=1))
    assert torch.equal(shared["learner"]["params"], lrn.params) and shared["learner"]["step_count"] == 7
    assert "rng_states" not in shared["learner"] and len(mine["rng_states"]) == 1
    assert mine["history"] == [[1.0, 2.0, 3.0]] and mine["pool"] == "pool" and mine["episodes"] == 3
    assert shared["replica_fingerprint"] == int(C.replica_fingerprint(lrn.params, lrn.exp_avg, lrn.exp_avg_sq))


def test_latest_skips_a_save_that_failed(tmp_path, monkeypatch):
    """A save whose rank-file write raises leaves a half-written temp file and no COMPLETE marker: latest() and
    resume="latest" take the previous checkpoint, resuming the failed one by path is refused."""
    root = str(tmp_path)
    assert C.latest(root) is None and C.resolve("latest", root) is None
    lrn = _stub_learner()
    C.save(root, 2, 0, lrn, {}, {})
    real_save = torch.save

    def failing(obj, f, *a, **k):
        if getattr(f, "name", "").endswith(C.rank_file(0) + ".tmp"):
            f.write(b"half a file")
            raise OSError("disk full")
        return real_save(obj, f, *a, **k)
    monkeypatch.setattr(torch, "save", failing)
    with pytest.raises(CadreError, match="failed to write"):
        C.save(root, 4, 0, lrn, {}, {})
    monkeypatch.undo()
    ep4 = os.path.join(root, "ep_4")
    assert sorted(os.listdir(ep4)) == ["learner.pt", "rank_0.pt.tmp"]
    os.makedirs(os.path.join(root, "ep_10"))                   # an empty directory and unrelated names are ignored
    os.makedirs(os.path.join(root, "ep_x"))
    assert C.latest(root) == os.path.join(root, "ep_2")
    assert C.resolve("latest", root) == os.path.join(root, "ep_2")
    with pytest.raises(CadreError, match="COMPLETE"):
        C.resolve(ep4, root)
    with pytest.raises(CadreError, match="checkpoint_dir"):
        C.resolve("latest", None)
    C.save(root, 4, 0, lrn, {}, {})                            # saving the episode again completes it
    assert C.latest(root) == ep4


def test_resave_removes_the_old_marker_first(tmp_path, monkeypatch):
    """Saving an episode that already has a complete checkpoint (a run resumed from an earlier one) takes its marker
    away before the files are replaced, so a failure in between cannot leave a COMPLETE directory of mixed files."""
    root = str(tmp_path)
    C.save(root, 2, 0, _stub_learner(0), {}, {})

    def no_space(*args):
        raise OSError("no space")
    monkeypatch.setattr(C, "_write_durable", no_space)
    with pytest.raises(CadreError):
        C.save(root, 2, 0, _stub_learner(1), {}, {})
    assert C.latest(root) is None


def _config(**over):
    cfg = load_config()
    cfg.train_cfg["target_kl"] = None
    c = C.run_config(1, 4, cfg.train_cfg, cfg.agent_cfg, cfg.env_cfg, cfg.rollout_cfg, 530, 19_000_000, True, False,
                     "abc")
    c.update(over)
    return c


CHANGED = dict(world_size=2, workers=8, num_steps=100, mini_batch_num=4, seq_length=4, feature_dims=512,
               hidden_size=256, param_count=1, env_seed=5, batched_acting=False, device_rollout=True,
               encoder_fingerprint="def")


def test_every_structural_field_is_checked():
    assert set(CHANGED) == set(C.STRUCTURAL)
    saved = _config()
    for k, v in CHANGED.items():
        with pytest.raises(CadreError, match=k):
            C.check_config(saved, _config(**{k: v}))


def test_hyperparameter_differences_are_logged_not_rejected():
    lines = []
    assert C.check_config(_config(), _config(), lines.append) == [] and lines == []
    diff = C.check_config(_config(), _config(lr=1e-4, target_kl=0.02, ppo_epoch=2), lines.append)
    assert diff == ["lr", "target_kl", "ppo_epoch"] and len(lines) == 1
    assert "lr 0.0003 -> 0.0001" in lines[0] and "target_kl None -> 0.02" in lines[0] and "ppo_epoch 4 -> 2" in lines[0]
    assert set(C.HYPERPARAMETERS) <= set(_config())


def test_encoder_fingerprint():
    sd = R.danet_fixture_state(0)
    fp = C.encoder_fingerprint(sd)
    assert fp == C.encoder_fingerprint(dict(reversed(list(sd.items()))))      # name order, not dict order
    name = next(k for k, v in sd.items() if v.dtype == torch.float32 and v.numel() > 1)
    changed = dict(sd)
    changed[name] = sd[name].clone()
    changed[name].view(-1)[0] = torch.nextafter(changed[name].view(-1)[0], torch.tensor(1e30))
    assert C.encoder_fingerprint(changed) != fp
    with pytest.raises(CadreError, match="encoder_fingerprint"):
        C.check_config(_config(encoder_fingerprint=fp), _config(encoder_fingerprint=C.encoder_fingerprint(changed)))


def test_replica_fingerprint_sees_one_word():
    g = torch.Generator().manual_seed(0)
    t = [torch.randn(n, generator=g) for n in (1000, 1000, 7)]
    fp = int(C.replica_fingerprint(*t))
    for k, i in ((0, 0), (1, 999), (2, 6)):
        u = [x.clone() for x in t]
        u[k].view(torch.int32)[i] ^= 1
        assert int(C.replica_fingerprint(*u)) != fp, (k, i)
    # the same words in another tensor (position) give another fingerprint
    assert int(C.replica_fingerprint(t[1], t[0], t[2])) != fp


def _rank(rank, world, port, root, corrupt):
    sys.path.insert(0, ROOT)
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    torch.distributed.init_process_group("gloo", rank=rank, world_size=world)
    from cadre_b200 import checkpoint as C
    lrn = _stub_learner()
    lrn.world = world
    if corrupt and rank == 1:
        lrn.params[5] += 1e-3
    try:
        C.save(root, 1, rank, lrn, {}, dict(rank=rank))
        res = "saved"
    except CadreError as e:
        res = str(e)
    torch.save(res, os.path.join(root, f"res{rank}.pt"))
    torch.distributed.barrier()
    torch.distributed.destroy_process_group()


@pytest.mark.parametrize("corrupt", [False, True])
def test_two_ranks_replica_check(tmp_path, corrupt):
    """Two gloo ranks: identical replicas give one complete checkpoint with a rank file each; one perturbed parameter on
    rank 1 makes the save raise on both ranks and leaves no COMPLETE marker."""
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    root = str(tmp_path)
    mp.spawn(_rank, args=(2, port, root, corrupt), nprocs=2, join=True)
    res = [torch.load(os.path.join(root, f"res{r}.pt")) for r in range(2)]
    if corrupt:
        assert all("replicas of the ranks differ" in r for r in res), res
        assert C.latest(root) is None
        assert not os.path.exists(os.path.join(root, "ep_1", "learner.pt"))
    else:
        assert res == ["saved", "saved"]
        assert C.latest(root) == os.path.join(root, "ep_1")
        assert [C.load(C.latest(root), r, {})[1]["rank"] for r in range(2)] == [0, 1]
