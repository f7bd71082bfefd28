"""Training checkpoints on the GPU: a run of 4 episodes equals 2 episodes with checkpoint_dir followed by
resume="latest" up to 4, bit for bit (params, Adam moments and step, history, pool tensors and cursors, actor,
environments, RNG states), on every acting path, with target-KL stops on both sides of the checkpoint, with
diagnostics, in a fresh process and across two ranks; plus the replica check, in-place loading, no files without
checkpoint_dir, and the reference-format snapshot read back by eval.load_agent_group."""
import math
import os
import socket
import sys

import numpy as np
import pytest
import torch
import torch.multiprocessing as mp

from oracle import restate as R

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _cfg(**train):
    from cadre_b200.config import load_config
    cfg = load_config()
    cfg.rollout_cfg.num_steps = 8
    cfg.rollout_cfg.mini_batch_num = 2
    cfg.train_cfg.log_interval = 1
    cfg.train_cfg.save_interval = 2
    cfg.train_cfg.update(train)
    cfg.env_cfg["done_prob"] = 0.1
    return cfg


def _train(max_episode, checkpoint_dir=None, resume=None, seed=1234, rank=0, train_cfg=None, **kw):
    """One train() call on cuda:(rank % GPUs) with 2 workers; returns (learner, history, log lines)."""
    from cadre_b200.train import train
    cfg = _cfg(**(train_cfg or {}))
    cfg.agent_cfg.model_cfg.device_num = cfg.agent_cfg.model_cfg.vae_device = rank % torch.cuda.device_count()
    torch.manual_seed(seed)
    lines = []
    learner, hist = train(rank, cfg.train_cfg, cfg.agent_cfg, cfg.env_cfg, cfg.rollout_cfg, R.danet_fixture_state(0),
                          ppo_state=R.ppo_fixture_state(0), workers=2, max_episode=max_episode,
                          checkpoint_dir=checkpoint_dir, resume=resume, log=lines.append, **kw)
    return learner, hist, lines


def _equal(a, b, where="state"):
    """Deep, bit-exact equality of checkpoint contents (NaN equals NaN)."""
    assert type(a) is type(b), (where, type(a), type(b))
    if isinstance(a, dict):
        assert list(a) == list(b), (where, list(a), list(b))
        for k in a:
            _equal(a[k], b[k], f"{where}.{k}")
    elif isinstance(a, (list, tuple)):
        assert len(a) == len(b), where
        for i, (x, y) in enumerate(zip(a, b)):
            _equal(x, y, f"{where}[{i}]")
    elif isinstance(a, torch.Tensor):
        assert a.dtype == b.dtype and a.shape == b.shape, where
        assert torch.equal(a.contiguous().view(-1).view(torch.uint8), b.contiguous().view(-1).view(torch.uint8)), where
    elif isinstance(a, np.ndarray):
        np.testing.assert_array_equal(a, b, err_msg=where)
    elif isinstance(a, float):
        assert a == b or (math.isnan(a) and math.isnan(b)), (where, a, b)
    else:
        assert a == b, (where, a, b)


def _files(path, rank=0):
    from cadre_b200 import checkpoint as C
    return (torch.load(os.path.join(path, C.LEARNER_FILE), weights_only=False),
            torch.load(os.path.join(path, C.rank_file(rank)), weights_only=False))


def _summary(learner, history):
    return dict(params=learner.params.cpu(), exp_avg=learner.exp_avg.cpu(), exp_avg_sq=learner.exp_avg_sq.cpu(),
                step_count=learner.step_count, history=history)


def _resume_in_fresh_process(_, path, out, kw):
    sys.path.insert(0, ROOT)
    learner, hist, _ = _train(4, path, "latest", seed=99, **kw)
    torch.save(_summary(learner, hist), out)


CASES = {
    "default": dict(),                                    # batched acting: torch.multinomial on the CUDA generator
    "default_fresh_process": dict(),
    "per_worker_act": dict(batched_acting=False),         # CadreAgent.act: Categorical.sample on the CPU generator
    "device_rollout": dict(device_rollout=True),
    "device_rollout_target_kl": dict(device_rollout=True, train_cfg=dict(target_kl=1e-6)),
    "diagnostics": dict(diagnostics=True),
}


@pytest.mark.parametrize("case", list(CASES))
def test_resume_is_bit_exact(tmp_path, case):
    kw = CASES[case]
    straight_dir, split = str(tmp_path / "straight"), str(tmp_path / "split")
    straight = _train(4, straight_dir, **kw)
    first = _train(2, split, **kw)
    assert len(first[1]) == 2
    assert sorted(os.listdir(split)) == ["ep_1", "ep_2", "models"]
    if case == "default_fresh_process":
        out = str(tmp_path / "resumed.pt")
        mp.spawn(_resume_in_fresh_process, args=(split, out, kw), nprocs=1, join=True)
        resumed = torch.load(out, weights_only=False)
    else:
        learner, hist, lines = _train(4, split, "latest", seed=99, **kw)   # another seed: the RNG states are restored
        assert any(line.startswith("Resume: ") and "ep_2" in line for line in lines), lines
        resumed = _summary(learner, hist)
    _equal(_summary(*straight[:2]), resumed)
    assert sorted(os.listdir(split)) == ["ep_1", "ep_2", "ep_3", "ep_4", "models"]
    assert sorted(os.listdir(os.path.join(split, "models"))) == ["ppo_model_0.pt", "ppo_model_2.pt"]
    assert sorted(os.listdir(straight_dir)) == ["ep_1", "ep_3", "ep_4", "models"]
    for ep in ("ep_1", "ep_3", "ep_4"):     # params, moments, step, config, pool, cursors, actor, envs, obs, RNG, history
        _equal(_files(os.path.join(straight_dir, ep)), _files(os.path.join(split, ep)), ep)
    if "target_kl" in case:
        stops = [int(line.split(",")[0].split()[1]) for line in straight[2] if "early stop at update step" in line]
        assert stops and min(stops) < 2 <= max(stops), straight[2]
    if case == "default":
        plain = _train(4, None, **kw)     # checkpointing does not change the trajectory
        _equal(_summary(*plain[:2]), _summary(*straight[:2]))


def test_no_checkpoint_dir_writes_nothing(tmp_path, monkeypatch):
    work = tmp_path / "cwd"
    work.mkdir()
    monkeypatch.chdir(work)
    learner, hist, _ = _train(2, train_cfg=dict(save_interval=1))
    assert len(hist) == 2 and os.listdir(work) == []


def test_snapshot_loads_through_eval(tmp_path):
    """models/ppo_model_<ep>.pt of the last episode, read by eval.load_agent_group into an agent of other parameters,
    acts like an agent on the learner's live parameters."""
    from cadre_b200.agent import CadreAgent
    from cadre_b200.eval import load_agent_group
    from cadre_b200.synthetic_env import SyntheticEnv
    learner, _, _ = _train(3, str(tmp_path))
    assert sorted(os.listdir(tmp_path / "models")) == ["ppo_model_0.pt", "ppo_model_2.pt"]
    cfg = _cfg()
    make = lambda: CadreAgent(**dict(cfg.agent_cfg, rank=0), danet_state=R.danet_fixture_state(0),  # noqa: E731
                              ppo_state=R.ppo_fixture_state(7))
    loaded, = load_agent_group(make, str(tmp_path), [2])
    live = make()
    live.owner.params = learner.params
    assert not torch.equal(loaded.owner.params, make().owner.params)
    assert torch.equal(loaded.owner.params, learner.params)
    env = SyntheticEnv(dict(seed=5))
    tick = env.reset()
    for _ in range(3):
        outs = []
        for agent in (loaded, live):
            torch.manual_seed(11)
            feat, actions, log_probs, values, _ = agent.act(tick)
            outs.append([feat.cpu(), torch.stack(actions), torch.cat(log_probs).cpu(), torch.cat(values).cpu()])
        for a, b in zip(*outs):
            assert torch.equal(a, b)
        tick = env.step([0.0, 0.5, 0.0])[0]


def test_load_state_dict_in_place(tmp_path):
    """Learner / RolloutPool / BatchedActor.load_state_dict copy into the existing tensors: the acting replica keeps
    aliasing the learner's params, the storages stay views of the pool."""
    from cadre_b200._lib import CadreError
    from cadre_b200.actor import BatchedActor
    from cadre_b200.agent import CadreAgent
    from cadre_b200.learner import Learner, RolloutPool
    cfg = _cfg()
    dev = torch.device("cuda:0")
    agent = CadreAgent(**dict(cfg.agent_cfg, rank=0), danet_state=R.danet_fixture_state(0),
                       ppo_state=R.ppo_fixture_state(0), mini_batch=4)
    learner = Learner(2, 4, R.ppo_fixture_state(0), dev, seeds=[1, 2])
    agent.owner.params = learner.params
    state = learner.state_dict()
    state["params"] += 1.0
    state["exp_avg"] += 2.0
    state["step_count"] = 17
    state["rng_states"] = [torch.manual_seed(5).get_state(), torch.manual_seed(6).get_state()]
    ptrs = [t.data_ptr() for t in (learner.params, learner.exp_avg, learner.exp_avg_sq)]
    learner.load_state_dict(state)
    assert agent.owner.params is learner.params
    assert [t.data_ptr() for t in (learner.params, learner.exp_avg, learner.exp_avg_sq)] == ptrs
    assert torch.equal(learner.params.cpu(), state["params"]) and torch.equal(learner.exp_avg.cpu(), state["exp_avg"])
    assert learner.step_count == 17 and torch.equal(learner._rng_states[1], state["rng_states"][1])
    bad = dict(state, param_count=state["param_count"] - 1)
    with pytest.raises(CadreError, match="parameters"):
        learner.load_state_dict(bad)
    with pytest.raises(CadreError, match="RNG"):
        learner.load_state_dict(dict(state, rng_states=state["rng_states"][:1]))

    pool = RolloutPool(2, dict(cfg.rollout_cfg, num_steps=8, hidden_size=530), dev)
    ps = pool.state_dict()
    ps["batched"]["obs"].normal_()
    ps["steps"] = [[3, 3], [3, 3]]
    view = pool.storages[1][0].obs.data_ptr()
    pool.load_state_dict(ps)
    assert pool.storages[1][0].obs.data_ptr() == view and pool.storages[1][1].step == 3
    assert torch.equal(pool.storages[1][0].obs.cpu(), ps["batched"]["obs"][2])

    actor = BatchedActor(agent, 2, seed=4, env_ids=[6, 7])
    st = actor.state_dict()
    st.update(ticks=9, env_ids=[8, 9])
    st["feats"].fill_(0.5)
    actor.load_state_dict(st)
    assert actor.ticks == 9 and actor._env_ids_d.tolist() == [8, 9] and actor._st[0].obs is actor.feats
    assert bool((actor.feats == 0.5).all())


# ------------------------------------------------------------------------------------------------ two ranks
def _rank(rank, world, port, out_dir, backend, exchange):
    sys.path.insert(0, ROOT)
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), CADRE_ALLREDUCE=exchange)
    import torch.distributed as dist
    from cadre_b200 import checkpoint as C
    from cadre_b200._lib import CadreError
    from cadre_b200.learner import Learner
    dev = torch.device("cuda", rank % torch.cuda.device_count())
    torch.cuda.set_device(dev)
    if backend == "nccl":
        dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    else:
        dist.init_process_group(backend, rank=rank, world_size=world)
    straight_dir, split = os.path.join(out_dir, "straight"), os.path.join(out_dir, "split")
    straight = _train(4, straight_dir, rank=rank, device_rollout=True)
    _train(2, split, rank=rank, device_rollout=True)
    resumed = _train(4, split, "latest", seed=99, rank=rank, device_rollout=True)
    _equal(_summary(*straight[:2]), _summary(*resumed[:2]))
    _equal(_files(os.path.join(straight_dir, "ep_4"), rank), _files(os.path.join(split, "ep_4"), rank))
    # a corrupted replica: the save raises on both ranks and leaves no COMPLETE marker
    learner = Learner(2, 4, R.ppo_fixture_state(0), dev, seeds=[1, 2])
    if rank == 1:
        learner.params[123] += 1e-3
    bad = os.path.join(out_dir, "bad")
    try:
        C.save(bad, 1, rank, learner, {}, {})
        corrupt = "saved"
    except CadreError as e:
        corrupt = str(e)
    torch.save(dict(params=resumed[0].params.cpu(), corrupt=corrupt), os.path.join(out_dir, f"rank{rank}.pt"))
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.parametrize("backend,exchange", [("gloo", "nccl"), ("nccl", "nccl"), ("nccl", "switch")])
def test_two_ranks_resume(tmp_path, backend, exchange):
    """Two ranks with device_rollout: each rank's resumed run equals its straight run bit for bit (checked inside the
    ranks), the replicas agree, a corrupted replica makes the save raise on both ranks, and resuming the two-rank
    checkpoint with world size 1 is refused. With the gloo backend both ranks share one GPU; exchange "nccl" is the
    torch.distributed.all_reduce path."""
    if backend == "nccl" and torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    from cadre_b200 import checkpoint as C
    from cadre_b200._lib import CadreError
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    mp.spawn(_rank, args=(2, port, str(tmp_path), backend, exchange), nprocs=2, join=True)
    res = [torch.load(str(tmp_path / f"rank{r}.pt"), weights_only=False) for r in range(2)]
    assert torch.equal(res[0]["params"], res[1]["params"])
    assert all("replicas of the ranks differ" in r["corrupt"] for r in res), [r["corrupt"] for r in res]
    assert C.latest(str(tmp_path / "bad")) is None
    assert sorted(os.listdir(tmp_path / "split" / "ep_4")) == ["COMPLETE", "learner.pt", "rank_0.pt", "rank_1.pt"]
    with pytest.raises(CadreError, match="world_size"):
        _train(4, str(tmp_path / "split"), "latest", device_rollout=True)
