"""Worker loop (reference: ppo_agent/train.py:14-127) against the synthetic environment, with the
parameter-server handshake (train.py:101-110 + chief.py) replaced by `Learner.update_step` (batched local
workers + NCCL all-reduce + replicated clip/Adam). `main()` is the per-GPU launcher that replaces main.py:25-72:
one process per GPU (torchrun), each stepping `workers_per_gpu` logical workers."""
import os

import numpy as np
import torch

from . import checkpoint
from .actor import BatchedActor
from .agent import CadreAgent
from .config import load_config
from .eval import snapshot_path
from .learner import Learner, RolloutPool
from .models import get_vae_output, init_state
from .synthetic_env import SyntheticEnv


def train(rank, train_cfg, agent_cfg, env_cfg, rollout_cfg, danet_state, ppo_state=None, workers=1, max_episode=None,
          process_group=None, log=print, batched_acting=True, device_rollout=False, diagnostics=False,
          checkpoint_dir=None, resume=None):
    """One rank: `workers` logical workers (env + rollout pair each) sharing one agent replica. With
    `batched_acting` the rank's workers are stepped together through `BatchedActor` (one encoder batch of the newest
    frames + one routed LSTM / head evaluation per tick) instead of one `agent.act` call per worker.
    `device_rollout` (needs `batched_acting`) draws the actions on the device and writes each tick into the rollout
    pool with a fixed number of launches and copies (`BatchedActor.act_into`, `RolloutPool.write_env_results`), and
    bootstraps all workers' values in one forward (`BatchedActor.bootstrap_into`). Its draws come from a counter-based
    generator keyed by (env seed, worker id, tick), not from torch's RNG, so its trajectories differ from the default
    path's.
    `diagnostics` records the PPO update diagnostics of every episode (`Learner.diagnostics`, `RolloutPool.rollout_stats`):
    each `history` entry gains a dict of them as a fourth element, and rank 0 logs one more line per `log_interval`.
    Values are those of this rank's workers. Training itself is unchanged.
    `train_cfg.target_kl` (absent or None: off) stops each PPO phase early by SB3's rule (`Learner(target_kl=...)`);
    rank 0 logs one more line per `log_interval` when the phase stopped.
    `checkpoint_dir` (None: no file is written): rank 0 writes the reference's snapshot
    `<checkpoint_dir>/models/ppo_model_<episode>.pt` after every episode with episode % save_interval == 0
    (train.py:121-123), and at those points and after the last episode every rank takes part in a training checkpoint
    `<checkpoint_dir>/ep_<episodes completed>` (`cadre_b200.checkpoint`). `resume`: "latest" (the newest complete
    checkpoint under `checkpoint_dir`; none yet: start from episode 0) or an ep_<n> directory. The resumed run continues
    the same trajectory bit for bit, needs the same structural config (world size, workers per rank, shapes, env seed,
    acting path, encoder weights) and takes the hyperparameters from the current config. `max_episode` counts all
    episodes of the run, and the returned `history` includes the restored entries."""
    if device_rollout and not batched_acting:
        raise ValueError("device_rollout=True needs batched_acting=True")
    device = torch.device("cuda:" + str(agent_cfg.model_cfg.device_num))
    envs = [SyntheticEnv(dict(env_cfg, rank=rank * workers + w, seq_length=rollout_cfg.seq_length))
            for w in range(workers)]
    hidden_size, _ = get_vae_output(agent_cfg.model_cfg)
    ppo_state = ppo_state if ppo_state is not None else init_state(seed=0)
    num_steps = rollout_cfg.num_steps
    mb = num_steps // rollout_cfg.mini_batch_num
    agent = CadreAgent(**dict(agent_cfg, rank=rank), danet_state=danet_state, ppo_state=ppo_state, mini_batch=mb)
    learner = Learner(workers, mb, ppo_state, device, agent_cfg.clip, agent_cfg.value_coeff, agent_cfg.clip_coeff,
                      agent_cfg.ent_coeff, train_cfg.lr, train_cfg.max_grad_norm, process_group,
                      seeds=[env_cfg.get("seed", 0) + rank * workers + w for w in range(workers)],
                      diagnostics=diagnostics, target_kl=train_cfg.get("target_kl"))
    agent.owner.params = learner.params          # the acting replica reads the learner's parameters directly
    pool = RolloutPool(workers, dict(rollout_cfg, hidden_size=hidden_size), device)
    obs = [e.reset() for e in envs]
    done = [False] * workers
    history = []
    if device_rollout:   # the same env ids as the SyntheticEnvs: a rollout split over ranks draws what one rank would
        actor = BatchedActor(agent, workers, seed=env_cfg.get("seed", 0),
                             env_ids=[rank * workers + w for w in range(workers)])
    else:
        actor = BatchedActor(agent, workers) if batched_acting else None
    total = max_episode if max_episode is not None else train_cfg.max_episode
    start = 0
    if checkpoint_dir is not None or resume is not None:
        ckpt_cfg = checkpoint.run_config(learner.world, workers, train_cfg, agent_cfg, env_cfg, rollout_cfg, hidden_size,
                                         learner.params.numel(), batched_acting, device_rollout,
                                         checkpoint.encoder_fingerprint(danet_state))
    if resume is not None:
        path = checkpoint.resolve(resume, checkpoint_dir)
        if path is None:
            if rank == 0:
                log(f"Resume: no complete checkpoint under {checkpoint_dir}, starting from episode 0")
        else:
            start, history = _restore(path, rank, ckpt_cfg, learner, pool, actor, envs, obs, done, device,
                                      log if rank == 0 else None)
            if rank == 0:
                log(f"Resume: {path}, {start} episodes done")
    for episode in range(start, total):
        if device_rollout:
            _device_rollout(actor, agent, envs, pool, obs, done, num_steps)
            actor.bootstrap_into(pool, done)                              # train.py:76-79, into pool.next_value
            nv = None
        else:
            for _ in range(num_steps):                                    # train.py:55-74
                acted = actor.act(obs) if actor is not None else None
                for w, env in enumerate(envs):
                    command = obs[w]["command"]
                    feat, action, logp, value, hidden = acted[w] if acted is not None else agent.act(obs[w])
                    obs[w], reward, done[w], info = env.step(agent.convert_action(action))
                    for h in range(2):
                        mask = torch.tensor([[0.0] if info["action_done"][h] else [1.0]])
                        pool.storages[w][h].insert(feat, action[h], logp[h], value[h], reward[h], mask, hidden, command)
                    if done[w]:
                        obs[w] = env.reset()
                        if actor is not None:
                            actor.reset(w)
            nv = torch.zeros(workers, 2)
            for w in range(workers):                                      # train.py:76-79
                vs, vt = agent.get_value(done[w], pool.storages[w][0].get_last(), pool.storages[w][1].get_last())
                nv[w, 0], nv[w, 1] = float(vs.reshape(-1)[0]), float(vt.reshape(-1)[0])
        pool.compute_returns(nv, normalize=train_cfg.use_adv_norm)        # train.py:81-88
        learner.learn(pool, train_cfg.ppo_epoch)                          # train.py:93-110
        L = learner.scaled_losses(mean=True).mean(0)     # mean over update steps and workers
        history.append(L.tolist())
        if diagnostics:
            diag = dict(learner.diagnostics(), **pool.rollout_stats())
            history[-1].append(diag)
        if episode % train_cfg.log_interval == 0 and rank == 0:
            log("Episode: {}, value loss: {:.4f}, policy loss: {:.4f}, entropy loss: {:.4f}".format(episode, *L))
            if diagnostics:
                log(_diagnostics_line(episode, diag))
            if learner.target_kl is not None:
                es = learner.early_stop()
                if es["stopped_at"] is not None:
                    log("Episode: {}, early stop at update step {} of {} (kl {:.1e} > 1.5 x {:.1e})".format(
                        episode, es["stopped_at"], es["steps"], es["kl"][es["stopped_at"]], learner.target_kl))
        if checkpoint_dir is not None and (episode % train_cfg.save_interval == 0 or episode == total - 1):
            if rank == 0 and episode % train_cfg.save_interval == 0:         # train.py:121-123
                os.makedirs(os.path.join(checkpoint_dir, "models"), exist_ok=True)
                agent.save_snapshot(snapshot_path(checkpoint_dir, episode))
            rank_state = dict(pool=pool.state_dict(), actor=actor.state_dict() if actor is not None else None,
                              envs=[e.get_state() if hasattr(e, "get_state") else None for e in envs],
                              obs=list(obs), done=list(done), history=history,
                              cpu_rng=torch.get_rng_state(), cuda_rng=torch.cuda.get_rng_state(device))
            checkpoint.save(checkpoint_dir, episode + 1, rank, learner, ckpt_cfg, rank_state)
    return learner, history


def _restore(path, rank, cfg, learner, pool, actor, envs, obs, done, device, log):
    """Load checkpoint `path` into this rank's learner, pool, actor, environments, per-worker `obs` / `done` (updated in
    place) and RNG states. Returns (episodes completed, history). An environment without get_state / set_state (e.g.
    CARLA's) is left freshly reset: training continues, but not on the same trajectory."""
    shared, mine = checkpoint.load(path, rank, cfg, log)
    learner.load_state_dict(dict(shared["learner"], rng_states=mine["rng_states"]))
    checkpoint.check_restored(learner, shared)
    pool.load_state_dict(mine["pool"])
    if actor is not None:
        actor.load_state_dict(mine["actor"])
    for w, (env, st) in enumerate(zip(envs, mine["envs"])):
        if st is not None and hasattr(env, "set_state"):
            env.set_state(st)
            obs[w], done[w] = mine["obs"][w], mine["done"][w]
        elif actor is not None:
            actor.reset(w)
    torch.set_rng_state(mine["cpu_rng"])
    torch.cuda.set_rng_state(mine["cuda_rng"], device)
    return mine["episodes"], list(mine["history"])


def _diagnostics_line(episode, d):
    """One log line: per head (steer / throttle) the mean approximate KL and clip fraction over the phase's update steps
    and the workers, the explained variance (mean over workers), and the largest module gradient norm of the phase with
    the number of modules clipped in at least one step."""
    kl, cf = d["approx_kl"].mean((0, 1)), d["clip_frac"].mean((0, 1))
    ev = [np.nanmean(c) if np.isfinite(c).any() else np.nan for c in d["explained_variance"].T]
    return ("Episode: {}, approx kl: {:.2e} / {:.2e}, clip fraction: {:.3f} / {:.3f}, explained variance: {:.3f} / {:.3f}, "
            "max grad norm: {:.2f}, modules clipped: {} of 16".format(
                episode, kl[0], kl[1], cf[0], cf[1], ev[0], ev[1], d["grad_norm"].max(),
                int(d["grad_clipped"].any(0).sum())))


def _device_rollout(actor, agent, envs, pool, obs, done, num_steps):
    """num_steps ticks of train.py:55-74 through the device path: act_into -> env.step x W -> write_env_results."""
    W = len(envs)
    rewards = np.zeros((W, 2), dtype=np.float32)
    masks = np.zeros((W, 2), dtype=np.float32)
    for _ in range(num_steps):
        slot = pool.storages[0][0].step
        actions = actor.act_into(obs, pool)
        for w, env in enumerate(envs):
            obs[w], reward, done[w], info = env.step(agent.convert_action(actions[w]))
            rewards[w] = reward
            masks[w] = [0.0 if d else 1.0 for d in info["action_done"]]
            if done[w]:
                obs[w] = env.reset()
                actor.reset(w)
        pool.write_env_results(slot, rewards, masks)


def main():
    cfg = load_config(os.environ.get("CADRE_CONFIG") or None) if os.environ.get("CADRE_CONFIG") else load_config()
    rank = int(os.environ.get("RANK", 0))
    local = int(os.environ.get("LOCAL_RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    torch.cuda.set_device(local)
    if world > 1:
        os.environ.setdefault("NCCL_ALGO", "Ring")   # faster than NCCL's default for the 36 - 78 MB gradient ranges (8 x B200)
        torch.distributed.init_process_group("nccl", device_id=torch.device("cuda", local))
    cfg.agent_cfg.model_cfg.device_num = cfg.agent_cfg.model_cfg.vae_device = local
    ckpt = os.environ.get("CADRE_ENCODER_CKPT")
    if not ckpt:
        raise SystemExit("set CADRE_ENCODER_CKPT to the reference perception checkpoint ({'autoencoder': state_dict})")
    danet_state = torch.load(ckpt, map_location="cpu")["autoencoder"]
    # env_cfg.num_processes logical workers in total (main.py:41-60), split evenly over the ranks. Gradients are SUMMED
    # over workers like the reference (models.py:231-239), so the effective step (clip at max_grad_norm, Adam's eps)
    # depends on the total worker count: it must match the configured one, not grow with the number of GPUs.
    if cfg.env_cfg.num_processes % world:
        raise SystemExit(f"env_cfg.num_processes={cfg.env_cfg.num_processes} is not divisible by WORLD_SIZE={world}")
    workers = cfg.env_cfg.num_processes // world
    # CADRE_CHECKPOINT_DIR: snapshots + training checkpoints; CADRE_RESUME: "latest" or an ep_<n> directory
    train(rank, cfg.train_cfg, cfg.agent_cfg, cfg.env_cfg, cfg.rollout_cfg, danet_state, workers=workers,
          checkpoint_dir=os.environ.get("CADRE_CHECKPOINT_DIR") or None, resume=os.environ.get("CADRE_RESUME") or None)


if __name__ == "__main__":
    main()
