"""Rollout collection cost per tick: the existing loop body (BatchedActor.act + 2W RolloutStorage.insert) against the
device path (BatchedActor.act_into + RolloutPool.write_env_results), W workers of SyntheticEnv, T = 200, and the
bootstrap (W x CadreAgent.get_value against BatchedActor.bootstrap_into). Each per-tick figure is split into host
env.step time (the synthetic env draws ~147 KB of random frame data per env per tick) and everything else.
Prints the card name and power limit of the run. Usage: python tools/gpu_probe_rollout.py [W ...]"""
import os
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from cadre_b200 import fixtures as R                    # noqa: E402
from cadre_b200.actor import BatchedActor               # noqa: E402
from cadre_b200.agent import CadreAgent                 # noqa: E402
from cadre_b200.config import load_config               # noqa: E402
from cadre_b200.learner import RolloutPool              # noqa: E402
from cadre_b200.synthetic_env import SyntheticEnv       # noqa: E402

T, WARM = 200, 8


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=30).stdout.strip().splitlines()[0]
    except Exception as e:      # the name still comes from torch
        q = f"{torch.cuda.get_device_name(0)}, power limit unknown ({e})"
    return q


def make(W):
    envs = [SyntheticEnv(dict(rank=w, seq_length=8)) for w in range(W)]
    pool = RolloutPool(W, dict(num_steps=T, mini_batch_num=2, feature_dims=530, seq_length=8, hidden_size=530,
                               use_gae=True, gamma=0.99, tau=0.95), "cuda:0")
    return envs, pool, [e.reset() for e in envs], [False] * W


def run_insert(agent, W, ticks):
    envs, pool, obs, done = make(W)
    actor = BatchedActor(agent, W)
    t_env = 0.0

    def tick():
        nonlocal t_env
        acted = actor.act(obs)
        for w, env in enumerate(envs):
            command = obs[w]["command"]
            feat, action, logp, value, hidden = acted[w]
            t0 = time.perf_counter()
            obs[w], reward, done[w], info = env.step(agent.convert_action(action))
            t_env += time.perf_counter() - t0
            for h in range(2):
                mask = torch.tensor([[0.0] if info["action_done"][h] else [1.0]])
                pool.storages[w][h].insert(feat, action[h], logp[h], value[h], reward[h], mask, hidden, command)
            if done[w]:
                obs[w] = env.reset()
                actor.reset(w)
    for _ in range(WARM):
        tick()
    torch.cuda.synchronize()
    t_env = 0.0
    t0 = time.perf_counter()
    for _ in range(ticks):
        tick()
    torch.cuda.synchronize()
    total = time.perf_counter() - t0
    # bootstrap: W x get_value (train.py:76-79 as the existing loop runs it)
    for _ in range(2):
        [agent.get_value(done[w], pool.storages[w][0].get_last(), pool.storages[w][1].get_last()) for w in range(W)]
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    reps = 5
    for _ in range(reps):
        nv = torch.zeros(W, 2)
        for w in range(W):
            vs, vt = agent.get_value(done[w], pool.storages[w][0].get_last(), pool.storages[w][1].get_last())
            nv[w, 0], nv[w, 1] = float(vs.reshape(-1)[0]), float(vt.reshape(-1)[0])
    torch.cuda.synchronize()
    return total / ticks, t_env / ticks, (time.perf_counter() - t0) / reps


def run_device(agent, W, ticks):
    envs, pool, obs, done = make(W)
    actor = BatchedActor(agent, W)
    rewards, masks = np.zeros((W, 2), np.float32), np.zeros((W, 2), np.float32)
    t_env = 0.0

    def tick():
        nonlocal t_env
        slot = pool.storages[0][0].step
        actions = actor.act_into(obs, pool)
        for w, env in enumerate(envs):
            t0 = time.perf_counter()
            obs[w], reward, done[w], info = env.step(agent.convert_action(actions[w]))
            t_env += time.perf_counter() - t0
            rewards[w] = reward
            masks[w] = [0.0 if d else 1.0 for d in info["action_done"]]
            if done[w]:
                obs[w] = env.reset()
                actor.reset(w)
        pool.write_env_results(slot, rewards, masks)
    for _ in range(WARM):
        tick()
    torch.cuda.synchronize()
    t_env = 0.0
    t0 = time.perf_counter()
    for _ in range(ticks):
        tick()
    torch.cuda.synchronize()
    total = time.perf_counter() - t0
    for _ in range(2):
        actor.bootstrap_into(pool, done)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    reps = 5
    for _ in range(reps):
        actor.bootstrap_into(pool, done)
    torch.cuda.synchronize()
    return total / ticks, t_env / ticks, (time.perf_counter() - t0) / reps


def main():
    assert torch.cuda.is_available(), "this probe measures on a CUDA device"
    Ws = [int(a) for a in sys.argv[1:]] or [4, 16, 64]
    torch.set_num_threads(8)
    print(f"card: {card()}", flush=True)
    cfg = load_config()
    agent = CadreAgent(**cfg.agent_cfg, danet_state=R.danet_fixture_state(0), ppo_state=R.ppo_fixture_state(0),
                       max_encoder_batch=64)
    print("W | path | ms/tick | env.step ms/tick | rest ms/tick | bootstrap ms", flush=True)
    for W in Ws:
        for name, fn in (("act + 2W insert", run_insert), ("act_into", run_device)):
            tot, env, boot = fn(agent, W, T)
            print(f"{W} | {name} | {tot * 1e3:.2f} | {env * 1e3:.2f} | {(tot - env) * 1e3:.2f} | {boot * 1e3:.3f}",
                  flush=True)


if __name__ == "__main__":
    main()
