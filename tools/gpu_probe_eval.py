"""Ensemble evaluation cost per environment tick: the reference-shaped `eval.evaluate` loop (K CadreAgents, each
re-encoding the full 8-frame window and drawing on the host, one environment) against `eval.DeviceEnsemble` (one frame
cache, E environments per tick, K routed forwards and one draw + average kernel) at E = 1, 16, 64 and K = 1, 3, 5 in
sampled mode. SyntheticEnv with done_prob = 0 (no reset inside the timed window); host clock around `--ticks` ticks
after `--warmup` ticks, each tick ending in a device synchronise. env.step is the host time inside SyntheticEnv.step,
"rest" everything else of the tick. Prints the card name and power limit of the run; --out PATH also writes JSON.
Usage: python tools/gpu_probe_eval.py [--ticks N] [--warmup N] [--out PATH]"""
import argparse
import json
import os
import sys
import time

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from gpu_probe_diagnostics import card    # noqa: E402


def timed_envs(E):
    from cadre_b200.synthetic_env import SyntheticEnv
    envs = [SyntheticEnv(dict(rank=e, seq_length=8, done_prob=0.0)) for e in range(E)]
    spent = [0.0]
    for env in envs:
        step = env.step

        def timed_step(control, step=step):
            t0 = time.perf_counter()
            r = step(control)
            spent[0] += time.perf_counter() - t0
            return r
        env.step = timed_step
    return envs, spent


def window(tick_fn, warmup, ticks, spent):
    for _ in range(warmup):
        tick_fn()
    torch.cuda.synchronize()
    spent[0] = 0.0
    t0 = time.perf_counter()
    for _ in range(ticks):
        tick_fn()
    torch.cuda.synchronize()
    total = (time.perf_counter() - t0) / ticks
    env = spent[0] / ticks
    return total * 1e3, env * 1e3


def probe_reference(cfg, R, K, warmup, ticks):
    from cadre_b200.agent import CadreAgent
    agents = [CadreAgent(**cfg.agent_cfg, danet_state=R.danet_fixture_state(0), ppo_state=R.ppo_fixture_state(k),
                         max_encoder_batch=8) for k in range(K)]
    (env,), spent = timed_envs(1)
    obs = [env.reset()]

    def tick():
        actions = [agent.act(obs[0])[1] for agent in agents]
        obs[0] = env.step(agents[-1].avg_action(actions))[0]
    return window(tick, warmup, ticks, spent)


def probe_device(agent, params, E, K, warmup, ticks):
    from cadre_b200.eval import DeviceEnsemble
    envs, spent = timed_envs(E)
    obs = [env.reset() for env in envs]
    ens = DeviceEnsemble(agent, params[:K], E)

    def tick():
        controls = ens.act(obs)
        for e, env in enumerate(envs):
            obs[e] = env.step([float(v) for v in controls[e]])[0]
    return window(tick, warmup, ticks, spent)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--ticks", type=int, default=40)
    ap.add_argument("--warmup", type=int, default=6)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("gpu_probe_eval needs a CUDA device")
    from cadre_b200.agent import CadreAgent
    from cadre_b200.config import load_config
    from cadre_b200.models import FlatParams
    from oracle import restate as R
    cfg = load_config()
    gpu = card()
    print(f"card: {gpu}", flush=True)
    res = {"card": gpu, "ticks": args.ticks, "warmup": args.warmup, "reference": {}, "device": {}}
    for K in (1, 3, 5):
        ms, env = probe_reference(cfg, R, K, args.warmup, args.ticks)
        res["reference"][K] = {"ms_per_tick": ms, "env_ms": env}
        print(f"evaluate(): K={K} E=1: {ms:.2f} ms/tick (env.step {env:.2f} + rest {ms - env:.2f})", flush=True)
    agent = CadreAgent(**cfg.agent_cfg, danet_state=R.danet_fixture_state(0), ppo_state=R.ppo_fixture_state(0),
                       max_encoder_batch=64)
    params = [FlatParams(agent.device, R.ppo_fixture_state(k)).params for k in range(5)]
    for E in (1, 16, 64):
        for K in (1, 3, 5):
            ms, env = probe_device(agent, params, E, K, args.warmup, args.ticks)
            res["device"][f"E{E}_K{K}"] = {"E": E, "K": K, "ms_per_tick": ms, "env_ms": env}
            print(f"DeviceEnsemble: K={K} E={E}: {ms:.2f} ms/tick (env.step {env:.2f} + rest {ms - env:.2f}; "
                  f"rest per env {(ms - env) / E:.3f} ms)", flush=True)
    print("\n| K | evaluate(), E = 1 | DeviceEnsemble E = 1 | E = 16 | E = 64 |")
    print("|---|---|---|---|---|")
    for K in (1, 3, 5):
        r = res["reference"][K]
        cells = [f"{r['ms_per_tick']:.2f} ({r['env_ms']:.2f} + {r['ms_per_tick'] - r['env_ms']:.2f})"]
        for E in (1, 16, 64):
            d = res["device"][f"E{E}_K{K}"]
            cells.append(f"{d['ms_per_tick']:.2f} ({d['env_ms']:.2f} + {d['ms_per_tick'] - d['env_ms']:.2f})")
        print(f"| {K} | " + " | ".join(cells) + " |")
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
