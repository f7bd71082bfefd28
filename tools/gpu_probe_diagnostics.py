"""Cost of the PPO update diagnostics. Times the staged update step (cadre_ppo_update on the staged table, then clip +
Adam with the device-side step) at cfg 3 (4 workers x 100 rows, T = 200) and cfg 5 (8 x 400, T = 800) with CUDA events,
diagnostics off and on in alternating rounds of 8 steps (one learn() phase) in the same process. Then, in a separate
torch.profiler pass, the device time of head_kernel and sqnorm_final_kernel alone, off and on, and the time of
cadre_rollout_stats over 128 sequences x 800 steps (CUDA events). Prints the card name and power limit of the run and
the figures; --out PATH also writes them as JSON. Usage: python tools/gpu_probe_diagnostics.py [--rounds N] [--out PATH]"""
import argparse
import json
import os
import subprocess
import sys
from types import SimpleNamespace

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from cadre_b200 import fixtures, ppo, ppo_params    # noqa: E402

DEV = "cuda:0"
STEPS = 8


def card():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                              capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
    except Exception as e:
        return f"{torch.cuda.get_device_name(0)}, power limit unknown ({e})"


def make(W, mb, T, seed):
    g = torch.Generator(device=DEV).manual_seed(seed)
    storages, advs = [], []
    for w in range(W):
        pair, apair = [], []
        for A in (33, 3):
            st = SimpleNamespace(
                obs=torch.randn(T + 1, 8, 530, device=DEV, generator=g),
                action=torch.randint(0, A, (T + 1, 1), device=DEV, generator=g),
                value_preds=torch.randn(T + 1, 1, device=DEV, generator=g),
                returns=torch.randn(T + 1, 1, device=DEV, generator=g),
                action_log_probs=torch.rand(T + 1, 1, device=DEV, generator=g) * -2.5 - 0.5,
                hn=torch.zeros(T + 1, 530, device=DEV), cn=torch.zeros(T + 1, 530, device=DEV),
                command=torch.randint(0, 4, (T + 1, 1), device=DEV, generator=g, dtype=torch.int32))
            pair.append(st)
            apair.append(torch.randn(T, 1, device=DEV, generator=g))
        storages.append(tuple(pair))
        advs.append(tuple(apair))
    rs = np.random.RandomState(seed)
    idx = np.stack([np.stack([np.stack([rs.permutation(T)[:mb] for _ in range(2)]) for _ in range(W)])
                    for _ in range(STEPS)]).astype(np.int32)
    flat = ppo_params.pack_state(fixtures.ppo_fixture_state(0), DEV)
    eng = ppo.PpoEngine(W, mb, device=DEV)
    bufs = SimpleNamespace(params=flat, grads=torch.zeros_like(flat), m=torch.zeros_like(flat), v=torch.zeros_like(flat),
                           losses=torch.zeros(W, 2, 3, device=DEV), diag=torch.zeros(STEPS, W, 2, 4, device=DEV),
                           norms=torch.zeros(STEPS, 16, device=DEV))
    return eng, storages, advs, idx, bufs


def phase(eng, storages, advs, idx, b, diag, events=None):
    """One learn() phase of STEPS staged steps; events: list of (start, mid, end) per step to record into."""
    eng.stage(storages, advs, idx, 1)
    for k in range(STEPS):
        if diag:
            eng.set_diagnostics(b.diag[k], b.norms[k])
        if events is not None:
            events[k][0].record()
        eng.update_staged(b.params, b.grads, b.losses)
        if events is not None:
            events[k][1].record()
        eng.adam_step(b.params, b.grads, b.m, b.v, 0)
        if events is not None:
            events[k][2].record()
        if diag:
            eng.set_diagnostics(None, None)


def time_config(name, W, mb, T, rounds):
    eng, storages, advs, idx, b = make(W, mb, T, 7)
    for diag in (False, True, False, True):       # warm-up
        phase(eng, storages, advs, idx, b, diag)
    torch.cuda.synchronize()
    res = {False: ([], []), True: ([], [])}
    for r in range(rounds):
        for diag in ((False, True) if r % 2 == 0 else (True, False)):
            ev = [[torch.cuda.Event(enable_timing=True) for _ in range(3)] for _ in range(STEPS)]
            phase(eng, storages, advs, idx, b, diag, ev)
            torch.cuda.synchronize()
            res[diag][0].append(np.mean([e[0].elapsed_time(e[1]) for e in ev]))
            res[diag][1].append(np.mean([e[1].elapsed_time(e[2]) for e in ev]))
    eng.check()
    out = {}
    for diag, (fb, ad) in res.items():
        key = "on" if diag else "off"
        out[key] = dict(fwd_bwd_ms=float(np.median(fb)), fwd_bwd_ms_min=float(np.min(fb)),
                        fwd_bwd_ms_max=float(np.max(fb)), clip_adam_ms=float(np.median(ad)),
                        clip_adam_ms_min=float(np.min(ad)), clip_adam_ms_max=float(np.max(ad)))
        print(f"{name} diagnostics {key}: fwd+bwd {out[key]['fwd_bwd_ms']:.4f} ms (rounds {np.min(fb):.4f} .. "
              f"{np.max(fb):.4f}), clip+Adam {out[key]['clip_adam_ms']:.4f} ms ({np.min(ad):.4f} .. {np.max(ad):.4f})")
    return out, (eng, storages, advs, idx, b)


def profile_kernels(name, setup, reps=10):
    """device time per launch of head_kernel and sqnorm_final_kernel, diagnostics off and on (torch.profiler)."""
    from torch.profiler import ProfilerActivity, profile
    eng, storages, advs, idx, b = setup
    out = {}
    for diag in (False, True):
        phase(eng, storages, advs, idx, b, diag)
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(reps):
                phase(eng, storages, advs, idx, b, diag)
            torch.cuda.synchronize()
        key = "on" if diag else "off"
        for evt in prof.key_averages():
            for kname in ("head_kernel", "sqnorm_final_kernel"):
                if kname in evt.key:
                    total = getattr(evt, "device_time_total", None) or getattr(evt, "cuda_time_total", 0.0)
                    out[f"{kname}_{key}_us"] = total / max(1, evt.count)
    print(f"{name} kernels (profiler, us per launch): " + ", ".join(f"{k} {v:.2f}" for k, v in sorted(out.items())))
    return out


def time_rollout_stats(E=128, T=800, reps=500):
    g = torch.Generator(device=DEV).manual_seed(1)
    ret = torch.randn(E, T + 1, device=DEV, generator=g)
    val = torch.randn(E, T + 1, device=DEV, generator=g)
    out = torch.empty(E, 6, device=DEV)
    for _ in range(20):
        ppo.rollout_stats(ret, val, out)
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        ppo.rollout_stats(ret, val, out)
    b.record()
    torch.cuda.synchronize()
    us = a.elapsed_time(b) * 1000.0 / reps
    print(f"rollout_stats {E} x {T}: {us:.2f} us per launch (back-to-back, {reps} launches)")
    return us


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=30, help="alternating off / on rounds of one phase each")
    ap.add_argument("--out", default=None, help="JSON file for the results")
    args = ap.parse_args()
    rounds = args.rounds
    result = {"card": card(), "rounds": rounds, "steps_per_round": STEPS}
    print(result["card"])
    for name, (W, mb, T) in (("cfg3", (4, 100, 200)), ("cfg5", (8, 400, 800))):
        result[name], setup = time_config(name, W, mb, T, rounds)
        result[name]["kernels"] = profile_kernels(name, setup)
    result["rollout_stats_128x800_us"] = time_rollout_stats()
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(result, f, indent=1)


if __name__ == "__main__":
    main()
