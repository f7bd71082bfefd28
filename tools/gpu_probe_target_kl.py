"""Cost of target-KL early stopping. Times the staged update step (cadre_ppo_update on the staged table, the KL gate,
then clip + Adam with the device-side step) at cfg 3 (4 workers x 100 rows, T = 200) and cfg 5 (8 x 400, T = 800) with
CUDA events per step, three arms alternating in rounds of one 8-step phase in the same process: target_kl off, on but
never triggered (1e9), and on with a threshold the first step exceeds (1e-12 against the random stored log-probs), whose
steps 1..7 are skipped steps. Prints the card name and power limit of the run and the figures; --out PATH also writes
them as JSON. Usage: python tools/gpu_probe_target_kl.py [--rounds N] [--out PATH]"""
import argparse
import json
import os
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from gpu_probe_diagnostics import STEPS, card, make    # noqa: E402

ARMS = {"off": None, "never": 1e9, "stopped": 1e-12}


def phase(eng, storages, advs, idx, b, kl_sum, arm, events=None):
    """One phase of STEPS staged steps; events: per step (start, after the update, after the gate, after clip + Adam)."""
    tkl = ARMS[arm]
    eng.set_target_kl(tkl, eng.workers, kl_sum)
    if tkl is not None:
        eng.kl_begin()
    eng.stage(storages, advs, idx, 1)
    for k in range(STEPS):
        if events is not None:
            events[k][0].record()
        eng.update_staged(b.params, b.grads, b.losses)
        if events is not None:
            events[k][1].record()
        if tkl is not None:
            eng.kl_gate()
        if events is not None:
            events[k][2].record()
        eng.adam_step(b.params, b.grads, b.m, b.v, 0)
        if events is not None:
            events[k][3].record()


def time_config(name, W, mb, T, rounds):
    eng, storages, advs, idx, b = make(W, mb, T, 7)
    kl_sum = torch.zeros(4, device=b.params.device)
    keep = b.params.clone()
    for arm in list(ARMS) * 2:      # warm-up
        phase(eng, storages, advs, idx, b, kl_sum, arm)
    torch.cuda.synchronize()
    res = {arm: dict(fwd_bwd=[], gate=[], clip_adam=[], skipped_fwd_bwd=[], skipped_clip_adam=[]) for arm in ARMS}
    for r in range(rounds):
        order = list(ARMS) if r % 2 == 0 else list(ARMS)[::-1]
        for arm in order:
            b.params.copy_(keep)     # every arm starts from the same parameters (and so the same routing and work)
            ev = [[torch.cuda.Event(enable_timing=True) for _ in range(4)] for _ in range(STEPS)]
            phase(eng, storages, advs, idx, b, kl_sum, arm, ev)
            torch.cuda.synchronize()
            fb = [e[0].elapsed_time(e[1]) for e in ev]
            g = [e[1].elapsed_time(e[2]) for e in ev]
            ad = [e[2].elapsed_time(e[3]) for e in ev]
            if arm == "stopped":
                st = eng.early_stop()
                assert st["stopped_at"] == 0 and st["applied"] == 0, st
                res[arm]["skipped_fwd_bwd"].append(np.mean(fb[1:]))
                res[arm]["skipped_clip_adam"].append(np.mean(ad[1:]))
                fb, g, ad = fb[:1], g[:1], ad[:1]
            res[arm]["fwd_bwd"].append(np.mean(fb))
            res[arm]["gate"].append(np.mean(g))
            res[arm]["clip_adam"].append(np.mean(ad))
    eng.check()
    out = {}
    for arm, d in res.items():
        out[arm] = {}
        for key, vals in d.items():
            if vals:
                out[arm][key + "_ms"] = float(np.median(vals))
                out[arm][key + "_ms_min"] = float(np.min(vals))
                out[arm][key + "_ms_max"] = float(np.max(vals))
        print(f"{name} target_kl {arm}: " + ", ".join(
            f"{k[:-3]} {v:.4f} ms ({out[arm][k + '_min']:.4f} .. {out[arm][k + '_max']:.4f})"
            for k, v in out[arm].items() if k.endswith("_ms")))
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=30, help="alternating rounds of one phase per arm")
    ap.add_argument("--out", default=None, help="JSON file for the results")
    args = ap.parse_args()
    result = {"card": card(), "rounds": args.rounds, "steps_per_round": STEPS,
              "arms": {k: v for k, v in ARMS.items()}, "two_gpu_nccl_kl_exchange": "not measured"}
    print(result["card"])
    for name, (W, mb, T) in (("cfg3", (4, 100, 200)), ("cfg5", (8, 400, 800))):
        result[name] = time_config(name, W, mb, T, args.rounds)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(result, f, indent=1)


if __name__ == "__main__":
    main()
