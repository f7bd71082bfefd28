"""Cost of training checkpoints. Runs one episode of train(device_rollout=True, checkpoint_dir=...) at cfg 3 (4 workers,
T = 200) and at a cfg-5-sized rank (8 workers, T = 800), then resumes from the checkpoint it wrote. Reports the save
time (from the end of the episode's learn(), with the device synchronised, until every file and the COMPLETE marker are
durable), the load time (reading the files, the config and replica checks, and copying the state into the learner,
pool, actor and environments) and the file sizes. Prints the card name and power limit of the run; --out PATH also
writes the figures as JSON. Usage: python tools/gpu_probe_checkpoint.py [--dir DIR] [--out PATH]"""
import argparse
import json
import os
import sys
import tempfile
import time

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from gpu_probe_diagnostics import card    # noqa: E402

CONFIGS = {"cfg3": (4, 200), "cfg5_rank": (8, 800)}


def timed(fn, into):
    def wrapper(*a, **k):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        r = fn(*a, **k)
        torch.cuda.synchronize()
        into.append(time.perf_counter() - t0)
        return r
    return wrapper


def probe(name, W, T, root):
    from cadre_b200 import checkpoint as C
    from cadre_b200 import train as TR
    from cadre_b200.config import load_config
    from oracle import restate as R
    cfg = load_config()
    cfg.rollout_cfg.num_steps = T
    cfg.train_cfg.log_interval = 1000
    saves, loads = [], []
    real_save, real_restore = C.save, TR._restore
    C.save, TR._restore = timed(real_save, saves), timed(real_restore, loads)
    try:
        run = os.path.join(root, name)
        kw = dict(ppo_state=R.ppo_fixture_state(0), workers=W, device_rollout=True, log=lambda *a: None)
        TR.train(0, cfg.train_cfg, cfg.agent_cfg, cfg.env_cfg, cfg.rollout_cfg, R.danet_fixture_state(0), max_episode=1,
                 checkpoint_dir=run, **kw)
        TR.train(0, cfg.train_cfg, cfg.agent_cfg, cfg.env_cfg, cfg.rollout_cfg, R.danet_fixture_state(0), max_episode=1,
                 checkpoint_dir=run, resume="latest", **kw)
    finally:
        C.save, TR._restore = real_save, real_restore
    ep = C.latest(run)
    mb = lambda f: os.path.getsize(os.path.join(ep, f)) / 1e6     # noqa: E731
    return dict(config=name, workers=W, T=T, save_s=saves[0], load_s=loads[0], learner_pt_MB=mb(C.LEARNER_FILE),
                rank_0_pt_MB=mb(C.rank_file(0)), snapshot_MB=os.path.getsize(
                    os.path.join(run, "models", "ppo_model_0.pt")) / 1e6)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--dir", default=None, help="where the checkpoints go (default: a temporary directory)")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    res = dict(card=card(), runs=[])
    with tempfile.TemporaryDirectory() as tmp:
        root = args.dir or tmp
        for name, (W, T) in CONFIGS.items():
            r = probe(name, W, T, root)
            print(json.dumps(r), flush=True)
            res["runs"].append(r)
    print("card:", res["card"])
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
