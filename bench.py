"""bench.py — CADRE learner hot path on B200: encoder forward + GAE + PPO update (+ gradient all-reduce + Adam).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl cadre|reference] [--config cfg3|cfg5]
                    [--dump-outputs DIR]
    torchrun --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...        (N > 1)

One STEP = one learner iteration on every rank (weak scaling: per-GPU work is fixed):
  cfg3 (default; BASELINE config 3, and config 4 for N > 1): 4 logical workers x T=200 env ticks x 8 stacked frames ->
       encoder forward over 6400 camera frames (uint8 rgb + route map + measurements), features written into the 8
       RolloutStorages, GAE + advantage normalisation, then ppo_epoch=4 x 2 minibatches of (routed LSTM / actor-critic
       forward + backward over 400 rows x 2 heads, gradient all-reduce for N > 1 - the library's in-switch kernel from 4
       ranks on, NCCL between 2 -, per-module clip + Adam).
  cfg5 (BASELINE config 5 when run with --gpus 8): 8 envs per GPU, T=800, minibatches of 400 rows per env
       (51 200 window frames and 8 x 3200-row update steps per GPU and step).
value = window frames/s with inputs resident in HBM; EVERY window frame is encoded (device-timed, max over ranks).
e2e   = the same metric through the package's ingest API (cadre_b200.ingest.RolloutIngest) from pinned HOST frames,
        H2D copies inside the timed region, losses read back D2H. The API ships and encodes each DISTINCT frame once
        (the 8-frame window slides by one frame per tick) and assembles the windows on the device; `e2e_full_windows`
        repeats the measurement shipping + encoding every window frame like round 1 did.
--impl reference times the reference's own CPU implementation (oracle port: the reference is pure Python and
/root/reference is not on the GPU box) with all host threads: each step is a REAL, fully executed 1/8 slice of the cfg3
step (100 ticks of one worker), nothing is extrapolated.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True     # a benchmark run leaves the tree as build() left it (it may be read-only)

DUMP_MAX_ELEMS = 1 << 22           # --dump-outputs: a larger output is written as a fixed, seeded sample of this size
DUMP_MAX_BYTES = 64 << 20

SEQ, MB_NUM, PPO_EPOCH = 8, 2, 4
CONFIGS = {
    "cfg3": dict(workers=4, T=200),
    "cfg5": dict(workers=8, T=800),
}
ENC_CHUNK = int(os.environ.get("CADRE_BENCH_CHUNK", "640"))   # frames per encoder call
METRIC = "encoder+PPO-update frames/sec"
PPO_FLOP_PER_ROW = 217.8e6       # routed forward + backward, SURVEY.md §8d


def workload_name(cfg):
    W, T = CONFIGS[cfg]["workers"], CONFIGS[cfg]["T"]
    return (f"{cfg} learner iteration per GPU: {W} workers x T={T} x 8 frames encoder fwd ({W * T * SEQ} u8 frames "
            f"144x256) + GAE + {PPO_EPOCH} epochs x {MB_NUM} minibatches x {W * T // MB_NUM} rows PPO update "
            "(fwd+bwd, allreduce, clip+Adam)")


# ---------------------------------------------------------------------------------------------- helpers
def encoder_flops_per_frame():
    """name -> FLOPs/frame of each encoder launch as EXECUTED here (SURVEY.md §8d counts 3.0875 GFLOP/frame for
    the unfused reference graph; the folded fc1 does less work)."""
    f = {}
    f["stem+pool"] = 2 * 72 * 128 * 64 * 196
    H, W, C = 36, 64, 64
    for li, planes in enumerate((64, 128, 256, 512), start=1):
        for bi in range(2):
            s = 2 if (li > 1 and bi == 0) else 1
            Ho = (H + 2 - 3) // s + 1
            Wo = (W + 2 - 3) // s + 1
            f[f"layer{li}.{bi}.conv1"] = 2 * Ho * Wo * planes * C * 9
            f[f"layer{li}.{bi}.conv2"] = 2 * Ho * Wo * planes * planes * 9
            if s == 2:
                f[f"layer{li}.0.downsample"] = 2 * Ho * Wo * planes * C
                f[f"layer{li}.0.conv2+shortcut"] = f[f"layer{li}.0.conv2"] + f[f"layer{li}.0.downsample"]
            H, W, C = Ho, Wo, planes
    f["conv5a|conv5c"] = 2 * 40 * 256 * 512 * 9
    f["conv51"] = f["conv52+sum"] = 2 * 40 * 128 * 128 * 9
    f["fc1(folded)"] = 2 * 5120 * 3072
    f["fc2"] = 2 * 6 * 512 * 256
    return f


def sample_clocks_start():
    path = tempfile.mktemp(prefix="cadre_clocks_", suffix=".csv")
    q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")
    try:
        p = subprocess.Popen(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", "100",
                              "-i", os.environ.get("LOCAL_RANK", "0")], stdout=open(path, "w"),
                             stderr=subprocess.DEVNULL)
    except Exception:
        return None, path
    return p, path


def sample_clocks_stop(p, path):
    out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": []}
    if p is None:
        return out
    p.terminate()
    try:
        p.wait(timeout=5)
    except Exception:
        p.kill()
    sm, mx, reasons = [], [], set()
    try:
        for line in open(path):
            c = [x.strip() for x in line.split(",")]
            if len(c) < 9:
                continue
            try:
                sm.append(float(c[1]))
                mx.append(float(c[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), c[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        os.unlink(path)
    except Exception:
        pass
    if sm:
        busy = sorted(sm)[len(sm) // 2:]          # the sampler also sees start-up and warm-up: keep the loaded half
        out["sm_mhz"] = float(np.median(busy))
        out["sm_max_mhz"] = float(max(mx))
        out["reasons"] = sorted(reasons)
    return out


def ncu_traffic():
    """DRAM bytes (read + write) of the tcgen05 launches of one encoder forward at batch 640, from the committed
    `ncu --set full` capture (profiles/*_traffic.json); None if the summary is missing."""
    for name in ("r2_traffic.json", "r1_traffic.json"):
        try:
            return json.load(open(os.path.join(ROOT, "profiles", name)))["tcgen05_family_dram_bytes_per_forward_b640"]
        except Exception:
            continue
    return None


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return d.get("bf16_tflops_sustained", 1417.3), d.get("hbm_gbs", 6453.1), "measured"
    return 1400.0, 6650.0, "fallback"


def bind_to_gpu_numa_node(local_rank):
    """Pin this rank's host threads to the CPUs NVML reports as local to its GPU BEFORE the pinned staging buffers
    are allocated (first-touch puts their pages on that NUMA node)."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(local_rank)
        words = (os.cpu_count() + 63) // 64
        mask = pynvml.nvmlDeviceGetCpuAffinity(h, words)
        cpus = [64 * w + b for w in range(words) for b in range(64) if (mask[w] >> b) & 1]
        orig = os.sched_getaffinity(0)
        cpus = [c for c in cpus if c in orig]
        if cpus:
            os.sched_setaffinity(0, cpus)
            return len(cpus), orig
    except Exception:
        pass
    return None, None


def dump_outputs(out_dir, arrays):
    """Write each array as <out_dir>/<name>.npy in float32. An array of more than DUMP_MAX_ELEMS elements is written as
    the elements at DUMP_MAX_ELEMS flat positions drawn without replacement from a generator seeded with 0, in
    ascending order: the same positions for the same shape, so that two runs or two builds compare element for
    element."""
    os.makedirs(out_dir, exist_ok=True)
    total = 0
    for name, t in arrays.items():
        flat = t.detach().reshape(-1)
        if flat.numel() > DUMP_MAX_ELEMS:
            pos = np.sort(np.random.default_rng(0).choice(flat.numel(), DUMP_MAX_ELEMS, replace=False))
            a = flat[torch.from_numpy(pos).to(flat.device)].float().cpu().numpy()
        else:
            a = t.detach().float().cpu().numpy()
        np.save(os.path.join(out_dir, name + ".npy"), a)
        total += a.nbytes
    assert total <= DUMP_MAX_BYTES, f"--dump-outputs wrote {total} bytes"


# ---------------------------------------------------------------------------------------------- reference arm
class CpuReferenceSlice:
    """A fully executed slice of the learner step on the CPU oracle (the reference's PyTorch code path restated,
    oracle/restate.py): `ticks` env ticks of ONE worker, with everything the reference does for them:
      ticks x get_latent_feature on the 8-frame window (agent.py:97-112), GAE + advantage normalisation of one storage
      pair (storage.py:68-76, train.py:82-88), ticks * ppo_epoch rows of update_policy in minibatches of `mb` rows
      (agent.py:166-237, dense 4-command formulation) and the chief's clip + Adam steps that fall into the slice
      (chief.py:13-21). Nothing is extrapolated: run() returns the wall time of exactly this work."""

    def __init__(self, cfg, ticks, threads):
        from oracle import restate as R
        self.R = R
        torch.set_num_threads(threads)
        W, T = CONFIGS[cfg]["workers"], CONFIGS[cfg]["T"]
        self.ticks, self.mb = ticks, T // MB_NUM
        self.update_calls = max(1, ticks * PPO_EPOCH // self.mb)
        self.chief_steps = max(1, round(PPO_EPOCH * MB_NUM * ticks / (W * T)))
        rs = np.random.RandomState(0)
        self.sd = R.danet_fixture_state(0)
        psd = R.ppo_fixture_state(0)
        self.params = {m: {n: t.clone().requires_grad_(True) for n, t in d.items()} for m, d in psd.items()}
        self.adam = {m: {n: {"exp_avg": torch.zeros_like(t), "exp_avg_sq": torch.zeros_like(t)} for n, t in d.items()}
                     for m, d in psd.items()}
        self.tick_data = [R.synthetic_tick(rs) for _ in range(8)]          # 8 distinct windows, cycled
        self.storages = [R.synthetic_storage(rs, T=T, actions=a) for a in (R.STEER_ACTIONS, R.THROTTLE_ACTIONS)]
        self.idx = [list(rs.permutation(T)[:self.mb]) for _ in range(2)]
        self.step = 0
        self.frames = ticks * SEQ
        self.description = (f"each step = {ticks} ticks of one {cfg} worker, fully executed on the CPU: {ticks} x "
                            f"get_latent_feature(8 frames) = {self.frames} frames, GAE + adv-norm of one storage pair "
                            f"(T={T}), {self.update_calls} x update_policy at mb={self.mb} rows x 2 heads (dense "
                            f"4-command compute), {self.chief_steps} chief clip+Adam step(s); = 1/{W * T // ticks} of "
                            "the per-GPU step")

    def run(self):
        R = self.R
        t0 = time.perf_counter()
        with torch.no_grad():
            for i in range(self.ticks):
                tk = self.tick_data[i % len(self.tick_data)]
                R.agent_latent_feature(tk["rgb"], tk["route_fig"].copy(), tk["measurements"], self.sd)
        t_enc = time.perf_counter() - t0
        advs = []
        for st in self.storages:
            ret, vp = R.compute_returns(st["rewards"], st["value_preds"], st["masks"], torch.tensor([[0.1]]))
            st["returns"] = ret
            advs.append(R.normalized_advantages(ret, vp))
        t1 = time.perf_counter()
        for _ in range(self.update_calls):
            samples = [R.gather_minibatch(st, adv, ix) for st, adv, ix in zip(self.storages, advs, self.idx)]
            R.update_policy(samples[0], samples[1], self.params)
        t_upd = time.perf_counter() - t1
        grads = {m: {n: p.grad for n, p in d.items()} for m, d in self.params.items()}
        for _ in range(self.chief_steps):
            self.step += 1
            R.chief_step(self.params, grads, self.adam, step=self.step)
        dt = time.perf_counter() - t0
        return dt, {"encoder_s": t_enc, "update_policy_s": t_upd, "gae_chief_s": dt - t_enc - t_upd}


def run_reference(args):
    rank = int(os.environ.get("RANK", 0))
    if rank != 0:
        return
    threads = os.cpu_count() or 1
    sl = CpuReferenceSlice(args.config, int(os.environ.get("CADRE_REF_TICKS", "100")), threads)
    times, detail = [], None
    for i in range(args.warmup + args.steps):
        dt, detail = sl.run()
        if i >= args.warmup:
            times.append(dt)
    t_step = float(np.mean(times))
    value = sl.frames / t_step
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": "frames/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * t_step,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": workload_name(args.config)},
        "cpu_baseline": {"value": value, "unit": "frames/s", "cores": threads, "kind": "port",
                         "sample": sl.description, "frames_per_step": sl.frames,
                         **{k: round(v, 4) for k, v in detail.items()}},
        "e2e": {"value": value, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


# ---------------------------------------------------------------------------------------------- cadre arm
def run_cadre(args):
    rank = int(os.environ.get("RANK", 0))
    local = int(os.environ.get("LOCAL_RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the product has no CPU path (use --impl reference for the "
                         "CPU baseline)")
    WORKERS, T = CONFIGS[args.config]["workers"], CONFIGS[args.config]["T"]
    FRAMES_PER_STEP = WORKERS * T * SEQ
    K = T + SEQ - 1
    torch.cuda.set_device(local)
    dev = torch.device(f"cuda:{local}")

    # ---- CPU baseline FIRST (N = 1 only): before any process group exists and before the affinity is narrowed, so that
    # it really has every host core (round 1 measured it while the other ranks were spinning in a barrier)
    cpu_baseline = None
    if world == 1 and not args.no_cpu_baseline:
        threads = os.cpu_count() or 1
        sl = CpuReferenceSlice(args.config, int(os.environ.get("CADRE_CPU_BASELINE_TICKS", "50")), threads)
        sl.run()                                   # warm-up (thread pools, allocator)
        dt, detail = sl.run()
        cpu_baseline = {"value": sl.frames / dt, "unit": "frames/s", "cores": threads, "kind": "port",
                        "sample": sl.description, "seconds": round(dt, 3),
                        **{k: round(v, 4) for k, v in detail.items()}}

    numa, full_affinity = bind_to_gpu_numa_node(local)
    dist = torch.distributed
    if world > 1:
        # measured on 8 x B200 (tools/gpu_probe_allreduce.py): the 78 MB / 36 MB gradient all-reduces take 0.27 / 0.15 ms
        # with the ring algorithm against 0.32 / 0.17 ms with NCCL's default choice (NVLS) for these sizes
        os.environ.setdefault("NCCL_ALGO", "Ring")
        dist.init_process_group("nccl", device_id=dev)
    import __graft_entry__
    if rank == 0:
        __graft_entry__.build()
    if world > 1:
        dist.barrier()
    from cadre_b200 import fixtures as FX   # seeded synthetic weights (no checkpoint on the box)
    from cadre_b200 import ppo as PPO
    from cadre_b200 import ppo_params
    from cadre_b200.ingest import RolloutIngest
    from cadre_b200.learner import Learner, RolloutPool

    ingest = RolloutIngest(FX.danet_fixture_state(0), dev, WORKERS, T, SEQ, 530, max_chunk=ENC_CHUNK,
                           streams=max(1, int(os.environ.get("CADRE_ENC_STREAMS", "2"))))
    enc = ingest.encoders[0]
    mb = T // MB_NUM
    learner = Learner(WORKERS, mb, FX.ppo_fixture_state(0), dev, seeds=[rank * WORKERS + w for w in range(WORKERS)],
                      process_group=None)
    pool = RolloutPool(WORKERS, dict(num_steps=T, mini_batch_num=MB_NUM, feature_dims=530, seq_length=SEQ,
                                     use_gae=True, gamma=0.99, tau=0.95), dev)
    # synthetic rollout (SURVEY.md §8d), seeded per rank: K = T + 7 distinct frames per worker; tick t sees frames t..t+7
    g = torch.Generator(device=dev)
    g.manual_seed(1234 + rank)
    rgb_u = torch.randint(0, 256, (WORKERS, K, 144, 256, 3), device=dev, dtype=torch.uint8, generator=g)
    route_u = (torch.rand(WORKERS, K, 256, 144, device=dev, generator=g) < 0.1).to(torch.uint8) * 255
    meas_u = torch.rand(WORKERS, K, 3, device=dev, dtype=torch.float64, generator=g)
    win = (torch.arange(T, device=dev).view(T, 1) + torch.arange(SEQ, device=dev).view(1, SEQ)).flatten()
    # every tick's full window, materialised like the env wrapper hands it out (7/8 of these frames are repeats)
    rgb_w = rgb_u[:, win].view(WORKERS, T, SEQ, 144, 256, 3)
    route_w = route_u[:, win].view(WORKERS, T, SEQ, 256, 144)
    meas_w = meas_u[:, win].view(WORKERS, T, SEQ, 3)
    b = pool.batched
    b["rewards"].copy_(torch.rand(b["rewards"].shape, device=dev, generator=g))
    b["masks"].copy_((torch.rand(b["masks"].shape, device=dev, generator=g) >= 0.02).float())
    b["command"].copy_(torch.randint(0, 4, b["command"].shape, device=dev, generator=g, dtype=torch.int32))
    b["action_log_probs"].copy_(-0.5 - 2.5 * torch.rand(b["action_log_probs"].shape, device=dev, generator=g))
    b["value_preds"].copy_(torch.randn(b["value_preds"].shape, device=dev, generator=g))
    for w in range(WORKERS):
        b["action"][2 * w].copy_(torch.randint(0, 33, (T + 1, 1), device=dev, generator=g))
        b["action"][2 * w + 1].copy_(torch.randint(0, 3, (T + 1, 1), device=dev, generator=g))
    next_values = torch.zeros(WORKERS, 2, device=dev)

    def step_resident():
        ingest.encode(rgb_w, route_w, meas_w, b["obs"], unique=False)     # all window frames, inputs in HBM
        pool.compute_returns(next_values)
        return learner.learn(pool, PPO_EPOCH)

    # host-resident inputs (pinned)
    def pinned(t):
        return torch.empty(t.shape, dtype=t.dtype, pin_memory=True).copy_(t)
    rgb_uh, route_uh, meas_uh = pinned(rgb_u), pinned(route_u), pinned(meas_u)
    losses_h = torch.empty(WORKERS, 2, 3, pin_memory=True)
    d2h_bytes = losses_h.numel() * 4

    # RolloutIngest.prefetch (the next rollout's frames cross PCIe under the update phase) is OFF here: measured, the
    # in-step staging already hides the copy behind the encoder and the DMA under the update phase costs ~0.8 ms per step
    # (1 x B200: 9.4 ms without / 10.2 ms with; 4 x B200: 11.2 / 12.1 ms). CADRE_PREFETCH=1 switches it on.
    prefetch = os.environ.get("CADRE_PREFETCH", "0") == "1"

    def step_e2e():
        ingest.encode(rgb_uh, route_uh, meas_uh, b["obs"], unique=True)   # distinct frames: H2D + encode once each
        if prefetch:     # the NEXT rollout's frames cross PCIe under this rollout's update phase (one copy per step)
            ingest.prefetch(rgb_uh, route_uh, meas_uh)
        pool.compute_returns(next_values)
        learner.learn(pool, PPO_EPOCH)
        losses_h.copy_(learner.losses, non_blocking=True)

    full_windows = args.config == "cfg3" and not args.no_full_windows
    if full_windows:
        rgb_wh, route_wh, meas_wh = pinned(rgb_w), pinned(route_w), pinned(meas_w)

        def step_e2e_full():
            ingest.encode(rgb_wh, route_wh, meas_wh, b["obs"], unique=False)
            pool.compute_returns(next_values)
            learner.learn(pool, PPO_EPOCH)
            losses_h.copy_(learner.losses, non_blocking=True)

    def timed(fn, steps, warmup, sample=False):
        proc = path = None
        if sample:      # nvidia-smi needs a few hundred ms to start: launch it before the warm-up steps
            proc, path = sample_clocks_start()
        for _ in range(warmup):
            fn()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        clocks = sample_clocks_stop(proc, path) if sample else None
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return ms.item() / steps, clocks

    if world > 1:
        learner.world = world   # all-reduce inside update_step
    if args.profile_step:
        # for `ncu --profile-from-start off`: exactly ONE resident step between cudaProfilerStart / Stop, then exit
        for _ in range(max(1, args.warmup)):
            step_resident()
        torch.cuda.synchronize()
        torch.cuda.profiler.start()
        step_resident()
        torch.cuda.synchronize()
        torch.cuda.profiler.stop()
        return
    ms_step, clocks = timed(step_resident, args.steps, args.warmup, sample=True)
    if args.dump_outputs and rank == 0:
        # what the last timed step handed its caller, before the e2e runs below go on updating the same learner
        dump_outputs(args.dump_outputs, {"features": b["obs"], "returns": b["returns"], "advantages": b["advantages"],
                                         "losses": learner.losses, "params": learner.params, "grads": learner.grads})
    if args.dump_outputs and world > 1:
        dist.barrier()      # the other ranks' next all-reduces must not wait on rank 0's dump
    ms_e2e, _ = timed(step_e2e, args.steps, max(3, args.warmup - 1))
    h2d_unique = ingest.h2d_bytes_last
    total_frames = FRAMES_PER_STEP * world
    value = total_frames / (ms_step * 1e-3)
    e2e = {"value": total_frames / (ms_e2e * 1e-3), "unit": "frames/s", "ms_per_step": ms_e2e,
           "h2d_bytes_per_step": h2d_unique, "d2h_bytes_per_step": d2h_bytes,
           "api": "cadre_b200.ingest.RolloutIngest.encode(unique=True) [+ .prefetch of the next rollout] + "
                  "RolloutPool.compute_returns + Learner.learn",
           "h2d_overlap": ("the next rollout's frames are copied under the current update phase (RolloutIngest.prefetch): "
                           "one full-rollout H2D copy per step inside the timed region") if prefetch else "in-step staging only",
           "frames_shipped_and_encoded_per_step": WORKERS * K,
           "unique_frames_per_s": WORKERS * K * world / (ms_e2e * 1e-3),
           "note": "value counts window frames (workers x T x 8) like `value`; each distinct frame crosses PCIe and "
                   "the encoder once, windows are assembled on the device (bit-identical features)"}
    e2e_full = None
    if full_windows:
        ms_full, _ = timed(step_e2e_full, args.steps, 3)
        e2e_full = {"value": total_frames / (ms_full * 1e-3), "unit": "frames/s", "ms_per_step": ms_full,
                    "h2d_bytes_per_step": ingest.h2d_bytes_last, "d2h_bytes_per_step": d2h_bytes,
                    "note": "round-1 definition: every window frame shipped over PCIe and encoded"}

    # ---- phase split of one resident step (every rank runs it: update_step contains the all-reduce)
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
    n_upd = 0
    for rep in range(2):    # second repetition is reported
        ev[0].record()
        ingest.encode(rgb_w, route_w, meas_w, b["obs"], unique=False)
        ev[1].record()
        pool.compute_returns(next_values)
        ev[2].record()
        n_upd = learner.learn(pool, PPO_EPOCH)
        ev[3].record()
        torch.cuda.synchronize()
    enc_ms, gae_ms, ppo_ms = (ev[i].elapsed_time(ev[i + 1]) for i in range(3))
    phase = {"encoder_ms": round(enc_ms, 3), "gae_ms": round(gae_ms, 3), "ppo_update_ms": round(ppo_ms, 3),
             "update_steps": n_upd, "encoder_frames_per_s": round(FRAMES_PER_STEP / (enc_ms * 1e-3)),
             "ppo_samples_per_s": round(WORKERS * T * PPO_EPOCH / (ppo_ms * 1e-3))}

    # ---- the one exchange step of the path (SURVEY.md §8e): all-reduce(sum) of the flat fp32 gradient, timed alone
    allreduce = None
    if world > 1:
        dist.barrier()
        if learner._switch is not None:      # the library's in-switch reduction on the symmetric gradient buffer
            def exchange():
                learner._switch.sum_()
        else:
            def exchange():
                dist.all_reduce(learner.grads, op=dist.ReduceOp.SUM)
        for _ in range(3):
            exchange()
        torch.cuda.synchronize()
        ar0, ar1 = torch.cuda.Event(True), torch.cuda.Event(True)
        ar0.record()
        for _ in range(10):
            exchange()
        ar1.record()
        torch.cuda.synchronize()
        ar = torch.tensor([ar0.elapsed_time(ar1) / 10], device=dev)
        dist.all_reduce(ar, op=dist.ReduceOp.MAX)
        nbytes = learner.grads.numel() * 4
        ar_ms = float(ar.item())
        allreduce = {"bytes": nbytes, "ms": round(ar_ms, 4), "algbw_GBps": round(nbytes / (ar_ms * 1e-3) / 1e9, 1),
                     "busbw_GBps": round(2 * (world - 1) / world * nbytes / (ar_ms * 1e-3) / 1e9, 1),
                     "per_step": n_upd,
                     "impl": ("cadre allreduce_kernel (multimem.ld_reduce / multimem.st)"
                              if learner._switch is not None and learner._switch.multicast else
                              "cadre allreduce_kernel (peer loads / stores)" if learner._switch is not None else
                              "ncclAllReduce, NCCL_ALGO=" + os.environ.get("NCCL_ALGO", "default"))}
        phase["allreduce"] = allreduce
        learner.grads.zero_()
        learner.check()

    # ---- per-kernel view (rank 0)
    if rank == 0:
        tf_peak, hbm_peak, peak_src = measured_peaks()

        def ev_time(fn, iters, warm=3):
            for _ in range(warm):
                fn()
            torch.cuda.synchronize()
            a, c = torch.cuda.Event(True), torch.cuda.Event(True)
            a.record()
            for _ in range(iters):
                fn()
            c.record()
            torch.cuda.synchronize()
            return a.elapsed_time(c) / iters

        # encoder launches, timed with CUDA events inside the library on the launching stream
        nb = min(ENC_CHUNK, FRAMES_PER_STEP)
        flat = (rgb_w.view(-1, 144, 256, 3), route_w.view(-1, 256, 144), meas_w.view(-1, 3))
        fbuf = torch.empty(nb, 530, device=dev)
        enc.forward_u8(flat[0][:nb], flat[1][:nb], flat[2][:nb], fbuf)
        prof = None
        for _ in range(3):
            prof = enc.profile(nb)
        fl = encoder_flops_per_frame()
        kernels = []
        for name, ms in prof:
            ent = {"name": name, "ms": round(ms, 4)}
            if name in fl:
                ent["tflops"] = round(fl[name] * nb / (ms * 1e-3) / 1e12, 1)
            kernels.append(ent)
        conv = [k for k in kernels if "tflops" in k]
        tot_ms = sum(k["ms"] for k in conv)
        tot_fl = sum(fl[k["name"]] for k in conv) * nb
        ach = tot_fl / (tot_ms * 1e-3) / 1e12
        roofline = {"kernel": "tcgen05 tile kernels (implicit-GEMM conv / linear launches of one encoder forward, "
                              f"{len(conv)} launches, batch {nb})",
                    "bound": "tensor", "achieved": round(ach, 1), "peak": tf_peak, "unit": "TFLOP/s",
                    "frac": round(ach / tf_peak, 4), "traffic": ncu_traffic(), "peak_source": peak_src + " (sustained bf16)",
                    "share_of_encoder_ms": round(tot_ms / sum(k["ms"] for k in kernels), 3),
                    "share_of_step_ms": round(enc_ms / (enc_ms + gae_ms + ppo_ms) * tot_ms / sum(k["ms"] for k in kernels), 3)}

        # the other kernel groups of the step, each against its own roofline (SURVEY.md §8d)
        rooflines = []
        idx0 = learner.sample_epoch_indices(pool.storages)[0]
        advs = [(s.advantages, t.advantages) for s, t in pool.storages]
        upd_ms = ev_time(lambda: learner.engine.update(pool.storages, advs, idx0, learner.params, learner.grads,
                                                       learner.losses), 10)
        rows = WORKERS * mb
        tf32_peak = tf_peak / 2.0
        upd_tf = PPO_FLOP_PER_ROW * rows / (upd_ms * 1e-3) / 1e12
        rooflines.append({"kernel": f"PPO update forward+backward ({learner.engine.launches} launches, {rows} rows x 2 "
                                    "heads, routed)", "bound": "tensor", "achieved": round(upd_tf, 1),
                          "peak": round(tf32_peak, 1), "unit": "TFLOP/s", "frac": round(upd_tf / tf32_peak, 4),
                          "ms": round(upd_ms, 4), "peak_source": peak_src + " sustained bf16 / 2 (tf32 operand rate)",
                          "note": "latency / L2-bound at <= 128 rows per expert (cfg 3); tensor-bound from ~2k rows"})
        m1 = torch.zeros_like(learner.params)
        m2 = torch.zeros_like(learner.params)
        ptmp = learner.params.clone()
        adam_ms = ev_time(lambda: learner.engine.adam_step(ptmp, learner.grads, m1, m2, step=3), 20)
        adam_gbs = 32.0 * ppo_params.NUM_REFERENCE_PARAMS / (adam_ms * 1e-3) / 1e9
        rooflines.append({"kernel": "per-module grad-norm + clip + Adam (sqnorm_partial/final + adam_kernel)",
                          "bound": "hbm", "achieved": round(adam_gbs, 1), "peak": hbm_peak, "unit": "GB/s",
                          "frac": round(adam_gbs / hbm_peak, 4), "ms": round(adam_ms, 4),
                          "algorithmic_bytes": "32 B / parameter (p, g, m, v read; p, m, v written; g re-read for the norm)"})
        del m1, m2, ptmp
        Eg, Tg = 65536, 1024
        r_ = torch.rand(Eg, Tg + 1, device=dev)
        v_ = torch.randn(Eg, Tg + 1, device=dev)
        mk = (torch.rand(Eg, Tg + 1, device=dev) > 0.02).float()
        nv_ = torch.randn(Eg, device=dev)
        ret_, adv_ = torch.empty(Eg, Tg + 1, device=dev), torch.empty(Eg, Tg, device=dev)
        gae_sweep_ms = ev_time(lambda: PPO.gae(r_, v_, mk, nv_, ret_, adv_), 10)
        gae_gbs = 20.0 * Eg * Tg / (gae_sweep_ms * 1e-3) / 1e9
        rooflines.append({"kernel": f"GAE + advantage normalisation, roofline sweep {Eg} sequences x {Tg} steps",
                          "bound": "hbm", "achieved": round(gae_gbs, 1), "peak": hbm_peak, "unit": "GB/s",
                          "frac": round(gae_gbs / hbm_peak, 4), "ms": round(gae_sweep_ms, 4),
                          "algorithmic_bytes": "20 B per (sequence, step)",
                          "config_latency_us": round(gae_ms * 1e3, 1),
                          "note": f"the configured call ({2 * WORKERS} sequences x {T}) is in the launch-latency regime"})
        del r_, v_, mk, nv_, ret_, adv_
        if allreduce is not None:
            if learner._switch is not None and learner._switch.multicast:
                # in-switch reduction: every GPU sends its copy of all W slices (S) plus its reduced slice (S / W) and
                # receives its reduced slice plus all W broadcast slices: S (1 + 1/W) bytes per direction
                wire = allreduce["bytes"] * (1.0 + 1.0 / world) / (allreduce["ms"] * 1e-3) / 1e9
                rooflines.append({"kernel": "gradient all-reduce: cadre allreduce_kernel (multimem.ld_reduce / multimem.st "
                                            "through NVSwitch)", "bound": "nvlink", "achieved": round(wire, 1),
                                  "peak": 770.0, "unit": "GB/s", "frac": round(wire / 770.0, 4), "ms": allreduce["ms"],
                                  "algbw_GBps": allreduce["algbw_GBps"],
                                  "algorithmic_bytes": "S (1 + 1/W) per direction per GPU, S = 77.9 MB",
                                  "peak_source": "measured peer-copy bandwidth per direction (B200_PROFILING.md); "
                                                 "nominal NVLink 5: 900"})
            else:
                rooflines.append({"kernel": "gradient all-reduce (NCCL over NVLink 5 / NVSwitch)", "bound": "nvlink",
                                  "achieved": allreduce["busbw_GBps"], "peak": 900.0, "unit": "GB/s",
                                  "frac": round(allreduce["busbw_GBps"] / 900.0, 4), "ms": allreduce["ms"],
                                  "peak_source": "nominal NVLink 5 per direction per GPU"})

        eager = None
        if world == 1 and not args.no_eager_baseline:
            # GPU-side bar (SURVEY.md §8d): the reference graph in torch eager (cuDNN / cuBLAS) on the same B200, in a
            # separate process so that no library kernel is ever loaded into the measured one
            try:
                r = subprocess.run([sys.executable, "-B", os.path.join(ROOT, "tools", "gpu_eager_baseline.py"),
                                    "--json-line"],
                                   capture_output=True, text=True, timeout=600)
                eager = json.loads(r.stdout.strip().splitlines()[-1])
                eager["cadre_encoder_ms_b640"] = round(sum(k["ms"] for k in kernels) * 640.0 / nb, 3)
                eager["cadre_ppo_update_step_ms"] = round(upd_ms + adam_ms, 3)
            except Exception as e:
                eager = {"error": repr(e)[:200]}

        enc_calls = len(ingest_schedule(FRAMES_PER_STEP))
        launches = enc_calls * enc.launches_per_forward + 2 + n_upd * (learner.engine.launches + 3)
        line = {
            "metric": METRIC, "value": value, "unit": "frames/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "fp16 operands / fp32 accumulate (encoder), tf32 / fp32 (PPO)",
            "data": "synthetic",
            "config": {"workload": workload_name(args.config), "workers_per_gpu": WORKERS, "num_steps": T,
                       "seq_length": SEQ, "mini_batch": mb, "ppo_epoch": PPO_EPOCH, "encoder_chunk": ENC_CHUNK,
                       "encoder_streams": ingest.NS,
                       "l2": f"inputs ({FRAMES_PER_STEP * 147480 // 1000000} MB of uint8 frames per step) and "
                             "activations exceed the 126 MB L2",
                       "host_cpus_bound_per_rank": numa},
            "clocks": clocks, "e2e": e2e, "e2e_full_windows": e2e_full,
            "gpu_launches": int(launches * args.steps),
            "roofline": roofline, "rooflines": rooflines,
            "cpu_baseline": cpu_baseline, "gpu_eager_baseline": eager,
            "phases": phase, "kernels": kernels,
        }
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def ingest_schedule(n):
    from cadre_b200.ingest import chunk_schedule
    return chunk_schedule(n, ENC_CHUNK, ramp=())


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="cadre", choices=["cadre", "reference"])
    ap.add_argument("--config", default=os.environ.get("CADRE_BENCH_CONFIG", "cfg3"), choices=sorted(CONFIGS))
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-eager-baseline", action="store_true")
    ap.add_argument("--no-full-windows", action="store_true")
    ap.add_argument("--profile-step", action="store_true",
                    help="run ONE resident step inside cudaProfilerStart/Stop and exit (ncu --profile-from-start off)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last resident step computed on rank 0 to DIR/<name>.npy "
                         "(float32): rollout features, returns, advantages, the raw losses [worker, head, (value loss, "
                         "action loss, entropy)] of the last update step before the loss coefficients, parameters and "
                         f"gradient; arrays of more than {DUMP_MAX_ELEMS} elements as a fixed, seeded sample")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl == "reference" or args.profile_step):
        ap.error("--dump-outputs needs the timed steps of --impl cadre (not --impl reference or --profile-step)")
    args.warmup = max(args.warmup, 0)
    if args.impl == "reference":
        run_reference(args)
    else:
        args.warmup = max(args.warmup, 3)
        run_cadre(args)


if __name__ == "__main__":
    main()
