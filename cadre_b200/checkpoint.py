"""Training checkpoints: the on-disk format, durable writes, the choice of checkpoint to resume from and the check that
a checkpoint belongs to the run that resumes it (used by `train(checkpoint_dir=, resume=)`).

Layout, one directory per checkpoint, n = episodes completed:
  <dir>/ep_<n>/learner.pt   rank 0: params, Adam moments and step, parameter count, run config, encoder fingerprint,
                            replica fingerprint
  <dir>/ep_<n>/rank_<r>.pt  every rank: its rollout pool, actor, environments, RNG states and history
  <dir>/ep_<n>/COMPLETE     rank 0, once every rank's file is durable
Every file is written under a temporary name, fsynced, renamed into place and its directory fsynced. A save that dies
part-way leaves no COMPLETE marker, and `latest` ignores such a directory. Nothing is ever deleted.

Files are read with `torch.load(weights_only=False)` (they hold numpy arrays and RandomState tuples): load only
checkpoints you wrote yourself."""
import hashlib
import os
import re

import torch

from ._lib import CadreError

LEARNER_FILE = "learner.pt"
COMPLETE = "COMPLETE"
# fields a resumed run must share with the checkpoint, otherwise it cannot continue the same trajectory
STRUCTURAL = ("world_size", "workers", "num_steps", "mini_batch_num", "seq_length", "feature_dims", "hidden_size",
              "param_count", "env_seed", "batched_acting", "device_rollout", "encoder_fingerprint")
# fields a resumed run takes from its own config (rank 0 logs the ones that differ from the checkpoint)
HYPERPARAMETERS = ("lr", "clip", "value_coeff", "clip_coeff", "ent_coeff", "max_grad_norm", "target_kl", "ppo_epoch",
                   "gamma", "tau", "use_adv_norm")
_EP = re.compile(r"^ep_(\d+)$")


def episode_dir(root, episodes):
    return os.path.join(root, "ep_{}".format(int(episodes)))


def rank_file(rank):
    return "rank_{}.pt".format(int(rank))


def encoder_fingerprint(danet_state):
    """sha256 (hex) over the names, dtypes, shapes and bytes of the encoder's state dict, in name order."""
    h = hashlib.sha256()
    for name in sorted(danet_state):
        t = torch.as_tensor(danet_state[name]).detach().cpu().contiguous()
        h.update("{}|{}|{}|".format(name, t.dtype, tuple(t.shape)).encode())
        h.update(t.reshape(-1).view(torch.uint8).numpy().tobytes())
    return h.hexdigest()


def replica_fingerprint(*tensors):
    """One int64 on the tensors' device: the 32-bit words of the tensors, concatenated, each weighted by its position
    + 1, summed modulo 2^64. Integer sums do not depend on the reduction order, so equal bits give equal fingerprints on
    every rank, and changing any one word changes it."""
    fp, base = None, 0
    for t in tensors:
        bits = t.detach().reshape(-1).view(torch.int32).to(torch.int64)
        w = torch.arange(base + 1, base + 1 + bits.numel(), dtype=torch.int64, device=bits.device)
        s = (bits * w).sum()
        fp = s if fp is None else fp + s
        base += bits.numel()
    return fp


def all_equal(value, learner):
    """True on every rank iff the int64 `value` (a one-element tensor) is the same on every rank of `learner`'s process
    group (all-reduce MIN and MAX; gloo reduces a host copy, NCCL a device one)."""
    if learner.world == 1:
        return True
    device = "cpu" if torch.distributed.get_backend(learner.pg) == "gloo" else learner.device
    lo = value.reshape(1).to(device).clone()
    hi = lo.clone()
    torch.distributed.all_reduce(lo, op=torch.distributed.ReduceOp.MIN, group=learner.pg)
    torch.distributed.all_reduce(hi, op=torch.distributed.ReduceOp.MAX, group=learner.pg)
    return bool(lo.item() == hi.item())


def _fsync_dir(path):
    fd = os.open(path, os.O_RDONLY)
    try:
        os.fsync(fd)
    finally:
        os.close(fd)


def _write_durable(path, obj):
    """torch.save to path + '.tmp', fsync, rename over `path`, fsync the directory."""
    tmp = path + ".tmp"
    with open(tmp, "wb") as f:
        torch.save(obj, f)
        f.flush()
        os.fsync(f.fileno())
    os.replace(tmp, path)
    _fsync_dir(os.path.dirname(path))


def is_complete(path):
    return os.path.isfile(os.path.join(path, COMPLETE))


def latest(root):
    """The newest complete checkpoint directory under `root` (the largest n of an ep_<n> with a COMPLETE marker), or
    None. Directories of saves that did not finish are ignored."""
    best = None
    if os.path.isdir(root):
        for name in os.listdir(root):
            m = _EP.match(name)
            if m and is_complete(os.path.join(root, name)) and (best is None or int(m.group(1)) > best):
                best = int(m.group(1))
    return None if best is None else episode_dir(root, best)


def resolve(resume, checkpoint_dir):
    """The checkpoint directory `resume` names: "latest" (the newest complete one under `checkpoint_dir`, or None when
    there is none yet) or a path to an ep_<n> directory, which must be complete."""
    if resume == "latest":
        if checkpoint_dir is None:
            raise CadreError('resume="latest" needs checkpoint_dir')
        return latest(checkpoint_dir)
    if not is_complete(resume):
        raise CadreError(f"resume={resume!r}: not a complete checkpoint directory (no {COMPLETE} marker)")
    return resume


def run_config(world_size, workers, train_cfg, agent_cfg, env_cfg, rollout_cfg, hidden_size, param_count,
               batched_acting, device_rollout, encoder_fingerprint):
    """The structural fields and hyperparameters of a run, as stored in learner.pt and compared on resume."""
    return dict(
        world_size=int(world_size), workers=int(workers), num_steps=int(rollout_cfg["num_steps"]),
        mini_batch_num=int(rollout_cfg["mini_batch_num"]), seq_length=int(rollout_cfg["seq_length"]),
        feature_dims=int(rollout_cfg["feature_dims"]), hidden_size=int(hidden_size), param_count=int(param_count),
        env_seed=int(env_cfg.get("seed", 0)), batched_acting=bool(batched_acting), device_rollout=bool(device_rollout),
        encoder_fingerprint=encoder_fingerprint,
        lr=train_cfg["lr"], clip=agent_cfg["clip"], value_coeff=agent_cfg["value_coeff"],
        clip_coeff=agent_cfg["clip_coeff"], ent_coeff=agent_cfg["ent_coeff"], max_grad_norm=train_cfg["max_grad_norm"],
        target_kl=train_cfg.get("target_kl"), ppo_epoch=train_cfg["ppo_epoch"], gamma=rollout_cfg["gamma"],
        tau=rollout_cfg["tau"], use_adv_norm=train_cfg["use_adv_norm"])


def check_config(saved, current, log=None):
    """Raise CadreError naming the first structural field in which `current` differs from the checkpoint's `saved`;
    log one line naming the hyperparameters that differ (the current values are used)."""
    for k in STRUCTURAL:
        if saved.get(k) != current.get(k):
            raise CadreError(f"checkpoint does not match this run: {k} is {saved.get(k)!r} in the checkpoint and "
                             f"{current.get(k)!r} now")
    diff = [k for k in HYPERPARAMETERS if saved.get(k) != current.get(k)]
    if diff and log is not None:
        log("Resume: hyperparameters differ from the checkpoint, using the current ones: " +
            ", ".join(f"{k} {saved.get(k)!r} -> {current.get(k)!r}" for k in diff))
    return diff


def save(root, episodes, rank, learner, config, rank_state):
    """Write checkpoint `root`/ep_<episodes>. Collective: every rank of `learner`'s process group calls it at the same
    point. Before anything is written, the ranks check that their replicas (params and both Adam moments) are
    bit-identical; rank 0 then writes learner.pt, every rank its rank file, and rank 0 writes COMPLETE once every rank
    has reported its file durable. A replica mismatch or a failed write on any rank raises CadreError on every rank and
    leaves no COMPLETE marker. Returns the checkpoint directory."""
    path = episode_dir(root, episodes)
    if rank == 0:
        os.makedirs(path, exist_ok=True)
        if is_complete(path):             # an older save of the same episode is being replaced
            os.remove(os.path.join(path, COMPLETE))
            _fsync_dir(path)
    fp = replica_fingerprint(learner.params, learner.exp_avg, learner.exp_avg_sq)
    if not all_equal(fp, learner):   # (also orders the marker removal before every rank's write)
        raise CadreError(f"checkpoint ep_{episodes}: the replicas of the ranks differ (params / Adam moments); "
                         "nothing was saved")
    error = None
    try:
        os.makedirs(path, exist_ok=True)
        state = learner.state_dict()
        rng = state.pop("rng_states")                  # per rank: one minibatch RNG stream per local worker
        if rank == 0:
            _write_durable(os.path.join(path, LEARNER_FILE), dict(
                learner=state, config=config, replica_fingerprint=int(fp.item()), episodes=int(episodes)))
        _write_durable(os.path.join(path, rank_file(rank)), dict(rank_state, rng_states=rng, episodes=int(episodes)))
    except Exception as e:   # every rank has to learn that the save failed, not only this one
        error = e
    failed = torch.tensor([0 if error is None else 1], dtype=torch.int64)
    if not all_equal(failed, learner) or error is not None:
        raise CadreError(f"checkpoint ep_{episodes}: a rank failed to write its files ({error!r} on this rank); "
                         "the checkpoint is not complete") from error
    if rank == 0:
        with open(os.path.join(path, COMPLETE), "w") as f:
            f.write("{}\n".format(int(episodes)))
            f.flush()
            os.fsync(f.fileno())
        _fsync_dir(path)
    return path


def load(path, rank, config, log=None):
    """Read checkpoint `path` for `rank` after checking it against this run's `config` (check_config). Returns
    (learner.pt contents, this rank's rank-file contents)."""
    if not is_complete(path):
        raise CadreError(f"{path}: not a complete checkpoint directory (no {COMPLETE} marker)")
    shared = torch.load(os.path.join(path, LEARNER_FILE), map_location="cpu", weights_only=False)
    check_config(shared["config"], config, log)
    mine = torch.load(os.path.join(path, rank_file(rank)), map_location="cpu", weights_only=False)
    if mine["episodes"] != shared["episodes"]:
        raise CadreError(f"{path}: {rank_file(rank)} belongs to episode {mine['episodes']}, "
                         f"{LEARNER_FILE} to {shared['episodes']}")
    return shared, mine


def check_restored(learner, shared):
    """After `learner.load_state_dict`: the replica fingerprint of the loaded params and moments equals the stored one."""
    fp = int(replica_fingerprint(learner.params, learner.exp_avg, learner.exp_avg_sq).item())
    if fp != shared["replica_fingerprint"]:
        raise CadreError("checkpoint: the restored params / Adam moments do not match the fingerprint saved with them")
