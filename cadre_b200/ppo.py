"""ctypes front of the PPO update plan in libcadre_sm100.so (cadre_ppo_* in include/cadre_b200.h).

`PpoEngine` is the device-side replacement of `CadreAgent.update_policy` + `Shared_grad_buffers.add_gradient`
+ the `chief` step (ppo_agent/agent.py:166-237, models.py:231-239, chief.py:13-21) for W logical workers whose
rollouts live on this GPU. Host logic here is only pointer / index marshalling.
"""
import ctypes

import numpy as np
import torch

from . import _lib, ppo_params


class PpoConfigC(ctypes.Structure):
    _fields_ = [("workers", ctypes.c_int32), ("mini_batch", ctypes.c_int32), ("clip", ctypes.c_float),
                ("value_coeff", ctypes.c_float), ("clip_coeff", ctypes.c_float), ("ent_coeff", ctypes.c_float)]


class StorageRefC(ctypes.Structure):
    _fields_ = [(n, ctypes.c_void_p) for n in ("obs", "action", "value_preds", "returns", "action_log_probs", "adv",
                                               "hn", "cn", "command")]


class RolloutPoolC(ctypes.Structure):
    """Mirror of `cadre_rollout_pool`: the batched device tensors of a RolloutPool (storage n = 2 * worker + head)."""
    _fields_ = [(n, ctypes.c_void_p) for n in ("obs", "action", "action_log_probs", "value_preds", "rewards", "masks",
                                               "command", "hn", "cn")] + \
               [(n, ctypes.c_int32) for n in ("storages", "num_steps", "seq_length", "feature_dims", "hidden_size")]


ROW_OUT = 36
DIAG_TERMS = ("approx_kl", "kl_k1", "clip_frac", "value_clip_frac")      # last axis of the update diagnostics
ROLLOUT_STATS = ("explained_variance", "adv_mean", "adv_std", "return_mean", "return_std", "value_mean")


def _check_tensor(t, dtype, name):
    if t.dtype != dtype or not t.is_contiguous() or not t.is_cuda:
        raise _lib.CadreError(f"storage tensor `{name}` must be a contiguous CUDA {dtype} tensor "
                              f"(got {t.dtype}, contiguous={t.is_contiguous()}, device={t.device})")


def storage_ref(st, adv):
    """cadre_storage_ref for one RolloutStorage-like object (attributes of ppo_agent/storage.py:8-26)."""
    r = StorageRefC()
    for name, dtype in (("obs", torch.float32), ("action", torch.int64), ("value_preds", torch.float32),
                        ("returns", torch.float32), ("action_log_probs", torch.float32), ("hn", torch.float32),
                        ("cn", torch.float32), ("command", torch.int32)):
        t = getattr(st, name)
        _check_tensor(t, dtype, name)
        setattr(r, name, t.data_ptr())
    _check_tensor(adv, torch.float32, "advantages")
    r.adv = adv.data_ptr()
    return r


class PpoEngine:
    def __init__(self, workers, mini_batch, clip=0.1, value_coeff=0.1, clip_coeff=1.0, ent_coeff=0.01,
                 device="cuda:0"):
        self.device = torch.device(device)
        if self.device.type != "cuda":
            raise _lib.CadreError("PpoEngine needs a CUDA device: there is no CPU fallback")
        self.workers, self.mini_batch = int(workers), int(mini_batch)
        self._lib = _lib.lib()
        self._lib.cadre_ppo_param_count.restype = ctypes.c_int64
        assert self._lib.cadre_ppo_param_count() == ppo_params.TOTAL, "ppo_layout.h / ppo_params.py mismatch"
        cfg = PpoConfigC(self.workers, self.mini_batch, clip, value_coeff, clip_coeff, ent_coeff)
        h = ctypes.c_void_p()
        with torch.cuda.device(self.device):
            _lib.check(self._lib.cadre_ppo_create(ctypes.byref(h), ctypes.byref(cfg)))
        self._h = h
        self._refs = (StorageRefC * (2 * self.workers))()
        self._keep = None
        self.grad_groups = 1

    def __del__(self):
        h = getattr(self, "_h", None)
        if h:
            self._lib.cadre_ppo_destroy(h)
            self._h = None

    def _marshal(self, storages, advantages, indices):
        assert len(storages) == self.workers and len(advantages) == self.workers
        for w in range(self.workers):
            for h in range(2):
                self._refs[w * 2 + h] = storage_ref(storages[w][h], advantages[w][h])
        idx = np.ascontiguousarray(np.asarray(indices, dtype=np.int32))
        assert idx.shape == (self.workers, 2, self.mini_batch), idx.shape
        self._keep = (storages, advantages, idx)  # keep alive until the stream has consumed them
        return idx

    def update(self, storages, advantages, indices, params, grads, losses=None):
        """storages[w] = (steer_storage, throttle_storage); advantages[w] = (adv_steer [T,1], adv_throttle);
        indices int [W,2,mb]. Overwrites `grads` with the sum over workers of d(total_loss)/d(params) and
        returns the device tensor losses [W,2,3] = un-scaled (value, action, entropy) means per worker/head."""
        idx = self._marshal(storages, advantages, indices)
        if losses is None:
            losses = torch.empty(self.workers, 2, 3, device=self.device, dtype=torch.float32)
        with torch.cuda.device(self.device):
            _lib.check(self._lib.cadre_ppo_update(self._h, self._refs, idx.ctypes.data_as(ctypes.c_void_p),
                                                  _lib.ptr(params), _lib.ptr(grads), _lib.ptr(losses),
                                                  _lib.stream_ptr(self.device)))
        return losses

    def stage(self, storages, advantages, indices_all, first_adam_step):
        """Upload the storage references and the indices of a SEQUENCE of update steps, int [n_steps, W, 2, mb]; each
        following `update_staged` consumes the next slice and advances the device-side Adam step (the first one is
        `first_adam_step`, 1-based; 0 continues the device counter), which `adam_step*` use when called with step=0."""
        assert len(storages) == self.workers and len(advantages) == self.workers
        for w in range(self.workers):
            for h in range(2):
                self._refs[w * 2 + h] = storage_ref(storages[w][h], advantages[w][h])
        idx = np.ascontiguousarray(np.asarray(indices_all, dtype=np.int32))
        assert idx.ndim == 4 and idx.shape[1:] == (self.workers, 2, self.mini_batch), idx.shape
        self._keep = (storages, advantages, idx)
        with torch.cuda.device(self.device):
            _lib.check(self._lib.cadre_ppo_stage(self._h, self._refs, idx.ctypes.data_as(ctypes.c_void_p), idx.shape[0],
                                                 int(first_adam_step), _lib.stream_ptr(self.device)))
        return idx.shape[0]

    def update_staged(self, params, grads, losses):
        """`update` on the next staged index slice: no host data, capturable in a CUDA graph."""
        with torch.cuda.device(self.device):
            _lib.check(self._lib.cadre_ppo_update(self._h, None, None, _lib.ptr(params), _lib.ptr(grads),
                                                  _lib.ptr(losses), _lib.stream_ptr(self.device)))
        return losses

    def evaluate(self, storages, advantages, indices, params):
        """Forward only: returns [2, W*mb, 36] = value, log-prob(action), entropy, 33 normalised logits."""
        idx = self._marshal(storages, advantages, indices)
        out = torch.zeros(2, self.workers * self.mini_batch, ROW_OUT, device=self.device, dtype=torch.float32)
        with torch.cuda.device(self.device):
            _lib.check(self._lib.cadre_ppo_evaluate(self._h, self._refs, idx.ctypes.data_as(ctypes.c_void_p),
                                                    _lib.ptr(params), _lib.ptr(out), _lib.stream_ptr(self.device)))
        return out

    def act(self, storages, advantages, indices, params, row_out, pool_ref, slot, seed, tick, env_ids, hidden, actions):
        """cadre_ppo_act (workers = 1, mini_batch = E): `evaluate` into row_out [2, E, 36], then one kernel that draws
        both heads' actions of every environment (env_ids int32 [E] on the device, counter-based sampler keyed by
        seed / tick) and writes the tick into the pool `pool_ref` (RolloutPoolC) at `slot`; actions int64 [E, 2]."""
        idx = self._marshal(storages, advantages, indices)
        hn, cn = hidden
        with torch.cuda.device(self.device):
            _lib.check(self._lib.cadre_ppo_act(
                self._h, self._refs, idx.ctypes.data_as(ctypes.c_void_p), _lib.ptr(params), _lib.ptr(row_out),
                ctypes.byref(pool_ref), int(slot), ctypes.c_uint64(seed), ctypes.c_uint64(tick), _lib.ptr(env_ids),
                _lib.ptr(hn), _lib.ptr(cn), _lib.ptr(actions), _lib.stream_ptr(self.device)))
        return actions

    def ensemble_act(self, storages, advantages, indices, params_list, row_out, seed, tick, env_ids, greedy, steer_table,
                     throttle_table, controls, actions):
        """cadre_ppo_ensemble_act (workers = 1, mini_batch = E): `evaluate` with each of the K flat parameter tensors of
        `params_list` into row_out [K, 2, E, 36], then one kernel that picks every snapshot's actions (sampler keyed by
        seed / tick / env_ids / snapshot index, or the first argmax if `greedy`) into actions int64 [K, E, 2] and
        averages their controls into controls fp64 [E, 3] (steer_table fp64 [33], throttle_table fp64 [6])."""
        idx = self._marshal(storages, advantages, indices)
        K = len(params_list)
        ptrs = (ctypes.c_void_p * max(K, 1))(*[p.data_ptr() for p in params_list])
        with torch.cuda.device(self.device):
            _lib.check(self._lib.cadre_ppo_ensemble_act(
                self._h, self._refs, idx.ctypes.data_as(ctypes.c_void_p), ptrs, int(K), _lib.ptr(row_out),
                ctypes.c_uint64(seed), ctypes.c_uint64(tick), _lib.ptr(env_ids), int(greedy), _lib.ptr(steer_table),
                _lib.ptr(throttle_table), _lib.ptr(controls), _lib.ptr(actions), _lib.stream_ptr(self.device)))
        return controls, actions

    def bootstrap(self, storages, advantages, indices, params, row_out, done_mask, next_value):
        """cadre_ppo_bootstrap (mini_batch = 1): next_value [W, 2] = the value of each worker's row, 0 where bit w of
        done_mask is set; no host synchronisation."""
        idx = self._marshal(storages, advantages, indices)
        with torch.cuda.device(self.device):
            _lib.check(self._lib.cadre_ppo_bootstrap(
                self._h, self._refs, idx.ctypes.data_as(ctypes.c_void_p), _lib.ptr(params), _lib.ptr(row_out),
                ctypes.c_uint64(done_mask), _lib.ptr(next_value), _lib.stream_ptr(self.device)))
        return next_value

    def adam_step(self, params, grads, exp_avg, exp_avg_sq, step, max_grad_norm=250.0, lr=3e-4, betas=(0.9, 0.999),
                  eps=1e-8):
        with torch.cuda.device(self.device):
            _lib.check(self._lib.cadre_ppo_adam_step(
                self._h, _lib.ptr(params), _lib.ptr(grads), _lib.ptr(exp_avg), _lib.ptr(exp_avg_sq),
                ctypes.c_float(max_grad_norm), ctypes.c_float(lr), ctypes.c_float(betas[0]), ctypes.c_float(betas[1]),
                ctypes.c_float(eps), int(step), _lib.stream_ptr(self.device)))

    def module_norms(self):
        """{module name: gradient norm seen by the last adam_step} (16 entries, reference module names)."""
        buf = (ctypes.c_float * 16)()
        _lib.check(self._lib.cadre_ppo_module_norms(self._h, buf))
        out = {}
        for e in range(8):
            head, c = ppo_params.HEADS[e // 4], e % 4
            out[f"{head}_lstm_{c}"] = buf[e]
            out[f"{head}_ppo_{c}"] = buf[8 + e]
        return out

    # ---- data-parallel pipeline (see include/cadre_b200.h: cadre_ppo_set_grad_groups ...)
    def set_grad_groups(self, groups):
        _lib.check(self._lib.cadre_ppo_set_grad_groups(self._h, int(groups)))
        self.grad_groups = int(groups)

    def grad_range(self, group):
        """(offset, count, mod_begin, mod_end) of group `group`'s LSTM tensors in the flat buffers; group = -1: the
        actor-critic tensors of all experts."""
        off, cnt = ctypes.c_int64(), ctypes.c_int64()
        m0, m1 = ctypes.c_int(), ctypes.c_int()
        _lib.check(self._lib.cadre_ppo_grad_range(self._h, int(group), ctypes.byref(off), ctypes.byref(cnt),
                                                  ctypes.byref(m0), ctypes.byref(m1)))
        return off.value, cnt.value, m0.value, m1.value

    def wait_grads(self, group, stream):
        """`stream` (torch.cuda.Stream) waits until the last update() has finished that range of the gradient."""
        _lib.check(self._lib.cadre_ppo_wait_grads(self._h, int(group), ctypes.c_void_p(stream.cuda_stream)))

    def adam_step_modules(self, params, grads, exp_avg, exp_avg_sq, step, mod_begin, mod_end, max_grad_norm=250.0,
                          lr=3e-4, betas=(0.9, 0.999), eps=1e-8):
        with torch.cuda.device(self.device):
            _lib.check(self._lib.cadre_ppo_adam_step_modules(
                self._h, _lib.ptr(params), _lib.ptr(grads), _lib.ptr(exp_avg), _lib.ptr(exp_avg_sq),
                ctypes.c_float(max_grad_norm), ctypes.c_float(lr), ctypes.c_float(betas[0]), ctypes.c_float(betas[1]),
                ctypes.c_float(eps), int(step), int(mod_begin), int(mod_end), _lib.stream_ptr(self.device)))

    def set_diagnostics(self, diag=None, norms=None):
        """Destinations of the update diagnostics (cadre_ppo_set_diagnostics): every later `update*` writes `diag` fp32
        [W, 2, 4] (DIAG_TERMS per worker and head) and every later `adam_step*` writes the pre-clip norms of the modules
        it steps into `norms` fp32 [16]. None turns either off. The tensors must stay alive while they are set."""
        for t, n, name in ((diag, self.workers * 2 * len(DIAG_TERMS), "diag"), (norms, 16, "norms")):
            if t is not None:
                _check_tensor(t, torch.float32, name)
                if t.numel() != n or (self.device.index is not None and t.device.index != self.device.index):
                    raise _lib.CadreError(f"set_diagnostics: `{name}` must hold {n} floats on {self.device} "
                                          f"(got {t.numel()} on {t.device})")
        _lib.check(self._lib.cadre_ppo_set_diagnostics(self._h, _lib.ptr(diag), _lib.ptr(norms)))

    def set_target_kl(self, target_kl, total_workers=None, kl_sum=None):
        """Target-KL early stopping of staged phases (cadre_ppo_set_target_kl): None or 0 turns it off; otherwise
        `total_workers` is the worker count of all ranks and `kl_sum` fp32 [4] on this device receives each staged
        update's per-head KL sums in [0:2] (sum it over ranks, then `kl_gate`). It must stay alive while it is set."""
        if target_kl is None or target_kl == 0:
            _lib.check(self._lib.cadre_ppo_set_target_kl(self._h, ctypes.c_float(0.0), 0, None))
            return
        if kl_sum is not None:
            _check_tensor(kl_sum, torch.float32, "kl_sum")
            if kl_sum.numel() < 2:
                raise _lib.CadreError(f"set_target_kl: `kl_sum` must hold at least 2 floats (got {kl_sum.numel()})")
        _lib.check(self._lib.cadre_ppo_set_target_kl(
            self._h, ctypes.c_float(target_kl), int(total_workers if total_workers is not None else self.workers),
            _lib.ptr(kl_sum)))

    def kl_begin(self):
        """Start a phase of staged steps: clear the early stop (cadre_ppo_kl_begin)."""
        with torch.cuda.device(self.device):
            _lib.check(self._lib.cadre_ppo_kl_begin(self._h, _lib.stream_ptr(self.device)))

    def kl_gate(self):
        """The stop decision of the current staged step (cadre_ppo_kl_gate), after the cross-rank sum of `kl_sum`."""
        with torch.cuda.device(self.device):
            _lib.check(self._lib.cadre_ppo_kl_gate(self._h, _lib.stream_ptr(self.device)))

    def early_stop(self, kl_count=0):
        """Wait for the current stream and read the phase's early-stop state (cadre_ppo_early_stop): dict with `gated`, `run`,
        `applied`, `stopped_at` (None: no stop), `adam_step` (the device Adam step) and `kl` float32 [kl_count]."""
        st = (ctypes.c_int32 * 5)()
        kl = np.zeros(int(kl_count), dtype=np.float32)
        with torch.cuda.device(self.device):
            _lib.check(self._lib.cadre_ppo_early_stop(self._h, st, kl.ctypes.data_as(ctypes.c_void_p) if kl_count else None,
                                                      int(kl_count), _lib.stream_ptr(self.device)))
        return dict(gated=st[0], run=st[1], applied=st[2], stopped_at=None if st[3] < 0 else st[3], adam_step=st[4],
                    kl=kl)

    def check(self):
        """Synchronise and raise CadreError if a recurrence kernel of an earlier call timed out on a hand-off."""
        with torch.cuda.device(self.device):
            _lib.check(self._lib.cadre_ppo_check(self._h))

    @property
    def launches(self):
        return int(self._lib.cadre_ppo_launches(self._h))


def categorical_sample(logp, A, seed, tick, env_ids, word, u_out=None):
    """cadre_categorical_sample (include/cadre_b200.h): one draw per row of log-probabilities logp fp32 [rows, ld]
    (columns >= A are never read) for environments env_ids int32 [rows]. Returns (action int64 [rows], logp fp32
    [rows]); u_out (fp32 [rows] or None) receives the uniform of each draw."""
    rows, ld = logp.shape
    _check_tensor(logp, torch.float32, "logp")
    _check_tensor(env_ids, torch.int32, "env_ids")
    action = torch.empty(rows, dtype=torch.int64, device=logp.device)
    lp = torch.empty(rows, dtype=torch.float32, device=logp.device)
    with torch.cuda.device(logp.device):
        _lib.check(_lib.lib().cadre_categorical_sample(
            _lib.ptr(logp), int(ld), int(rows), int(A), ctypes.c_uint64(seed), ctypes.c_uint64(tick), _lib.ptr(env_ids),
            int(word), _lib.ptr(action), _lib.ptr(lp), _lib.ptr(u_out), _lib.stream_ptr(logp.device)))
    return action, lp


def ensemble_control(row_out, seed, tick, env_ids, steer_table, throttle_table, greedy=False):
    """cadre_ensemble_control (include/cadre_b200.h): rows fp32 [K, 2, E, 36] in `evaluate`'s format, env_ids int32
    [E], steer_table fp64 [33], throttle_table fp64 [6]. Returns (controls fp64 [E, 3], actions int64 [K, E, 2])."""
    _check_tensor(row_out, torch.float32, "row_out")
    _check_tensor(env_ids, torch.int32, "env_ids")
    _check_tensor(steer_table, torch.float64, "steer_table")
    _check_tensor(throttle_table, torch.float64, "throttle_table")
    if row_out.dim() != 4 or row_out.shape[1] != 2 or row_out.shape[3] != ROW_OUT or env_ids.numel() != row_out.shape[2]:
        raise _lib.CadreError(f"ensemble_control: row_out must be [K, 2, E, {ROW_OUT}] with E = len(env_ids) "
                              f"(got {tuple(row_out.shape)}, {env_ids.numel()} env ids)")
    if steer_table.numel() != 33 or throttle_table.numel() != 6:
        raise _lib.CadreError("ensemble_control: steer_table needs 33 entries and throttle_table 3 x 2")
    K, E = row_out.shape[0], row_out.shape[2]
    controls = torch.empty(E, 3, dtype=torch.float64, device=row_out.device)
    actions = torch.empty(K, E, 2, dtype=torch.int64, device=row_out.device)
    with torch.cuda.device(row_out.device):
        _lib.check(_lib.lib().cadre_ensemble_control(
            _lib.ptr(row_out), int(K), int(E), ctypes.c_uint64(seed), ctypes.c_uint64(tick), _lib.ptr(env_ids),
            int(greedy), _lib.ptr(steer_table), _lib.ptr(throttle_table), _lib.ptr(controls), _lib.ptr(actions),
            _lib.stream_ptr(row_out.device)))
    return controls, actions


def gae(rewards, values, masks, next_value, returns, adv, gamma=0.99, tau=0.95, normalize=True):
    """cadre_gae over E sequences: rewards/values/masks/returns fp32 [E,T+1], next_value [E], adv [E,T]."""
    E, T1 = rewards.shape
    for t in (rewards, values, masks, next_value, returns, adv):
        _check_tensor(t, torch.float32, "gae input")
    with torch.cuda.device(rewards.device):
        _lib.check(_lib.lib().cadre_gae(_lib.ptr(rewards), _lib.ptr(values), _lib.ptr(masks), _lib.ptr(next_value),
                                        _lib.ptr(returns), _lib.ptr(adv), E, T1 - 1, ctypes.c_float(gamma),
                                        ctypes.c_float(tau), int(bool(normalize)), _lib.stream_ptr(rewards.device)))
    return returns, adv


def rollout_stats(returns, values, out=None):
    """cadre_rollout_stats over E sequences: returns / values fp32 [E, T+1] after `gae` (steps t < T are used). Returns
    out fp32 [E, 6] = ROLLOUT_STATS: explained variance (NaN where Var(R) = 0), mean and std of R - V, mean and std of
    R, mean of V (fp64 sums, population variances)."""
    for t, name in ((returns, "returns"), (values, "values")):
        _check_tensor(t, torch.float32, name)
        if t.dim() != 2 or t.shape != returns.shape or t.shape[1] < 2:
            raise _lib.CadreError(f"rollout_stats: `{name}` must be [E, T+1] with T >= 1 like `returns` "
                                  f"(got {tuple(t.shape)})")
    E, T = returns.shape[0], returns.shape[1] - 1
    if out is None:
        out = torch.empty(E, len(ROLLOUT_STATS), device=returns.device, dtype=torch.float32)
    _check_tensor(out, torch.float32, "out")
    if out.shape != (E, len(ROLLOUT_STATS)):
        raise _lib.CadreError(f"rollout_stats: `out` must be [{E}, {len(ROLLOUT_STATS)}] (got {tuple(out.shape)})")
    with torch.cuda.device(returns.device):
        _lib.check(_lib.lib().cadre_rollout_stats(_lib.ptr(returns), _lib.ptr(values), E, T, _lib.ptr(out),
                                                  _lib.stream_ptr(returns.device)))
    return out
