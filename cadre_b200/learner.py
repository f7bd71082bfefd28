"""Data-parallel learner: the B200 replacement of the worker/chief handshake
(ppo_agent/train.py:76-110, ppo_agent/chief.py:8-27, ppo_agent/models.py:219-258).

Contract kept from the reference: every logical worker contributes exactly one gradient per update step;
the step applied is Adam on the SUM of the workers' gradients with a per-module clip at max_grad_norm; all
replicas hold identical parameters afterwards. How it is done here:
  * the W_local workers of a rank are processed by ONE batched cadre_ppo_update call (their gradients are
    summed on the device by construction);
  * across ranks the flat fp32 gradient (77.9 MB) is summed with one NCCL all-reduce over NVLink
    (`torch.distributed.all_reduce`), which replaces Shared_grad_buffers + the 1 Hz polling chief;
  * every rank then runs the same deterministic clip + Adam kernel, so no parameter broadcast
    (agent.py:239-243) is needed and replicas stay bit-identical.
"""
import ctypes
import math
import numbers
import os

import numpy as np
import torch

from . import _lib
from . import ppo as _ppo
from ._lib import CadreError
from . import ppo_params
from .storage import RolloutStorage

KL_TAIL = 4              # floats past the gradient that carry the per-head KL sums through the gradient exchange
KL_HIST_STEPS = 4096     # update steps of one learn() phase the engine keeps the KL of (csrc/ppo.cu, KL_HIST_CAP)


def check_target_kl(target_kl):
    """None (early stopping off) or a finite float > 0 that stays finite and > 0 in float32; raises CadreError."""
    if target_kl is None:
        return None
    v = float(target_kl) if isinstance(target_kl, numbers.Real) and not isinstance(target_kl, bool) else math.nan
    if not (math.isfinite(v) and v <= float(np.finfo(np.float32).max) and np.float32(v) > 0):
        raise CadreError(f"target_kl={target_kl!r}: expected None (off) or a finite float > 0")
    return v


class RolloutPool:
    """W x 2 RolloutStorage objects (steer, throttle per worker; train.py:44-48) whose tensors are views of
    batched device tensors, so that one GAE launch covers all 2W sequences."""

    def __init__(self, workers, rollout_cfg, device):
        self.workers, self.device = workers, torch.device(device)
        cfg = dict(rollout_cfg)
        cfg.setdefault("hidden_size", cfg["feature_dims"])
        T, S, Fd, Hd = cfg["num_steps"], cfg["seq_length"], cfg["feature_dims"], cfg["hidden_size"]
        n = workers * 2
        z = lambda *shape, dtype=torch.float32: torch.zeros(*shape, dtype=dtype, device=self.device)  # noqa: E731
        self.batched = dict(
            command=z(n, T + 1, 1, dtype=torch.int32), obs=z(n, T + 1, S, Fd), rewards=z(n, T + 1, 1),
            value_preds=z(n, T + 1, 1), returns=z(n, T + 1, 1), action_log_probs=z(n, T + 1, 1),
            action=z(n, T + 1, 1, dtype=torch.int64), masks=z(n, T + 1, 1), hn=z(n, T + 1, Hd), cn=z(n, T + 1, Hd),
            advantages=z(n, T, 1))
        self.next_value = z(n)
        self.storages = []
        for w in range(workers):
            pair = []
            for h in range(2):
                st = RolloutStorage(**cfg)
                for name, t in self.batched.items():
                    setattr(st, name, t[w * 2 + h])
                pair.append(st)
            self.storages.append(tuple(pair))
        self.num_steps, self.gamma, self.tau = T, cfg["gamma"], cfg["tau"]
        self._ref = None
        self._env_h = None

    def c_ref(self):
        """The pool's batched tensors as a `cadre_rollout_pool` (ppo.RolloutPoolC) for the device-side rollout path."""
        if self._ref is None:
            b = self.batched
            r = _ppo.RolloutPoolC()
            for name in ("obs", "action", "action_log_probs", "value_preds", "rewards", "masks", "command", "hn", "cn"):
                setattr(r, name, b[name].data_ptr())
            r.storages, r.num_steps = self.workers * 2, self.num_steps
            r.seq_length, r.feature_dims, r.hidden_size = b["obs"].shape[2], b["obs"].shape[3], b["hn"].shape[2]
            self._ref = r
        return self._ref

    def write_env_results(self, slot, rewards, masks):
        """Rewards and masks [W, 2] of every storage's slot `slot` (what `insert` stores from env.step, storage.py:45-58)
        with two host-to-device copies, whatever W is. They are staged in pinned memory. In the rollout loop the host
        rewrites that memory only after the next tick's action copy has synchronised the stream, so these copies are
        done by then and the event wait below returns at once; it guards callers that skip the act step."""
        if self._env_h is None:
            self._env_h = torch.empty(2, self.workers * 2, dtype=torch.float32, pin_memory=True)
            self._env_ev = torch.cuda.Event()
        self._env_ev.synchronize()
        h = self._env_h.numpy()
        h[0] = np.asarray(rewards, dtype=np.float32).reshape(-1)
        h[1] = np.asarray(masks, dtype=np.float32).reshape(-1)
        with torch.cuda.device(self.device):
            _lib.check(_lib.lib().cadre_rollout_env_results(
                ctypes.byref(self.c_ref()), int(slot), ctypes.c_void_p(self._env_h.data_ptr()),
                ctypes.c_void_p(self._env_h.data_ptr() + 4 * self.workers * 2), _lib.stream_ptr(self.device)))
            self._env_ev.record()

    def compute_returns(self, next_values=None, normalize=True):
        """All 2W sequences in one launch (storage.py:68-76 + train.py:82-88). next_values: [W,2] or None to use
        self.next_value."""
        if next_values is not None:
            self.next_value.copy_(torch.as_tensor(next_values, dtype=torch.float32).reshape(-1))
        b, T = self.batched, self.num_steps
        n = self.workers * 2
        _ppo.gae(b["rewards"].view(n, T + 1), b["value_preds"].view(n, T + 1), b["masks"].view(n, T + 1),
                 self.next_value, b["returns"].view(n, T + 1), b["advantages"].view(n, T), self.gamma, self.tau,
                 normalize)

    def rollout_stats(self):
        """Statistics of every storage's returns and values after `compute_returns`, one launch and one synchronisation:
        {name: float32 [W, 2]} for the names of ppo.ROLLOUT_STATS (explained variance, NaN where the returns are
        constant; mean / std of the raw advantage R - V; mean / std of the returns; mean of the values)."""
        n, T = self.workers * 2, self.num_steps
        b = self.batched
        out = _ppo.rollout_stats(b["returns"].view(n, T + 1), b["value_preds"].view(n, T + 1)).cpu().numpy()
        return {name: out[:, k].reshape(self.workers, 2) for k, name in enumerate(_ppo.ROLLOUT_STATS)}

    def state_dict(self):
        """Host copies of the batched tensors and `next_value`, and every storage's `step` cursor ([W][2]). The cursor is
        never reset (storage.py quirk 4), so the next rollout and its GAE read the slot the last one left."""
        return dict(batched={k: t.cpu() for k, t in self.batched.items()}, next_value=self.next_value.cpu(),
                    steps=[[st.step for st in pair] for pair in self.storages])

    def load_state_dict(self, state):
        """Restore a `state_dict()` in place (the storages are views of the batched tensors, and `c_ref` holds their
        addresses)."""
        for k, t in self.batched.items():
            if k not in state["batched"] or state["batched"][k].shape != t.shape:
                raise CadreError(f"RolloutPool.load_state_dict: tensor {k!r} missing or of another shape")
            t.copy_(state["batched"][k])
        self.next_value.copy_(state["next_value"])
        if len(state["steps"]) != self.workers:
            raise CadreError(f"RolloutPool.load_state_dict: {len(state['steps'])} workers in the state, {self.workers} here")
        for pair, steps in zip(self.storages, state["steps"]):
            for st, s in zip(pair, steps):
                st.step = int(s)


class Learner:
    def __init__(self, workers, mini_batch, ppo_state, device="cuda:0", clip=0.1, value_coeff=0.1, clip_coeff=1.0,
                 ent_coeff=0.01, lr=3e-4, max_grad_norm=250.0, process_group=None, seeds=None, diagnostics=False,
                 target_kl=None):
        """`diagnostics`: record, for every update step, the approximate KL, clip fractions and pre-clip module gradient
        norms in device-side histories (no host synchronisation inside a phase); read them with `diagnostics()`.
        `target_kl` (None: off): early stopping of each `learn()` phase by SB3's rule. The KL of update step n is the sum
        over the two heads of the mean over all workers of all ranks of the approximate KL; when it exceeds
        1.5 * target_kl, step n is not applied and the phase's later steps are skipped, decided on the device with the
        same bits on every rank. `early_stop()` reports the outcome."""
        target_kl = check_target_kl(target_kl)
        self.device = torch.device(device)
        self.workers, self.mini_batch = workers, mini_batch
        self.value_coeff, self.clip_coeff, self.ent_coeff = value_coeff, clip_coeff, ent_coeff
        self.lr, self.max_grad_norm = lr, max_grad_norm
        self.engine = _ppo.PpoEngine(workers, mini_batch, clip, value_coeff, clip_coeff, ent_coeff, self.device)
        self.params = ppo_params.pack_state(ppo_state, self.device)
        self.world = 1
        if process_group is not None or (torch.distributed.is_available() and torch.distributed.is_initialized()):
            self.world = torch.distributed.get_world_size(process_group)
        self.target_kl = target_kl
        # with target_kl the gradient buffer has a KL_TAIL-float tail past the parameters (the Adam chunk table never
        # reaches it): head_kernel writes this rank's per-head KL sums there, and the gradient exchange sums them
        n_grad = self.params.numel() + (KL_TAIL if target_kl is not None else 0)
        # Gradient exchange: "switch" = the library's in-switch reduction on a symmetric gradient buffer
        # (collective.SwitchAllReduce, csrc/allreduce.cu), "nccl" = torch.distributed.all_reduce. "auto" (default) takes
        # the switch from 4 ranks on when the fabric offers a multicast mapping: measured on 8 x B200 the 77.9 MB sum
        # takes 0.20 ms in the switch against 0.32 ms (NCCL default) / 0.27 ms (NCCL ring); between 2 GPUs NCCL's
        # ring is the faster one in situ.
        self.exchange = os.environ.get("CADRE_ALLREDUCE", "auto") if self.world > 1 else "none"
        if self.exchange not in ("auto", "switch", "nccl", "none"):
            raise CadreError(f"CADRE_ALLREDUCE={self.exchange!r}: expected 'auto', 'switch' or 'nccl'")
        self._switch = None
        if self.exchange == "switch" or (self.exchange == "auto" and self.world >= 4):
            from .collective import SwitchAllReduce
            try:
                self._switch = SwitchAllReduce(n_grad, self.device, process_group)
            except Exception as e:     # no symmetric memory between these devices (not one NVLink domain, two ranks per GPU)
                if self.exchange == "switch":
                    raise
                import warnings
                warnings.warn(f"cadre_b200: in-switch all-reduce unavailable ({e}); using NCCL")
            if self._switch is not None and self.exchange == "auto" and not self._switch.multicast:
                self._switch = None    # peer loads / stores only pay off between two GPUs
        if self._switch is not None:
            self.exchange = "switch"
            self._grad_buf = self._switch.buffer
        else:
            self.exchange = "nccl" if self.world > 1 else "none"
            self._grad_buf = torch.zeros(n_grad, dtype=self.params.dtype, device=self.device)
        self.grads = self._grad_buf if target_kl is None else self._grad_buf[:self.params.numel()]
        if target_kl is not None:
            self.engine.set_target_kl(target_kl, workers * self.world, self._grad_buf[self.params.numel():])
        self.exp_avg = torch.zeros_like(self.params)
        self.exp_avg_sq = torch.zeros_like(self.params)
        self.losses = torch.zeros(workers, 2, 3, device=self.device)       # last update step
        self.loss_sum = torch.zeros(workers, 2, 3, device=self.device)     # summed over the update steps of learn()
        self.loss_steps = 0
        self._step_count = 0
        self.diagnostics_on = bool(diagnostics)
        self._diag_hist = self._norm_hist = None      # [steps, W, 2, 4] and [steps, 16] of the last learn() / update_step
        self._diag_of_learn = False
        # target_kl: the last learn() phase while its outcome is on the device only (_resolve_phase reads it), its
        # per-step losses [steps, W, 2, 3], and the outcome once read
        self._phase = None
        self._loss_hist = None
        self._early_stop = None
        self.pg = process_group
        self.overlap_allreduce = os.environ.get("CADRE_NO_ALLREDUCE_OVERLAP", "0") != "1"
        self._comm_stream = None
        # one CPU RNG stream per logical worker (each reference worker is its own process with its own global RNG)
        self._rng_states = []
        if seeds is not None:
            keep = torch.get_rng_state()
            for s in seeds:
                torch.manual_seed(int(s))
                self._rng_states.append(torch.get_rng_state())
            torch.set_rng_state(keep)

    # ---------------------------------------------------------------- index sampling (bit-exact, host side)
    def sample_epoch_indices(self, storages):
        """One PPO epoch of minibatch indices for every worker: [n_minibatches][W][2][mb] (train.py:94-96: the
        steer generator draws its permutation first, then the throttle generator)."""
        per_worker = []
        keep = torch.get_rng_state() if self._rng_states else None
        for w, (st_s, st_t) in enumerate(storages):
            if self._rng_states:
                torch.set_rng_state(self._rng_states[w])
            s_chunks = st_s.sample_indices()
            t_chunks = st_t.sample_indices()
            if self._rng_states:
                self._rng_states[w] = torch.get_rng_state()
            per_worker.append((s_chunks, t_chunks))
        if keep is not None:
            torch.set_rng_state(keep)
        n_mb = min(min(len(s), len(t)) for s, t in per_worker)     # zip() of the two generators (train.py:94)
        out = np.empty((n_mb, len(storages), 2, self.mini_batch), dtype=np.int32)
        for w, (s_chunks, t_chunks) in enumerate(per_worker):
            for k in range(n_mb):
                for h, chunk in enumerate((s_chunks[k], t_chunks[k])):
                    if len(chunk) != self.mini_batch:
                        # BatchSampler(drop_last=False) yields a short last chunk when num_steps is not a multiple of
                        # num_steps // mini_batch_num (storage.py:93-97); the batched engine is sized for ONE
                        # minibatch length. CadreAgent.update_policy handles such tails (one engine per length).
                        raise CadreError(
                            f"ragged minibatch: chunk {k} of worker {w} has {len(chunk)} rows, the learner was built "
                            f"for mini_batch={self.mini_batch}; choose num_steps divisible by num_steps // "
                            "mini_batch_num or drive CadreAgent.update_policy per worker")
                    out[k, w, h] = chunk
        return out

    # ---------------------------------------------------------------- one synchronous update step
    def _setup_pipeline(self):
        """Streams, events and flat-buffer ranges of the data-parallel gradient pipeline (built on first use).
        Range k < groups - 1 = LSTM tensors of expert group k; the last range = LSTM tensors of the last group PLUS the
        actor-critic tensors of all experts, which follow them directly in the flat buffer (one collective less, and
        no collective is in flight next to the persistent BPTT kernel, which needs every SM it was launched on)."""
        # NCCL: two expert groups (range 0 is on the wire while group 1's weight-gradient GEMMs run); the in-switch
        # exchange measured no gain from splitting (8 x B200: PPO phase 7.86 ms with two ranges, 7.80 ms with one)
        default_groups = "1" if self._switch is not None else "2"
        groups = int(os.environ.get("CADRE_GRAD_GROUPS", default_groups)) if self.overlap_allreduce else 1
        self.engine.set_grad_groups(groups)
        self._comm_stream = torch.cuda.Stream(device=self.device)
        lstm = [self.engine.grad_range(g) for g in range(groups)]
        mlp = self.engine.grad_range(-1)
        assert lstm[-1][0] + lstm[-1][1] == mlp[0] and lstm[-1][3] == mlp[2]      # contiguous ranges and module ids
        self._ranges = lstm[:-1] + [(lstm[-1][0], lstm[-1][1] + mlp[1], lstm[-1][2], mlp[3])]
        self._waits = [[g] for g in range(groups - 1)] + [[groups - 1, -1]]
        self._kl_tail = None
        if self.target_kl is not None:
            # the KL sums must be summed before range 0 is stepped: in the one range when there is one, else by a
            # 16-byte exchange of their own issued before range 0's (after the BPTT kernel, like every collective here)
            if len(self._ranges) == 1:
                # (an exchange with no gated step before it - update_step, a skipped step - sums the stale tail again;
                # after a sum every rank holds the same values, so repeats only scale them, at worst to +-inf and never
                # to NaN, and the gate reads the tail only after head_kernel has rewritten it)
                off, cnt, m0, m1 = self._ranges[0]
                self._ranges[0] = (off, cnt + KL_TAIL, m0, m1)
            else:
                self._kl_tail = (self.params.numel(), KL_TAIL)
        self._reduced = [torch.cuda.Event() for _ in self._ranges]
        assert sum(r[1] for r in self._ranges) + (KL_TAIL if self._kl_tail else 0) == self._grad_buf.numel()
        assert all(r[0] % 4 == 0 and r[1] % 4 == 0 for r in self._ranges)        # 16-byte vectors in the exchange

    def _exchange_and_step(self, step):
        """all-reduce(sum) + per-module clip + Adam on the gradient the last engine.update left in self.grads.
        `step`: 1-based Adam step, or 0 to use the device-side counter (staged sequences of update steps).

        With more than one rank the gradient exchange is pipelined against the end of the backward pass: the LSTM
        weight gradients (72 of the 78 MB) are produced per group of experts, each group one contiguous range of the
        flat buffer; a communication stream all-reduces range k as soon as its event fires while the GEMMs of group
        k+1 still run, and the main stream applies clip + Adam to the modules of range k - a per-module operation,
        chief.py:16-21 - while range k+1 is on the wire. Sums, clip coefficients and Adam arithmetic are those of the
        single all-reduce + single step.
        With target_kl, a staged step (step = 0) is gated after the KL sums have been summed across ranks and before
        the first clip + Adam of the step."""
        gate = self.target_kl is not None and step == 0
        if self.world > 1:
            main = torch.cuda.current_stream(self.device)
            with torch.cuda.stream(self._comm_stream):
                for k, (off, cnt, _, _) in enumerate(self._ranges):
                    for g in self._waits[k]:
                        self.engine.wait_grads(g, self._comm_stream)
                    if k == 0 and gate and self._kl_tail is not None:
                        self._sum_over_ranks(*self._kl_tail)
                    self._sum_over_ranks(off, cnt)
                    self._reduced[k].record(self._comm_stream)
            for k, (_, _, m0, m1) in enumerate(self._ranges):
                main.wait_event(self._reduced[k])
                if k == 0 and gate:
                    self.engine.kl_gate()
                self.engine.adam_step_modules(self.params, self.grads, self.exp_avg, self.exp_avg_sq, step, m0, m1,
                                              self.max_grad_norm, self.lr)
        else:
            if gate:
                self.engine.kl_gate()
            self.engine.adam_step(self.params, self.grads, self.exp_avg, self.exp_avg_sq, step, self.max_grad_norm,
                                  self.lr)
        if not gate:        # (a gated phase keeps per-step losses instead: _resolve_phase)
            self.loss_sum += self.losses
            self.loss_steps += 1

    def _sum_over_ranks(self, off, cnt):
        """[off, off + cnt) of the gradient buffer <- its sum over ranks, on the current (communication) stream."""
        if self._switch is not None:
            self._switch.sum_(off, cnt, stream=self._comm_stream)
        else:
            torch.distributed.all_reduce(self._grad_buf[off:off + cnt], op=torch.distributed.ReduceOp.SUM, group=self.pg)

    def update_step(self, storages, indices, async_losses=True):
        """update_policy for all local workers -> all-reduce(sum) -> per-module clip + Adam (one step, eagerly).
        storages[w] = (steer, throttle) RolloutStorage with `.advantages`; indices int32 [W,2,mb]."""
        advs = [(s.advantages, t.advantages) for s, t in storages]
        self._resolve_phase()      # (after a gated learn(): the Adam step actually reached)
        if self.world > 1 and self._comm_stream is None:
            self._setup_pipeline()
        self._diag_of_learn = False
        self._diag_step(0, 1)
        self.engine.update(storages, advs, indices, self.params, self.grads, self.losses)
        self._step_count += 1
        self._exchange_and_step(self._step_count)
        self._diag_step(None)
        return self.losses if async_losses else self.scaled_losses()

    def scaled_losses(self, mean=False):
        """[W,3] = (value_loss*coeff, action_loss*coeff, entropy*coeff) per worker, like update_policy's return:
        of the LAST update step, or with `mean=True` averaged over the update steps since the last `learn()` began
        (what train.py:98-100, 112-116 logs). After a learn() stopped by target_kl: of the steps that ran their
        forward (the applied ones and the one that stopped the phase)."""
        self._resolve_phase()
        L = (self.loss_sum / max(1, self.loss_steps) if mean else self.losses).sum(1).cpu()
        return L * torch.tensor([self.value_coeff, self.clip_coeff, self.ent_coeff])

    # ---------------------------------------------------------------- a whole learn() phase
    def learn(self, pool_or_storages, ppo_epoch=4):
        """ppo_epoch x minibatches of update steps over already computed returns / advantages (train.py:93-110).
        All minibatch indices of the phase are drawn first (same per-worker RNG streams and order as one generator
        pair per epoch, train.py:94) and uploaded once together with the storage references; every update step then
        consumes the next slice of that device-side table (and the device-side Adam step), so no host data moves
        between the steps of a phase."""
        storages = pool_or_storages.storages if hasattr(pool_or_storages, "storages") else pool_or_storages
        self.loss_sum.zero_()
        self.loss_steps = 0
        if self.world > 1 and self._comm_stream is None:
            self._setup_pipeline()
        idx_all = np.concatenate([self.sample_epoch_indices(storages) for _ in range(ppo_epoch)], 0)
        advs = [(s.advantages, t.advantages) for s, t in storages]
        steps = idx_all.shape[0]
        gate = self.target_kl is not None
        if gate:
            if steps > KL_HIST_STEPS:
                raise CadreError(f"learn(): {steps} update steps in one phase; target_kl supports up to {KL_HIST_STEPS}")
            # the Adam step of the first staged step: the host's count, or, while the previous gated phase is unread,
            # the device counter it left (the steps it actually applied)
            first = 0 if self._phase is not None else self._step_count + 1
            self._loss_hist = torch.zeros(steps, self.workers, 2, 3, device=self.device)
            self._phase, self._early_stop = dict(steps=steps), None
            self.engine.kl_begin()
        self._diag_of_learn = True
        n = 0
        while n < steps:                                  # (the staging table holds 64 steps)
            m = min(64, steps - n)
            self.engine.stage(storages, advs, idx_all[n:n + m], (first if n == 0 else 0) if gate else self._step_count + 1)
            for k in range(m):
                self._diag_step(n + k, steps)
                self.engine.update_staged(self.params, self.grads, self._loss_hist[n + k] if gate else self.losses)
                self._exchange_and_step(0)
                if not gate:
                    self._step_count += 1
            n += m
        self._diag_step(None)
        self.loss_steps = steps
        return steps

    @property
    def step_count(self):
        """Adam steps applied so far (after a gated learn(), reading it synchronises once). Callers that step the
        optimizer themselves (utils.chief) may assign it, as with a plain attribute."""
        self._resolve_phase()
        return self._step_count

    @step_count.setter
    def step_count(self, value):
        self._resolve_phase()
        self._step_count = value

    def _resolve_phase(self):
        """After a learn() with target_kl: read its outcome (one synchronisation) into the Adam step count, the losses
        of the last step that ran and their sum over the steps that ran. Nothing to do otherwise."""
        if self._phase is None:
            return
        steps = self._phase["steps"]
        r = self.engine.early_stop(steps)
        kl = r["kl"]
        kl[r["run"]:] = np.nan
        self._early_stop = dict(steps=steps, applied=r["applied"], stopped_at=r["stopped_at"], kl=kl)
        self._step_count = r["adam_step"]
        self.loss_sum.zero_()
        for i in range(r["run"]):                         # the same sum, in the same order, as an ungated phase
            self.loss_sum += self._loss_hist[i]
        self.losses.copy_(self._loss_hist[r["run"] - 1])
        self.loss_steps = r["run"]
        self._phase = None

    def early_stop(self):
        """Outcome of the last learn() with target_kl (one synchronisation): {"steps": staged steps, "applied": steps
        whose Adam update was applied, "stopped_at": index of the step whose KL exceeded 1.5 * target_kl (it was not
        applied, nor were the steps after it) or None, "kl": float32 [steps] KL of each step, NaN for steps that did not
        run}."""
        if self.target_kl is None:
            raise CadreError("early_stop() needs Learner(..., target_kl=...)")
        self._resolve_phase()
        if self._early_stop is None:
            raise CadreError("early_stop(): no learn() phase has run yet")
        return dict(self._early_stop, kl=self._early_stop["kl"].copy())

    # ---------------------------------------------------------------- diagnostics
    def _diag_step(self, k, steps=None):
        """With diagnostics on: point the engine at row k of histories of `steps` update steps (new histories when k is
        0); k = None detaches them. Only host-side pointers change, so this costs no synchronisation."""
        if not self.diagnostics_on:
            return
        if k is None:
            self.engine.set_diagnostics(None, None)
            return
        if k == 0:    # (with target_kl, rows of steps that do not run stay NaN)
            fill = math.nan if self.target_kl is not None else 0.0
            self._diag_hist = torch.full((steps, self.workers, 2, len(_ppo.DIAG_TERMS)), fill, device=self.device)
            self._norm_hist = torch.full((steps, 16), fill, device=self.device)
        self.engine.set_diagnostics(self._diag_hist[k], self._norm_hist[k])

    def diagnostics(self):
        """Diagnostics of the update steps of the last `learn()` (or of the last `update_step`), one synchronisation.
        Per local worker and head, [steps, W, 2]: `approx_kl` (mean of expm1(d) - d, d = log-prob - old log-prob),
        `kl_k1` (mean of -d), `clip_frac` (rows with |ratio - 1| > clip) and `value_clip_frac` (rows with
        |value - old value| > clip); [steps, 16]: `grad_norm`, every module's gradient norm before clipping (after the
        all-reduce, so the same on every rank), columns in `modules` order (the reference's model_dict order), and
        `grad_clipped` = grad_norm > max_grad_norm.
        With target_kl also `applied`, bool [steps], and `stopped_at` (see `early_stop()`); rows of steps that did not
        run are NaN, the row of the step that stopped the phase holds its values."""
        if not self.diagnostics_on:
            raise CadreError("diagnostics() needs Learner(..., diagnostics=True)")
        if self._diag_hist is None:
            raise CadreError("diagnostics(): no update step has run yet")
        steps = self._diag_hist.shape[0]
        flat = torch.cat([self._diag_hist.reshape(-1), self._norm_hist.reshape(-1)]).cpu().numpy()
        d = flat[:self._diag_hist.numel()].reshape(self._diag_hist.shape)
        norms = flat[self._diag_hist.numel():].reshape(steps, 16)
        modules = list(ppo_params.MODULE_ORDER)
        # engine module ids: e = LSTM of expert e, 8 + e = actor-critic of expert e (expert = head * 4 + command)
        cols = [ppo_params.expert_of(m) + (0 if "_lstm_" in m else 8) for m in modules]
        out = {name: d[..., i] for i, name in enumerate(_ppo.DIAG_TERMS)}
        out["grad_norm"] = norms[:, cols]
        out["grad_clipped"] = out["grad_norm"] > self.max_grad_norm
        out["modules"] = modules
        if self.target_kl is not None:
            if self._diag_of_learn:
                es = self.early_stop()
                out["applied"] = np.arange(steps) < es["applied"]
                out["stopped_at"] = es["stopped_at"]
            else:
                out["applied"], out["stopped_at"] = np.ones(steps, dtype=bool), None
        return out

    def check(self):
        """Synchronise and raise CadreError if a bounded wait inside a kernel (LSTM hand-off, all-reduce barrier) ever
        timed out."""
        self.engine.check()
        if self._switch is not None:
            self._switch.check()

    def state(self):
        return ppo_params.unpack_state(self.params)

    # ---------------------------------------------------------------- checkpoints
    def state_dict(self):
        """Host copies of the optimizer state: params, exp_avg, exp_avg_sq, the Adam step count (after a gated learn(),
        the steps actually applied: one synchronisation), the parameter count of the library and the per-worker
        minibatch RNG states."""
        self._resolve_phase()
        return dict(params=self.params.cpu(), exp_avg=self.exp_avg.cpu(), exp_avg_sq=self.exp_avg_sq.cpu(),
                    step_count=self._step_count, param_count=int(_lib.lib().cadre_ppo_param_count()),
                    rng_states=[s.clone() for s in self._rng_states])

    def load_state_dict(self, state):
        """Restore a `state_dict()`. params and the moments are copied in place: the acting replica
        (`agent.owner.params`) aliases `params`, and the gradient buffer may be symmetric memory, so no tensor is
        rebound. The next learn() takes its first Adam step from the restored count."""
        n = self.params.numel()
        if int(state["param_count"]) != n or any(state[k].numel() != n for k in ("params", "exp_avg", "exp_avg_sq")):
            raise CadreError(f"load_state_dict: {state['param_count']} parameters in the state, the learner has {n}")
        if len(state["rng_states"]) != len(self._rng_states):
            raise CadreError(f"load_state_dict: {len(state['rng_states'])} minibatch RNG streams in the state, the "
                             f"learner has {len(self._rng_states)}")
        for k in ("params", "exp_avg", "exp_avg_sq"):
            getattr(self, k).copy_(state[k].reshape(-1))
        self._step_count = int(state["step_count"])
        self._rng_states = [s.clone() for s in state["rng_states"]]
        self._phase = self._early_stop = None
