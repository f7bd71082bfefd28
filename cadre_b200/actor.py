"""Batched acting with a per-environment frame cache (SURVEY.md §8f row 1; reference: CadreAgent.act,
ppo_agent/agent.py:114-141, one environment per process).

The env wrapper hands every tick the last `seq_length` = 8 frames (env_wrapper.py:900-914) and the window slides by
ONE frame per tick, while the frozen perception encoder maps each frame independently (eval-mode BN, per-frame
route normalisation, agent.py:43-75). So, per environment, seven of the eight [530] features of a tick were
already computed for the previous tick. `BatchedActor` keeps them in a device ring, encodes only the newest frame of
each of E environments in one batch (E frames instead of 8E), and runs the per-command LSTM + actor-critic once for
all E environments (rows routed by command). Results equal E independent `CadreAgent.act` calls on the full windows;
only the order of the host-side Categorical draws differs (environment-major here).

`act_into` / `bootstrap_into` are the device-side rollout path: actions are drawn on the device by a counter-based
sampler keyed by (seed, env id, tick) (include/cadre_b200.h, cadre_categorical_sample) and the whole tick is written
into a RolloutPool by one kernel, so a tick costs the same number of launches and copies for any number of workers."""
from types import SimpleNamespace

import numpy as np
import torch
import torch.nn.functional as F

from . import ppo as _ppo


class BatchedActor:
    def __init__(self, agent, num_envs, verify_window=True, seed=0, env_ids=None):
        """agent: a cadre_b200.agent.CadreAgent (owns the encoder and the flat PPO parameters). `seed` and `env_ids`
        (default 0..E-1) key the device-side sampler of `act_into`: environment e's draw at a tick depends only on
        (seed, env_ids[e], tick, its log-probabilities), not on the batch it is stepped in."""
        self.agent, self.E = agent, int(num_envs)
        self.device = agent.device
        self.F, self.S = agent.lstm_input, 8
        self.verify_window = verify_window
        self.feats = torch.zeros(self.E, self.S, self.F, device=self.device)
        # newest frame of the previous tick per env: the window slid by one iff it is now the second newest
        self._last = [None] * self.E
        self._engine = _ppo.PpoEngine(1, self.E, agent.clip, agent.value_coeff, agent.clip_coeff, agent.ent_coeff,
                                      self.device)
        z = lambda *s, dtype=torch.float32: torch.zeros(*s, dtype=dtype, device=self.device)  # noqa: E731
        self._st = [SimpleNamespace(obs=self.feats, action=z(self.E, 1, dtype=torch.int64), value_preds=z(self.E, 1),
                                    returns=z(self.E, 1), action_log_probs=z(self.E, 1), hn=z(self.E, self.F),
                                    cn=z(self.E, self.F), command=z(self.E, 1, dtype=torch.int32)) for _ in range(2)]
        self._adv = (z(self.E, 1), z(self.E, 1))
        self._idx = [[list(range(self.E)), list(range(self.E))]]
        # pinned staging for the newest frames (one H2D per tensor and tick)
        self._rgb_h = torch.empty(self.E, 144, 256, 3, dtype=torch.uint8, pin_memory=True)
        self._route_h = torch.empty(self.E, 256, 144, dtype=torch.uint8, pin_memory=True)
        self._meas_h = torch.empty(self.E, 3, dtype=torch.float64, pin_memory=True)
        self._cmd_h = torch.empty(self.E, 1, dtype=torch.int32, pin_memory=True)
        self.frames_encoded = 0
        # device-side rollout path (act_into / bootstrap_into)
        self.seed = int(seed)
        self.env_ids = list(range(self.E)) if env_ids is None else [int(i) for i in env_ids]
        if len(self.env_ids) != self.E:
            raise ValueError(f"env_ids has {len(self.env_ids)} entries for {self.E} environments")
        self.ticks = 0                                       # act_into calls so far: the sampler's tick counter
        self._env_ids_d = torch.tensor(self.env_ids, dtype=torch.int32, device=self.device)
        self._rows = z(2, self.E, _ppo.ROW_OUT)
        self._act_d = z(self.E, 2, dtype=torch.int64)
        self._act_h = torch.empty(self.E, 2, dtype=torch.int64, pin_memory=True)
        self._boot = None

    # ------------------------------------------------------------------ perception with the frame cache
    def _slid_by_one(self, e, tick):
        last = self._last[e]
        if last is None:
            return False
        if not self.verify_window:
            return True
        return (np.array_equal(tick["rgb"][-2], last[0]) and np.array_equal(tick["route_fig"][-2], last[1])
                and np.array_equal(tick["measurements"][-2], last[2]))

    def _env_list(self, ticks, envs):
        """The environments `ticks` belongs to: all E in order when `envs` is None, else the listed distinct ids."""
        if envs is None:
            assert len(ticks) == self.E
            return list(range(self.E))
        envs = [int(e) for e in envs]
        if len(ticks) != len(envs):
            raise ValueError(f"{len(ticks)} ticks for {len(envs)} environments")
        if len(set(envs)) != len(envs) or any(e < 0 or e >= self.E for e in envs):
            raise ValueError(f"envs must be distinct ids in [0, {self.E}) (got {envs})")
        return envs

    def encode(self, ticks, envs=None):
        """ticks: list of E tick_data dicts, or, with `envs` (distinct environment ids), one per listed environment:
        only those windows are updated, the others stay as they are. Returns the [E, 8, 530] feature windows."""
        envs = self._env_list(ticks, envs)
        full = [i for i, e in enumerate(envs) if not self._slid_by_one(e, ticks[i])]
        enc = self.agent.vae_model
        dev = self.agent.vae_device
        if len(full) < len(envs):   # newest frame of every environment whose window slid by one
            inc = [i for i in range(len(envs)) if i not in set(full)] if full else list(range(len(envs)))
            n = len(inc)
            rgb_np, route_np, meas_np = self._rgb_h.numpy(), self._route_h.numpy(), self._meas_h.numpy()
            for j, i in enumerate(inc):
                np.copyto(rgb_np[j], ticks[i]["rgb"][-1])
                np.copyto(route_np[j], ticks[i]["route_fig"][-1])
                meas_np[j] = ticks[i]["measurements"][-1]
            new = enc.forward_u8(self._rgb_h[:n].to(dev, non_blocking=True), self._route_h[:n].to(dev, non_blocking=True),
                                 self._meas_h[:n].to(dev, non_blocking=True)).to(self.device)
            inc_envs = [envs[i] for i in inc]
            if inc_envs == list(range(self.E)):
                self.feats[:, :-1] = self.feats[:, 1:].clone()
                self.feats[:, -1] = new
            else:
                ids = torch.as_tensor(inc_envs, device=self.device)
                self.feats[ids, :-1] = self.feats[ids, 1:].clone()
                self.feats[ids, -1] = new
            self.frames_encoded += n
        for i in full:   # first tick after a reset (or a window that did not slide): all eight frames
            t = ticks[i]
            self.feats[envs[i]] = enc.forward_u8(
                torch.from_numpy(np.ascontiguousarray(t["rgb"])).to(dev),
                torch.from_numpy(np.ascontiguousarray(t["route_fig"])).to(dev),
                torch.from_numpy(np.ascontiguousarray(t["measurements"], dtype=np.float64)).to(dev)).to(self.device)
            self.frames_encoded += self.S
        for i, e in enumerate(envs):
            t = ticks[i]
            self._last[e] = (np.array(t["rgb"][-1], copy=True), np.array(t["route_fig"][-1], copy=True),
                             np.array(t["measurements"][-1], copy=True))
        return self.feats

    def reset(self, env_id):
        """Forget environment `env_id`'s window (call after env.reset())."""
        self._last[env_id] = None

    # ------------------------------------------------------------------ checkpoints
    def state_dict(self):
        """What the next tick depends on: the sampler's counter (`ticks`, `seed`, `env_ids`), the frame cache (`feats`
        on the host, `_last`, whose arrays are private copies that are replaced, never modified) and `frames_encoded`."""
        return dict(ticks=self.ticks, seed=self.seed, env_ids=list(self.env_ids), feats=self.feats.cpu(),
                    last=list(self._last),
                    frames_encoded=self.frames_encoded)

    def load_state_dict(self, state):
        """Restore a `state_dict()` of an actor with the same number of environments (`feats` in place: the forward's
        storage views read it)."""
        if len(state["env_ids"]) != self.E or tuple(state["feats"].shape) != tuple(self.feats.shape):
            raise ValueError(f"actor state of {len(state['env_ids'])} environments, this actor steps {self.E}")
        self.ticks, self.seed, self.frames_encoded = int(state["ticks"]), int(state["seed"]), int(state["frames_encoded"])
        self.env_ids = [int(i) for i in state["env_ids"]]
        self._env_ids_d.copy_(torch.tensor(self.env_ids, dtype=torch.int32))
        self.feats.copy_(state["feats"])
        self._last = list(state["last"])

    # ------------------------------------------------------------------ acting
    def act_batch(self, ticks):
        """One tick of all E environments. Returns (features [E,8,530], actions int64 [E,2], log_probs [E,2],
        values [E,2]) on the device; column 0 = steer, 1 = throttle. One Categorical draw per head for the whole
        batch (distributions.py:96-99 semantics, environment-major draw order)."""
        feats = self.encode(ticks)
        self._upload_commands(ticks)
        out = self._engine.evaluate([tuple(self._st)], [self._adv], self._idx, self.agent.owner.params)  # [2, E, 36]
        actions, log_probs = [], []
        for h, A in ((0, 33), (1, 3)):
            logits = out[h, :, 3:3 + A]                                   # normalised logits = log-probabilities
            a = torch.multinomial(F.softmax(logits, dim=-1), 1)           # [E,1]
            actions.append(a)
            log_probs.append(logits.gather(1, a))
        return feats, torch.cat(actions, 1), torch.cat(log_probs, 1), out[:, :, 0].t().contiguous()

    def _upload_commands(self, ticks, envs=None):
        for e, t in zip(range(self.E) if envs is None else envs, ticks):
            self._cmd_h[e, 0] = int(t["command"])
        cmd = self._cmd_h.to(self.device, non_blocking=True)
        for st in self._st:
            st.command.copy_(cmd)

    def act_into(self, ticks, pool):
        """One tick of all E environments written straight into `pool` (a RolloutPool with E workers) at its cursor:
        encoder batch, PPO forward, then one kernel that draws both heads' actions on the device and stores obs,
        action, log-prob, value, command and (below slot num_steps) hn / cn of all 2E storages; one device-to-host
        copy of the actions. Every storage's cursor advances like `RolloutStorage.insert`'s (modulo num_steps + 1).
        Rewards and masks follow with `pool.write_env_results`. Returns the actions, int64 [E, 2] (host)."""
        if pool.workers != self.E:
            raise ValueError(f"pool has {pool.workers} workers, the actor steps {self.E} environments")
        slot = pool.storages[0][0].step
        self.encode(ticks)
        self._upload_commands(ticks)
        self._engine.act([tuple(self._st)], [self._adv], self._idx, self.agent.owner.params, self._rows, pool.c_ref(),
                         slot, self.seed, self.ticks, self._env_ids_d, self.agent.hidden_state, self._act_d)
        self._act_h.copy_(self._act_d, non_blocking=True)
        torch.cuda.current_stream(self.device).synchronize()
        self.ticks += 1
        for pair in pool.storages:
            for st in pair:
                st.step = (st.step + 1) % (st.num_steps + 1)
        return self._act_h.numpy().copy()

    def bootstrap_into(self, pool, done):
        """pool.next_value [2W] = the bootstrap values of agent.get_value (train.py:76-79) for all W workers in one
        forward: each storage's obs[T] / command[T] (get_last reads slot T whatever the cursor is) and the agent's
        hidden_state; exactly 0 for a worker whose last tick was `done`. No host synchronisation."""
        W, T = pool.workers, pool.num_steps
        if len(done) != W:
            raise ValueError(f"done has {len(done)} entries for {W} workers")
        if self._boot is None or self._boot[0] is not pool:
            z = lambda *s: torch.zeros(*s, device=self.device)  # noqa: E731
            eng = _ppo.PpoEngine(W, 1, self.agent.clip, self.agent.value_coeff, self.agent.clip_coeff,
                                 self.agent.ent_coeff, self.device)
            hid = z(2, T + 1, self.F)                  # row T: the agent's hidden_state, read through index T
            zero = z(T + 1, 1)                         # advantages slot: read by the gather, unused by the forward
            sts = [tuple(SimpleNamespace(obs=st.obs, action=st.action, value_preds=st.value_preds, returns=st.returns,
                                         action_log_probs=st.action_log_probs, hn=hid[0], cn=hid[1], command=st.command)
                         for st in pair) for pair in pool.storages]
            self._boot = (pool, eng, hid, sts, [(zero, zero)] * W, [[[T], [T]] for _ in range(W)], z(2, W, _ppo.ROW_OUT))
        _, eng, hid, sts, advs, idx, rows = self._boot
        hid[0, T].copy_(self.agent.hidden_state[0].reshape(-1))
        hid[1, T].copy_(self.agent.hidden_state[1].reshape(-1))
        mask = sum(1 << w for w in range(W) if done[w])
        eng.bootstrap(sts, advs, idx, self.agent.owner.params, rows, mask, pool.next_value)
        return pool.next_value

    def act(self, ticks):
        """Reference-shaped results: per environment the 5-tuple of CadreAgent.act: (feature [8,530],
        [a_steer, a_throttle] 0-dim int64, [lp_s, lp_t] [1,1], [v_s, v_t] [1,1], hidden_state)."""
        feats, actions, log_probs, values = self.act_batch(ticks)
        a_cpu = actions.cpu()
        return [(feats[e].clone(), [a_cpu[e, 0], a_cpu[e, 1]],
                 [log_probs[e, 0].reshape(1, 1), log_probs[e, 1].reshape(1, 1)],
                 [values[e, 0].reshape(1, 1), values[e, 1].reshape(1, 1)], self.agent.hidden_state)
                for e in range(self.E)]
