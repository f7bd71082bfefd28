"""Evaluation with an ensemble of snapshots (reference: eval.py:18-63).

The reference loads `agent_num = len(load_episode)` agents from `<pretrained_path>/models/ppo_model_<episode>.pt`
(eval.py:45-51), lets every agent act on each observation, averages the continuous controls
(`CadreAgent.avg_action`, agent.py:83-95: mean of [steer, throttle, brake]; with more than one agent a mean brake
below 0.5 is released) and steps the environment with the averaged control (eval.py:53-63). The same loop, with the
environment passed in (the CARLA EnvWrapper when a simulator is available, `cadre_b200.synthetic_env.SyntheticEnv`
otherwise: both keep the tick_data contract of env_wrapper.py:857-918).

`load_agent_group` + `evaluate` are that loop as the reference runs it (one agent and encoder per snapshot, the full
8-frame window re-encoded by every agent every tick, torch's CPU Categorical, one environment). `DeviceEnsemble` +
`evaluate_envs` run it on the device: one encoder and frame cache for all snapshots (one new frame per environment
and tick), E environments per tick, K routed PPO forwards, and one kernel that draws every snapshot's actions with the
counter-based sampler and averages them into the controls (include/cadre_b200.h, cadre_ppo_ensemble_act)."""
import os

import numpy as np
import torch


def snapshot_path(pretrained_path, episode):
    """eval.py:49."""
    return os.path.join(pretrained_path, "models", "ppo_model_{}.pt".format(episode))


def load_agent_group(make_agent, pretrained_path, load_episode, device=None):
    """eval.py:45-51: one agent per entry of `load_episode`, each restored from its snapshot.
    `make_agent()` builds a fresh agent (e.g. `lambda: CadreAgent(**agent_cfg)`)."""
    group = []
    for ep in load_episode:
        agent = make_agent()
        agent.load_snapshot(snapshot_path(pretrained_path, ep), device)
        group.append(agent)
    return group


def evaluate(agent_group, env, eval_episode, max_steps=None):
    """eval.py:53-63. Returns one dict per episode: number of steps, summed [steer, throttle] rewards and the
    controls that were applied (the reference only prints where the env wrapper saved its own statistics)."""
    if not agent_group:
        raise ValueError("evaluate() needs at least one agent")
    out = []
    for _ in range(eval_episode):
        obs = env.reset()
        done = False
        steps, ret, controls = 0, [0.0, 0.0], []
        while not done and (max_steps is None or steps < max_steps):
            action_list = []
            for agent in agent_group:
                _, action, *_ = agent.act(obs)
                action_list.append(action)
            control = agent_group[-1].avg_action(action_list)      # eval.py:62 uses the loop's last `agent`
            obs, reward, done, info = env.step(control)
            steps += 1
            ret[0] += float(reward[0])
            ret[1] += float(reward[1])
            controls.append(control)
        out.append({"steps": steps, "return": ret, "controls": controls})
    return out


def load_snapshot_params(model_cfg, pretrained_path, load_episode):
    """One flat parameter tensor (fp32 [ppo_params.TOTAL] on model_cfg's device) per entry of `load_episode`, read from
    `<pretrained_path>/models/ppo_model_<episode>.pt` like `CadreAgent.load_snapshot` (the reference's own files and
    this package's). Only the PPO parameters are built: no encoder."""
    from .models import create_model, load_model_dict
    _, model_dict = create_model(model_cfg, load_vae=False)
    out = []
    for ep in load_episode:
        load_model_dict(model_dict, snapshot_path(pretrained_path, ep))
        out.append(model_dict.owner.params.clone())
    return out


class DeviceEnsemble:
    """K policy snapshots acting together on E environments (eval.py:53-63 for E environments at once).

    agent: a CadreAgent, whose encoder (and device) the ensemble uses; its own parameters are not used unless they are
    one of `params_list`. params_list: K flat fp32 parameter tensors on the agent's device (`load_snapshot_params`,
    `learner.params`, `agent.owner.params`), 1 <= K <= 64; they are read at every `act`, so a live tensor that is
    updated in place is seen by the next tick. Actions are drawn with the counter-based sampler keyed by (seed,
    env_ids[e], tick, snapshot index k), so snapshot 0 draws what `BatchedActor.act_into` draws for the same seed, env id
    and tick; `greedy=True` takes each head's most likely action instead."""

    def __init__(self, agent, params_list, num_envs, seed=0, env_ids=None, greedy=False):
        from . import ppo as _ppo
        from . import ppo_params
        from .actor import BatchedActor
        self.params = list(params_list)
        self.K = len(self.params)
        if not 1 <= self.K <= 64:
            raise ValueError(f"an ensemble holds 1 to 64 snapshots (got {self.K})")
        self.actor = BatchedActor(agent, num_envs, seed=seed, env_ids=env_ids)
        self.E, self.device = self.actor.E, self.actor.device
        for k, p in enumerate(self.params):
            _ppo._check_tensor(p, torch.float32, f"params_list[{k}]")
            if p.numel() != ppo_params.TOTAL or p.device != self.device:
                raise ValueError(f"params_list[{k}] must hold {ppo_params.TOTAL} floats on {self.device} "
                                 f"(got {p.numel()} on {p.device})")
        self.seed, self.env_ids, self.greedy = self.actor.seed, self.actor.env_ids, bool(greedy)
        self.ticks = 0                                    # act() calls so far: the sampler's tick counter
        self._steer = torch.tensor([float(agent.STEER_CONTROL[i]) for i in range(33)], dtype=torch.float64,
                                   device=self.device)
        self._throttle = torch.tensor([[float(v) for v in agent.THROTTLE_CONTROL[i]] for i in range(3)],
                                      dtype=torch.float64, device=self.device).reshape(-1)
        self._rows = torch.zeros(self.K, 2, self.E, _ppo.ROW_OUT, device=self.device)
        # controls fp64 [E, 3] and actions int64 [K, E, 2] in one buffer of 8-byte words: one device-to-host copy
        n_ctl = 3 * self.E
        self._out_d = torch.zeros(n_ctl + 2 * self.K * self.E, dtype=torch.int64, device=self.device)
        self._out_h = torch.empty_like(self._out_d, device="cpu").pin_memory()
        self._controls_d = self._out_d[:n_ctl].view(torch.float64).view(self.E, 3)
        self._actions_d = self._out_d[n_ctl:].view(self.K, self.E, 2)
        self.last_actions = None

    @property
    def frames_encoded(self):
        return self.actor.frames_encoded

    def reset(self, env_id):
        """Forget environment `env_id`'s frame window (call after its env.reset())."""
        self.actor.reset(env_id)

    def act(self, ticks, envs=None):
        """One tick of the environments `envs` (default: all E; `ticks` holds one tick_data per listed environment):
        their newest frames are encoded, all K snapshots act and their controls are averaged on the device. Returns
        the controls float64 [len(envs), 3] (host); `last_actions` holds every snapshot's actions, int64 [K, E, 2] (the
        rows of environments that were not listed are meaningless). One copy to the host and one synchronisation."""
        a = self.actor
        envs = a._env_list(ticks, envs)
        a.encode(ticks, envs)
        a._upload_commands(ticks, envs)
        a._engine.ensemble_act([tuple(a._st)], [a._adv], a._idx, self.params, self._rows, self.seed, self.ticks,
                               a._env_ids_d, self.greedy, self._steer, self._throttle, self._controls_d,
                               self._actions_d)
        self._out_h.copy_(self._out_d, non_blocking=True)
        torch.cuda.current_stream(self.device).synchronize()
        self.ticks += 1
        n_ctl = 3 * self.E
        out = self._out_h.numpy()
        self.last_actions = out[n_ctl:].reshape(self.K, self.E, 2).copy()
        return out[:n_ctl].view(np.float64).reshape(self.E, 3)[envs].copy()


def evaluate_envs(ensemble, envs, eval_episode, max_steps=None):
    """`evaluate` for E environments stepped together by a `DeviceEnsemble` (or anything with its `act(ticks, envs)` /
    `reset(e)`): every environment runs `eval_episode` episodes of at most `max_steps` steps. An environment that has
    finished its episodes is neither stepped nor passed to `act` again. Returns, per environment, the list of dicts
    `evaluate` returns (`steps`, `return`, `controls`)."""
    E = len(envs)
    results = [[] for _ in range(E)]
    obs, cur = [None] * E, [None] * E

    def begin(e):
        obs[e] = envs[e].reset()
        ensemble.reset(e)
        cur[e] = {"steps": 0, "return": [0.0, 0.0], "controls": []}

    def settle(e):
        """Close the episodes of env e that have reached max_steps; False once e has run all of its episodes."""
        while max_steps is not None and cur[e]["steps"] >= max_steps:
            results[e].append(cur[e])
            if len(results[e]) == eval_episode:
                return False
            begin(e)
        return True

    active = []
    if eval_episode > 0:
        for e in range(E):
            begin(e)
            if settle(e):
                active.append(e)
    while active:
        controls = ensemble.act([obs[e] for e in active], active)
        still = []
        for i, e in enumerate(active):
            control = [float(v) for v in controls[i]]
            obs[e], reward, done, info = envs[e].step(control)
            c = cur[e]
            c["steps"] += 1
            c["return"][0] += float(reward[0])
            c["return"][1] += float(reward[1])
            c["controls"].append(control)
            if done:
                results[e].append(c)
                if len(results[e]) == eval_episode:
                    continue
                begin(e)
            if settle(e):
                still.append(e)
        active = still
    return results


def main():
    """eval.py's main on the device path: CADRE_ENCODER_CKPT (the perception checkpoint, {'autoencoder': state_dict}),
    CADRE_CHECKPOINT_DIR (`pretrained_path`: snapshots under models/), CADRE_LOAD_EPISODE (e.g. 100,200,300),
    CADRE_EVAL_EPISODE (episodes per environment, default 1), CADRE_MAX_STEPS (optional step limit per episode),
    CADRE_GREEDY=1 (most likely actions instead of draws); env_cfg.num_processes SyntheticEnvs are evaluated together.
    Prints one line per episode."""
    from .agent import CadreAgent
    from .config import load_config
    from .synthetic_env import SyntheticEnv
    cfg = load_config(os.environ["CADRE_CONFIG"]) if os.environ.get("CADRE_CONFIG") else load_config()
    ckpt, pretrained = os.environ.get("CADRE_ENCODER_CKPT"), os.environ.get("CADRE_CHECKPOINT_DIR")
    episodes = [int(v) for v in os.environ.get("CADRE_LOAD_EPISODE", "").split(",") if v.strip()]
    if not ckpt or not pretrained or not episodes:
        raise SystemExit("set CADRE_ENCODER_CKPT (perception checkpoint), CADRE_CHECKPOINT_DIR (the training run's "
                         "checkpoint directory) and CADRE_LOAD_EPISODE (e.g. 100,200,300)")
    eval_episode = int(os.environ.get("CADRE_EVAL_EPISODE", 1))
    max_steps = int(os.environ["CADRE_MAX_STEPS"]) if os.environ.get("CADRE_MAX_STEPS") else None
    danet_state = torch.load(ckpt, map_location="cpu")["autoencoder"]
    agent = CadreAgent(**cfg.agent_cfg, danet_state=danet_state)
    params = load_snapshot_params(cfg.agent_cfg.model_cfg, pretrained, episodes)
    E = int(cfg.env_cfg.num_processes)
    envs = [SyntheticEnv(dict(cfg.env_cfg, rank=e)) for e in range(E)]
    ens = DeviceEnsemble(agent, params, E, seed=int(cfg.env_cfg.seed), greedy=os.environ.get("CADRE_GREEDY") == "1")
    print(f"ensemble of {len(episodes)} snapshots {episodes}, {E} environments, {eval_episode} episode(s) each",
          flush=True)
    for e, res in enumerate(evaluate_envs(ens, envs, eval_episode, max_steps)):
        for i, r in enumerate(res):
            print(f"env {e} episode {i}: steps {r['steps']} return steer {r['return'][0]:.4f} "
                  f"throttle {r['return'][1]:.4f}", flush=True)


if __name__ == "__main__":
    main()
