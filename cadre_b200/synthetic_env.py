"""Synthetic stand-in for EnvWrapper (reference: env_wrapper.py:57, 581-690, 857-918): no simulator runs in the
box, so observations are seeded random tensors with the reference's `tick_data` contract:
  reset() -> tick_data;  step([steer, throttle, brake]) -> (tick_data, reward[2], done, {'action_done': [..]})
  tick_data = {'rgb': u8 [S,144,256,3], 'route_fig': u8 [S,256,144], 'measurements': f64 [S,3], 'command': int}
with an S-frame sliding history (the newest frame is appended each step, env_wrapper.py:900-914)."""
import numpy as np
import torch


class SyntheticEnv:
    def __init__(self, config=None, rank=0, seq_length=8, width=256, height=144, seed=0, done_prob=0.005,
                 action_done_prob=0.02):
        cfg = dict(config or {})
        self.rank = cfg.get("rank", rank)
        self.seq = cfg.get("seq_length", seq_length)
        self.w, self.h = cfg.get("width", width), cfg.get("height", height)
        self.done_prob = cfg.get("done_prob", done_prob)
        self.action_done_prob = cfg.get("action_done_prob", action_done_prob)
        self.rs = np.random.RandomState(cfg.get("seed", seed) + 1000 * self.rank)
        self.work_dir = cfg.get("root_path", "result")
        self._hist = None

    def _frame(self):
        rgb = self.rs.randint(0, 256, size=(self.h, self.w, 3)).astype(np.uint8)
        route = (self.rs.rand(self.w, self.h) < 0.1).astype(np.uint8) * 255
        meas = self.rs.rand(3)
        return rgb, route, meas

    def _tick(self):
        rgb, route, meas = zip(*self._hist)
        return {"rgb": np.array(rgb), "route_fig": np.array(route), "measurements": np.array(meas),
                "command": int(self.rs.randint(0, 4))}

    def reset(self):
        first = self._frame()
        self._hist = [first for _ in range(self.seq)]   # env_wrapper.py:680-688: history primed with frame 0
        return self._tick()

    def get_state(self):
        """What the next tick depends on: the generator state and the frame history (its frames are never modified in
        place, so the list is not copied)."""
        return {"rng": self.rs.get_state(), "hist": None if self._hist is None else list(self._hist)}

    def set_state(self, state):
        self.rs.set_state(state["rng"])
        self._hist = None if state["hist"] is None else list(state["hist"])

    def step(self, output_action):
        self._hist = self._hist[1:] + [self._frame()]
        reward = torch.tensor(self.rs.rand(2).astype(np.float32))
        done = bool(self.rs.rand() < self.done_prob)
        action_done = [bool(self.rs.rand() < self.action_done_prob) or done for _ in range(2)]
        return self._tick(), reward, done, {"action_done": action_done}
