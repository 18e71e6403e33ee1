"""oracle/tabletop3.py's Tabletop3Oracle with the three-object env's batched extras -- TEST INFRASTRUCTURE ONLY.

Adds what `TabletopManipulation(auto_reset=..., eval_stats=..., reset_stream_rows=...)` does on top of the reference
semantics the pinned oracle restates: the auto-reset of an env whose horizon fired (reset(mask=done) after the step),
the per-env episode statistics, and resets that take their qpos from a pre-drawn reset stream through a per-env cursor.
"""
import numpy as np

from oracle.tabletop3 import Tabletop3Oracle


class Tabletop3FeaturesOracle(Tabletop3Oracle):

    def __init__(self, num_envs, horizon, dense=False, auto_reset=False, reset_rows=None, **kw):
        super().__init__(num_envs, horizon, dense=dense, **kw)
        self.auto_reset = bool(auto_reset)
        self.reset_rows = None if reset_rows is None else np.asarray(reset_rows, np.float64)   # [R, N, 8]
        self.cursor = np.zeros(self.n, np.int64)
        self.ep_return = np.zeros(self.n, np.float64)
        self.success_last = np.zeros(self.n, bool)
        self.success_any = np.zeros(self.n, bool)

    def reset(self, mask=None, goal_rows=None, init_qpos=None):
        m = np.ones(self.n, bool) if mask is None else np.asarray(mask, bool)
        if init_qpos is None and self.reset_rows is not None:
            idx = np.flatnonzero(m)
            init_qpos = np.zeros((self.n, 8))
            init_qpos[idx] = self.reset_rows[self.cursor[idx] % len(self.reset_rows), idx]
            self.cursor[idx] += 1
        self.ep_return[m] = 0.0
        self.success_last[m] = False
        self.success_any[m] = False
        return super().reset(mask=m, goal_rows=goal_rows, init_qpos=init_qpos)

    def step(self, actions):
        """reward / done / success of the step that ended; the obs rows of auto-reset envs are post-reset"""
        o, rew, done, succ = super().step(actions)
        self.ep_return += rew.astype(np.float32).astype(np.float64)   # the device accumulates its fp32 reward
        self.success_last = succ.copy()
        self.success_any |= succ
        if self.auto_reset and done.any():
            o = self.reset(mask=done)
        return o, rew, done, succ

    def eval_stats(self):
        return np.array([self.ep_return.sum(), self.success_last.sum(), self.success_any.sum(), self.n], np.float64)
