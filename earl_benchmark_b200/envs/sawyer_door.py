"""Batched, device-resident `SawyerDoorV2`.

Mirror of the reference class `earl_benchmark/envs/sawyer_door.py:18-177` (constructor arguments `reward_type`,
`reset_at_goal`; methods `reset`, `step`, `_get_obs`, `get_next_goal`, `reset_goal`, `compute_reward`,
`is_successful`) with a leading environment dimension on every array.  The reference inherits `step()` from
metaworld's SawyerXYZEnv, which calls MuJoCo 2.1.0 through mujoco-py (5 x `sim.step()` per env step); here the
whole step -- mocap update, 5 engine substeps, observation, sparse reward, reset-free horizon bookkeeping -- is
one CUDA kernel launch with one warp per environment (csrc/mj_*.cuh) behind the C ABI of
include/earl_mj_b200.h (machinery shared with the peg task: envs/_sawyer_base.py).  Without the CUDA library or a
CUDA device this class raises; there is no CPU path.

The MJCF is compiled once on the host (mjcf/parser.py, mjcf/compile.py, tools/compile_models.py) into the
structure-of-arrays model file `models/sawyer_door.npz` that ships with the package.

Caller-visible differences from the reference:
  * every array has a leading [N] dimension; observations are float32 (the reference returns float64);
  * `reward_type='dense'` is not built (raises NotImplementedError);
  * `sim.reset()` + `_reset_hand()` is deterministic, so it is simulated once on the device and every later reset
    copies that state; the door-angle noise comes from a bit-exact replica of `np.random.seed(seed)` consumed in
    the order a Python loop over N reference envs would consume it.
"""
import os

import numpy as np

from .. import _lib, rng
from ._sawyer_base import ACT_DIM, MODEL_DIR, OBS_DIM, SawyerBatchedEnv  # noqa: F401

# reference module-level constants, earl_benchmark/envs/sawyer_door.py:13-16
initial_states = np.array([[0.00591636, 0.39968333, 0.19493164, 1.0,
                            0.01007495, 0.47104556, 0.10003595]])
goal_states = np.array([[0.29072163, 0.74286009, 0.10003595, 1.0,
                         0.29072163, 0.74286009, 0.10003595]])

MODEL_PATH = os.path.join(MODEL_DIR, "sawyer_door.npz")


def _angle_range(reset_at_goal):
    """(obj_init_angle, uniform low, uniform high) of reset_model(), sawyer_door.py:33,114-118"""
    return (0.0, -np.pi / 20, 0.0) if reset_at_goal else (-np.pi / 3, 0.0, np.pi / 20)


def reset_stream(seed, total_envs, env_offset, num_envs, rows, reset_at_goal=False):
    """Door angles of `rows` successive full resets, float64 [rows, num_envs, 1]: row e is what reset() of a handle
    without auto_reset draws at its e-th full reset (np.random.seed(seed), one uniform per env of the global batch,
    this shard's slice kept)."""
    angle0, lo, hi = _angle_range(reset_at_goal)
    r = rng.NumpyLegacyRandom(int(seed) & 0xFFFFFFFF)
    out = np.empty((rows, num_envs, 1), np.float64)
    for e in range(rows):
        out[e, :, 0] = np.full(num_envs, float(angle0)) + r.uniform(lo, hi, total_envs)[env_offset:env_offset + num_envs]
    return out


def task_spec(model, max_newton=0, hand_init_pos=(0.0, 0.4, 0.2)):
    """Constants of metaworld's SawyerXYZEnv / SawyerDoorEnvV2 and of sawyer_door.py that are not in the MJCF."""
    t = _lib.MjTask()
    t.frame_skip = 5                                  # SawyerXYZEnv frame_skip
    t.hand_site = model.site_id("body:hand")          # get_endeff_pos(): xpos of body 'hand'
    t.ree_site = model.site_id("rightEndEffector")
    t.lee_site = model.site_id("leftEndEffector")
    t.obj_geom, t.obj_site = model.geom_id("handle"), -1   # _get_pos_objects(): geom 'handle'
    t.max_newton = max_newton
    t.obj_qpos_count = 1                              # _set_obj_xyz(angle): the door hinge
    t.mocap_low[:] = [-0.5, 0.40, 0.05]               # hand_low / hand_high (sawyer_door.py:25-26)
    t.mocap_high[:] = [0.5, 1.0, 0.5]
    t.action_scale = 1.0 / 100
    t.success_radius = 0.02                           # is_successful(), sawyer_door.py:177
    t.obj_init_pos[:] = [0.1, 0.95, 0.1]              # dense reward margins (sawyer_door.py:36,150,156); float32 in the reference
    t.hand_init_pos[:] = [float(x) for x in hand_init_pos]
    t.grasp_site = t.lpad_site = t.rpad_site = -1
    t.corner_site[:] = [-1] * 4
    return t


class SawyerDoorV2(SawyerBatchedEnv):
    ENV_KIND = _lib.ENV_SAWYER_DOOR
    MODEL_FILE = "sawyer_door.npz"
    SUCCESS_RADIUS = 0.02
    HAS_DENSE_REWARD = True

    def __init__(self, reward_type="sparse", reset_at_goal=False, **batched):
        super().__init__(reward_type=reward_type, reset_at_goal=reset_at_goal, **batched)
        # reference attributes (sawyer_door.py:32-58)
        self.init_config = {
            "obj_init_angle": -np.pi / 3 if not self._reset_at_goal else 0,
            "obj_init_pos": np.array([0.1, 0.95, 0.1], dtype=np.float32),
            "hand_init_pos": np.array([0, 0.4, 0.2] if not self._reset_at_goal else [0.29, 0.74, 0.1], dtype=np.float32),
        }
        self.goal_states = goal_states.copy()
        self.obj_init_angle = self.init_config["obj_init_angle"]
        self.hand_init_pos = self.init_config["hand_init_pos"]
        self._goal_table = [goal_states[0].copy(), initial_states[0].copy()]

    def _task_spec(self):
        return task_spec(self.model, self._max_newton, self.hand_init_pos)

    def compute_reward(self, obs, actions=None):
        """compute_reward(obs)[0] of the reference (sawyer_door.py:141-171) on caller-supplied observations [M,14]
        (cold path, numpy / torch on the caller's device; the step kernel evaluates the same expressions in fp32)."""
        if self._reward_type == "sparse":
            return super().compute_reward(obs, actions)
        xp = __import__("torch") if not isinstance(obs, np.ndarray) else np
        o = obs.reshape(-1, OBS_DIM)
        norm = (lambda v: xp.linalg.norm(v, dim=1)) if xp is not np else (lambda v: np.linalg.norm(v, axis=1))
        tcp, obj, target = o[:, :3], o[:, 4:7], o[:, 11:14]
        to = lambda c: (xp.as_tensor(np.asarray(c, np.float32), device=o.device) if xp is not np else np.asarray(c, np.float64))  # noqa: E731
        d_to, d_ot = norm(tcp - obj), norm(obj - target)

        def tol(x, upper, margin):
            d = (x - upper) / margin
            v = xp.exp(-0.5 * d * d * 4.605170185988092)
            return xp.where(x <= upper, xp.ones_like(v), v)
        in_place = tol(d_ot, 0.05, norm(to(self.init_config["obj_init_pos"])[None, :] - target))
        hand = tol(d_to, 0.0125, norm(to(self.hand_init_pos)[None, :] - obj) + 0.1)
        r = 3 * hand + 6 * in_place
        return xp.where(d_ot < 0.05, xp.full_like(r, 10.0), r)

    def get_next_goal(self):  # sawyer_door.py:96-98
        return np.broadcast_to(self.goal_states[0], (self.num_envs, 7)).copy()

    def _reset_stream(self, rows):
        return reset_stream(self._seed, self._total_envs, self._env_offset, self.num_envs, rows, self._reset_at_goal), None

    def _draw_angles(self, mask):
        """obj_init_angle + np.random.uniform(0, pi/20)  (or (-pi/20, 0) when reset_at_goal), sawyer_door.py:114-118;
        one draw per reset env, in env order."""
        _, lo, hi = _angle_range(self._reset_at_goal)
        ang = np.full(self.num_envs, float(self.obj_init_angle))
        if mask is None:
            u = self._np_random.uniform(lo, hi, self._total_envs)[self._env_offset:self._env_offset + self.num_envs]
            return ang + u
        sel = mask.cpu().numpy().astype(bool)
        ang[sel] += self._np_random.uniform(lo, hi, int(sel.sum()))
        return ang

    def reset(self, mask=None, door_angle=None):
        """reset() of every env (or those in `mask`); `door_angle` [N] overrides the random draw.  On an auto_reset env the
        draw is each reset env's next row of the pre-drawn reset stream."""
        self._ensure()
        m = self._mask(mask)
        if door_angle is None and self._auto_reset:
            return self._reset_device(m, None)
        ang = self._draw_angles(m) if door_angle is None else np.broadcast_to(np.asarray(door_angle, np.float64), (self.num_envs,))
        return self._reset_device(m, np.asarray(ang, np.float64).reshape(self.num_envs, 1))
