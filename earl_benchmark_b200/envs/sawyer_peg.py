"""Batched, device-resident `SawyerPegV2`.

Mirror of the reference class `earl_benchmark/envs/sawyer_peg.py:60-305` (constructor arguments `reward_type`,
`reset_at_goal`, `wide_init`; methods `reset`, `step`, `_get_obs`, `get_next_goal`, `reset_goal`, `compute_reward`,
`is_successful`) with a leading environment dimension on every array, on the same articulated-body engine as the door
task (envs/_sawyer_base.py, csrc/mj_*.cuh): Sawyer arm + two fingers + a free-joint peg (nq 16, nv 15) and a static
block with a hole; box-box contacts (peg on table, pads on peg, peg in hole), condim-4 finger pads.

The random draws of `reset_model()` (sawyer_peg.py:192-229) replicate the reference's global `np.random` stream bit for
bit, consumed in the order a Python loop over N reference envs would consume it: `get_next_goal()` (`randint`, which
consumes nothing when there is a single goal), then the peg position (`_get_state_rand_vec()` = 6 uniforms, redrawn
while within 0.1 of the block; or the wide / reset-at-goal variants).

Parity status (see DESIGN.md): the kernels match the fp64 checker to 5e-7 per step on this scene, but the checker
itself does NOT reproduce the shipped peg demonstrations (the grasp is lost), so results are pinned only at the level
of free-space hand motion.
"""
import os

import numpy as np

from .. import _lib, rng
from ._sawyer_base import ACT_DIM, MODEL_DIR, OBS_DIM, SawyerBatchedEnv  # noqa: F401

# reference module-level constants, earl_benchmark/envs/sawyer_peg.py:18-58
_HAND0 = [0.00615235, 0.6001898, 0.19430117, 1.0]
initial_states = np.array([_HAND0 + p for p in (
    [0.00313463, 0.68326396, 0.02], [-0.04035005, 0.67949003, 0.02], [0.02531051, 0.6074387, 0.02],
    [0.05957219, 0.6271171, 0.02], [-0.07566337, 0.62575287, 0.02], [-0.01177235, 0.55206996, 0.02],
    [0.02779735, 0.54707706, 0.02], [0.01835314, 0.5329686, 0.02], [0.02690855, 0.6263067, 0.02],
    [0.01766127, 0.59630984, 0.02], [0.0560186, 0.6634998, 0.02], [-0.03950658, 0.6323736, 0.02],
    [-0.03216827, 0.5247563, 0.02], [0.01265727, 0.69466716, 0.02], [0.05076993, 0.6025737, 0.02])])
goal_states = np.array([[0.0, 0.6, 0.2, 1.0, -0.3 + 0.03, 0.6, 0.0 + 0.13]])
# peg positions only
wide_initial_states = np.array([[-0.3, 0.8, 0.02], [-0.4, 0.8, 0.02], [-0.3, 0.9, 0.02], [-0.4, 0.9, 0.02],
                                [-0.2, 0.8, 0.02], [-0.2, 0.75, 0.02], [-0.2, 0.9, 0.02], [-0.1, 0.77, 0.02],
                                [0.0, 0.9, 0.02], [0.1, 0.8, 0.02], [0.15, 0.75, 0.02], [-0.3, 0.4, 0.02],
                                [-0.4, 0.4, 0.02], [-0.3, 0.45, 0.02], [-0.4, 0.45, 0.02], [-0.2, 0.4, 0.02],
                                [-0.2, 0.45, 0.02], [-0.2, 0.38, 0.02], [-0.1, 0.42, 0.02], [0.0, 0.45, 0.02],
                                [0.1, 0.36, 0.02], [0.15, 0.44, 0.02]])

MODEL_PATH = os.path.join(MODEL_DIR, "sawyer_peg.npz")
# _random_reset_space = Box(hstack(obj_low, goal_low), hstack(obj_high, goal_high)), sawyer_peg.py:64-69,102-105
_RESET_LOW = np.array([0.0, 0.5, 0.02, -0.35, 0.4, -0.001])
_RESET_HIGH = np.array([0.2, 0.7, 0.02, -0.25, 0.7, 0.001])


def reset_stream(seed, total_envs, env_offset, num_envs, rows, reset_at_goal=False, wide_init=False):
    """Goal rows int32 [rows, num_envs] and peg positions float64 [rows, num_envs, 3] of `rows` successive full resets: row e
    is what reset() of a handle without auto_reset draws at its e-th full reset (_draw_one over the global batch in env
    order on np.random.seed(seed), this shard's slice kept), replayed natively (rng.NumpyLegacyRandom.peg_reset_draws)."""
    r = rng.NumpyLegacyRandom(int(seed) & 0xFFFFFFFF)
    goal_rows = np.empty((rows, num_envs), np.int32)
    pos = np.empty((rows, num_envs, 3), np.float64)
    for e in range(rows):
        g, p = r.peg_reset_draws(total_envs, wide_init, reset_at_goal)
        goal_rows[e], pos[e] = g[env_offset:env_offset + num_envs], p[env_offset:env_offset + num_envs]
    return goal_rows, pos


def task_spec(model, max_newton=0):
    t = _lib.MjTask()
    t.frame_skip = 5
    t.hand_site = model.site_id("body:hand")
    t.ree_site = model.site_id("rightEndEffector")
    t.lee_site = model.site_id("leftEndEffector")
    t.obj_geom, t.obj_site = -1, model.site_id("pegHead")   # _get_pos_objects(): site 'pegHead' (sawyer_peg.py:186-187)
    t.max_newton = max_newton
    t.obj_qpos_count = 3                                    # _set_obj_xyz(pos): qpos[9:12] = pos, qvel[9:15] = 0
    t.mocap_low[:] = [-0.5, 0.40, 0.05]                     # hand_low / hand_high (sawyer_peg.py:66-67)
    t.mocap_high[:] = [0.5, 1.0, 0.5]
    t.action_scale = 1.0 / 100
    t.success_radius = 0.05                                 # TARGET_RADIUS (sawyer_peg.py:62,305)
    # dense reward (sawyer_peg.py:231-299): pegGrasp, the pad body frames of metaworld's _gripper_caging_reward and the four
    # corner sites of the block's two no-go prisms
    names = model.names["site"]
    sid = lambda n: names.index(n) if n in names else -1  # noqa: E731
    t.grasp_site, t.lpad_site, t.rpad_site = sid("pegGrasp"), sid("body:leftpad"), sid("body:rightpad")
    t.corner_site[:] = [sid("bottom_right_corner_collision_box_1"), sid("top_left_corner_collision_box_1"),
                        sid("bottom_right_corner_collision_box_2"), sid("top_left_corner_collision_box_2")]
    return t


class SawyerPegV2(SawyerBatchedEnv):
    ENV_KIND = _lib.ENV_SAWYER_PEG
    MODEL_FILE = "sawyer_peg.npz"
    SUCCESS_RADIUS = 0.05
    TARGET_RADIUS = 0.05
    HAS_DENSE_REWARD = True   # sawyer_peg.py:231-299 with metaworld's reward_utils / _gripper_caging_reward restated (unpinned)

    def __init__(self, reward_type="dense", reset_at_goal=False, wide_init=False, **batched):
        super().__init__(reward_type=reward_type, reset_at_goal=reset_at_goal, **batched)
        self.init_config = {"obj_init_pos": np.array([0, 0.6, 0.02]), "hand_init_pos": np.array([0, 0.6, 0.2])}
        self.initial_states = initial_states
        self.goal_states = goal_states
        self.wide_initial_states = wide_initial_states
        self.wide_init = bool(wide_init)
        self.random_init = True   # metaworld SawyerXYZEnv default: reset_model() samples the peg position
        self.obj_init_pos = self.init_config["obj_init_pos"]
        self.hand_init_pos = self.init_config["hand_init_pos"]
        self._goal_table = [goal_states[0].copy()] + [s.copy() for s in initial_states]
        self._pos_box = goal_states[0][4:] - np.array([0.03, 0.0, 0.13])   # compiled into the model (tools/compile_models.py)

    def _task_spec(self):
        return task_spec(self.model, self._max_newton)

    def _reset_stream(self, rows):
        g, p = reset_stream(self._seed, self._total_envs, self._env_offset, self.num_envs, rows, self._reset_at_goal, self.wide_init)
        return p, g

    # ------------------------------------------------------------------ the reference's draws, one env at a time
    def _rand_vec(self):  # _get_state_rand_vec(): np.random.uniform(low, high, size=6)
        return _RESET_LOW + (_RESET_HIGH - _RESET_LOW) * self._np_random.uniform(0.0, 1.0, 6)

    def _sample_peg(self):
        pos = self._rand_vec()[:3]
        while np.linalg.norm(pos[:2] - self._pos_box[:2]) < 0.1:
            pos = self._rand_vec()[:3]
        return pos

    def _draw_one(self):
        """(goal row, peg position) of one reset_model() call, consuming np.random exactly as sawyer_peg.py:192-229."""
        if not self._reset_at_goal:
            self._np_random.randint(self.goal_states.shape[0], 1)          # get_next_goal(): consumes nothing for n = 1
            row = 0
            pos = self.init_config["obj_init_pos"].copy()
            if self.wide_init:
                if self._np_random.uniform(0.0, 1.0, 1)[0] < 0.5:
                    pos = self._sample_peg()
                else:
                    k = int(self._np_random.randint(self.wide_initial_states.shape[0], 1)[0])
                    pos = self.wide_initial_states[k] - np.array([-0.1, 0.0, 0.0])
                    pos = pos + self._np_random.uniform(-0.02, 0.02, 3)
            elif self.random_init:
                pos = self._sample_peg()
        else:
            k = int(self._np_random.randint(self.initial_states.shape[0], 1)[0])
            row = 1 + k
            goal_pos = self.goal_states[0][4:] - np.array([-0.1, 0.0, 0.0])
            pos = goal_pos + self._np_random.uniform(-0.02, 0.02, 3)
        return row, pos

    def get_next_goal(self):  # sawyer_peg.py:144-152 (advances the np.random stream like the reference)
        if not self._reset_at_goal:
            self._np_random.randint(self.goal_states.shape[0], self.num_envs)
            return np.broadcast_to(self.goal_states[0], (self.num_envs, 7)).copy()
        k = self._np_random.randint(self.initial_states.shape[0], self.num_envs)
        return self.initial_states[k].copy()

    def compute_reward(self, obs, actions=None):
        """Sparse: on caller-supplied observations (cold path).  Dense: the reference's compute_reward reads simulator state
        (sites, pad bodies, init_tcp) besides `obs`, so it only exists for the states the step kernel produces."""
        if self._reward_type == "dense":
            raise NotImplementedError("SawyerPegV2: the dense reward is computed by step() (it needs simulator state, not only obs)")
        return super().compute_reward(obs, actions)

    def reset(self, mask=None, peg_pos=None):
        """reset() of every env (or those in `mask`); `peg_pos` [N,3] overrides the random draw.  On an auto_reset env the
        draw (goal row and peg position) is each reset env's next row of the pre-drawn reset stream."""
        self._ensure()
        m = self._mask(mask)
        if peg_pos is None and self._auto_reset:
            return self._reset_device(m, None)
        n = self.num_envs
        pos = np.tile(self.init_config["obj_init_pos"], (n, 1)).astype(np.float64)
        rows = self._goal_rows.cpu().numpy().copy()
        if peg_pos is not None:
            pos = np.broadcast_to(np.asarray(peg_pos, np.float64), (n, 3)).copy()
        else:
            sel = np.ones(n, bool) if m is None else m.cpu().numpy().astype(bool)
            # a sharded job draws for all envs of the global batch and keeps its slice, so results do not depend on
            # the number of GPUs
            lo = self._env_offset if m is None else 0
            total = self._total_envs if m is None else n
            for g in range(total):
                if m is not None and not sel[g]:
                    continue
                row, p = self._draw_one()
                if lo <= g < lo + n:
                    rows[g - lo], pos[g - lo] = row, p
        import torch
        self._goal_rows.copy_(torch.from_numpy(rows.astype(np.int32)))
        return self._reset_device(m, pos)
