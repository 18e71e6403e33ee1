"""Batched, device-resident mirror of the reference's Kitchen task (`earl_benchmark/envs/kitchen.py` over adept_envs
`KitchenV0` / `Robot_VelAct`): N independent Franka kitchens stepped by one kernel launch, one warp per environment
(`csrc/earl_mj_kitchen.cu`, C ABI `include/earl_mj_kitchen_b200.h`).

Per step (reference file:line, ADEPT/ = kitchen_assets/adept_envs/adept_envs/):
  action clip / scale, mocap update and clipping                   ADEPT/franka/kitchen_multitask_v0.py:91-102
  Robot_VelAct control from the LAST NOISY observation, ctrl[0:2]   ADEPT/franka/robot/franka_robot.py:172-207,255-264
  40 x mj_step (friction loss, joint equalities, pyramidal cones)   ADEPT/mujoco_env.py:148-153
  observation noise from env.np_random (gym 0.23.1: PCG64)          franka_robot.py:137-168, kitchen_multitask_v0.py:127-139
  dense reward, success                                             earl_benchmark/envs/kitchen.py:141-183
Batch semantics: environment i of the GLOBAL batch owns the stream PCG64(SeedSequence(seed + i)); the `np.random.randint(6)`
of reset_model is drawn from ONE legacy numpy stream `np.random.seed(seed)` in environment order (so num_envs = 1 consumes
exactly what the reference does).  Observations and rewards are float64 like the reference's; the physics state is float32.
The physics has no golden data in the reference (SURVEY.md 8c): parity of the engine is against this repo's fp64 checker.
"""
import copy
import ctypes as C
import os

import numpy as np
import torch

from .. import _lib, rng
from ..mjcf.compile import Model
from ..spaces import Box

MODEL_PATH = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "models", "kitchen.npz")
OBS_DIM, ACT_DIM, N_ROBOT, N_OBJ = 46, 9, 9, 14
_NEVER = (1 << 62)

# earl_benchmark/envs/kitchen.py:15-25
component_to_state_idx = {
    'arm': [0, 1, 2, 3, 4, 5, 6, 7, 8],
    'burner0': [9, 10],
    'burner1': [11, 12],
    'burner2': [13, 14],
    'burner3': [15, 16],
    'light_switch': [17, 18],
    'slide_cabinet': [19],
    'hinge_cabinet': [20, 21],
    'microwave': [22],
}
# :28-52
goal_states = np.array([[-4.1336253e-01, -1.6970085e+00, 1.4286385e+00, -2.5005307e+00, 6.2198675e-01, 1.2632011e+00, 8.8903642e-01,
                         4.3514766e-02, 7.9217982e-03, -5.1586074e-04, 4.8548312e-04, -5.4527864e-06, 6.3510129e-06, 6.0837720e-05,
                         -3.3861103e-05, 6.6394619e-05, -1.9801613e-05, -1.2477605e-04, 3.8065159e-04, -1.5148541e-04,
                         -9.2229841e-04, 7.2293887e-03, 6.9650509e-03]])
shaped_reward_tasks = ['microwave', 'light_switch', 'slide_cabinet', 'hinge_cabinet']


# :54-85 -- object configurations the reference resets to: the goal state with one or two components displaced
# (values from d4rl's kitchen_envs.py, as cited there)
_DISPLACED = {'microwave': [-0.7], 'light_switch': [-0.69, -0.05], 'slide_cabinet': [0.37], 'hinge_cabinet': [0., 1.45]}
_PAIR_NAMES = {'micro_hinge': ('microwave', 'hinge_cabinet'), 'micro_slide': ('microwave', 'slide_cabinet'),
               'micro_light': ('microwave', 'light_switch'), 'light_slide': ('light_switch', 'slide_cabinet'),
               'light_hinge': ('light_switch', 'hinge_cabinet'), 'slide_hinge': ('slide_cabinet', 'hinge_cabinet')}


def _displaced_state(*components):
    state = goal_states[0].copy()
    for name in components:
        state[component_to_state_idx[name]] = _DISPLACED[name]
    return state


initial_states = {name: _displaced_state(name) for name in _DISPLACED}
initial_states.update({key: _displaced_state(*pair) for key, pair in _PAIR_NAMES.items()})
initial_states['all_pairs'] = np.array([initial_states[key] for key in _PAIR_NAMES])   # order of kitchen.py:80-85

# ADEPT/franka/kitchen_multitask_v0.py:65-70
INIT_QPOS = np.array([1.48388023e-01, -1.76848573e+00, 1.84390296e+00, -2.47685760e+00, 2.60252026e-01, 7.12533105e-01,
                      1.59515394e+00, 4.79267505e-02, 3.71350919e-02, -2.66279850e-04, -5.18043486e-05, 3.12877220e-05,
                      -4.51199853e-05, -3.90842156e-06, -4.22629655e-05, 6.28065475e-05, 4.04984708e-05, 4.62730939e-04,
                      -2.26906415e-04, -4.65501369e-04, -6.44129196e-03, -1.77048263e-03, 1.08009684e-03])
MIDPOINT = np.array([-0.440, 0.1, 2.226])                                           # :44
MOCAP_LOW, MOCAP_HIGH = np.array([-0.7, -0.1, 1.8]), np.array([0.4, 0.5, 2.6])     # :47-48
FRAME_SKIP, NOISE_RATIO = 40, 0.1                                                   # :38, :41
# ADEPT/franka/robot/franka_config.xml:17-45
POS_BOUND = np.array([[-2.9, 2.9], [-1.8, 1.8], [-2.9, 2.9], [-3.1, 0.0], [-2.9, 2.9], [0.0, 3.8], [-2.9, 2.9], [0.0, 0.04], [0.0, 0.04]])
VEL_BOUND = np.array([[-10.0, 10.0]] * 9)
POS_NOISE_AMP = np.array([0.1] * 9 + [0.005] * 2 + [0.0005] * 6 + [0.005] * 3 + [0.1] * 3)
# earl_benchmark/envs/kitchen.py:149-156, in component_to_state_idx order (burner0..3, light_switch, slide, hinge, microwave)
REWARD_SITES = ("knob1_site", "knob2_site", "knob3_site", "knob4_site", "light_site", "slide_site", "hinge_site2", "microhandle_site")


class MjkConfig(C.Structure):   # earl_mjk_config (include/earl_mj_kitchen_b200.h)
    _fields_ = [("num_envs", C.c_int32), ("device", C.c_int32), ("flags", C.c_uint32), ("frame_skip", C.c_int32),
                ("episode_horizon", C.c_int64), ("goal_change_frequency", C.c_int64), ("goal", C.c_double * 23), ("init_qpos", C.c_double * 23),
                ("pos_noise_amp", C.c_double * 23), ("pos_bound", C.c_double * 18), ("vel_bound", C.c_double * 18),
                ("midpoint", C.c_double * 3), ("mocap_low", C.c_double * 3), ("mocap_high", C.c_double * 3),
                ("noise_ratio", C.c_double), ("site", C.c_int32 * 8)]


def pcg64_states(seeds):
    """[len(seeds), 4] uint64 = (state hi, state lo, inc hi, inc lo) of numpy's PCG64(SeedSequence(seed)): the stream gym
    0.23.1's seeding.np_random(seed) gives env.np_random (ADEPT/mujoco_env.py:113-118)."""
    out = np.empty((len(seeds), 4), np.uint64)
    m = (1 << 64) - 1
    for i, s in enumerate(seeds):
        st = np.random.PCG64(np.random.SeedSequence(None if s is None else int(s))).state["state"]
        out[i] = [st["state"] >> 64, st["state"] & m, st["inc"] >> 64, st["inc"] & m]
    return out


def reset_stream(seed, total_envs, env_offset, num_envs, rows, task='all_pairs'):
    """Initial configurations of `rows` successive full resets, (config uint8 [rows, num_envs], object-qpos table float64
    [K,14]): row e is what reset() of a handle without auto_reset draws at its e-th full reset (np.random.randint(6) per
    env of the global batch on np.random.seed(seed), this shard's slice kept).  Single-component tasks draw nothing: one
    table row, all-zero configs."""
    if task == 'all_pairs':
        table = initial_states['all_pairs'][:, 9:]
        r = rng.NumpyLegacyRandom(int(seed) & 0xFFFFFFFF)
        config = np.empty((rows, num_envs), np.uint8)
        for e in range(rows):
            config[e] = r.randint(table.shape[0], total_envs)[env_offset:env_offset + num_envs]
    else:
        table = initial_states[task][None, 9:]
        config = np.zeros((rows, num_envs), np.uint8)
    return config, np.ascontiguousarray(table, np.float64)


def _stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


class Kitchen:
    """N independent kitchens.  Mirrors the reference class surface: get_task, get_init_states, get_next_goal, reset_goal,
    reset, step, compute_reward, is_successful, seed."""
    max_path_length = int(1e8)

    def __init__(self, task="all_pairs", reward_type="dense", num_envs=1, device=None, seed=0, env_offset=0, total_envs=None,
                 model_path=None, auto_reset=False, reset_stream_rows=64, eval_stats=False, final_obs=False, **_unused):
        if final_obs and not auto_reset:
            raise ValueError("final_obs=True needs auto_reset=True: without it, the observation step() returns on done is the final one")
        if reward_type != 'dense':
            raise ValueError("Kitchen environment only supports dense rewards.")     # kitchen.py:91-92
        self._initial_states = copy.deepcopy(initial_states)
        self._goal_states = copy.deepcopy(goal_states)
        if task not in self._initial_states:
            raise KeyError(task)
        self._reward_type, self._task = reward_type, task
        self.num_envs, self._seed, self._env_offset = int(num_envs), int(seed), int(env_offset)
        self._total_envs = int(total_envs) if total_envs is not None else self.num_envs + self._env_offset
        if device is None:
            device = torch.cuda.current_device() if torch.cuda.is_available() else 0
        self.device = torch.device(device if not isinstance(device, int) else f"cuda:{device}")
        if self.device.type != "cuda":
            raise ValueError("earl_benchmark_b200 environments live on a CUDA device; there is no CPU path")
        self.model = Model.load(model_path or MODEL_PATH)
        self.goal = goal_states[0].copy()
        self.init_qpos = INIT_QPOS.copy()
        self.midpoint_pos = MIDPOINT.copy()
        self.action_space = Box(-1.0, 1.0, (ACT_DIM,), np.float32)
        self.observation_space = Box(-8.0, 8.0, (OBS_DIM,), np.float32)
        self.obs_dim = OBS_DIM
        self._episode_horizon, self._lifelong, self._goal_change_frequency = _NEVER, False, 0
        self._handle = None
        self._np_random = rng.NumpyLegacyRandom(self._seed & 0xFFFFFFFF)     # the global np.random of reset_model
        self._env_seed = self._seed
        # auto_reset=True: an env whose horizon fires is reset inside step() on the device, and every reset without
        # config_index takes its configuration from a pre-drawn stream of `reset_stream_rows` full resets (reset_stream())
        self._auto_reset, self._reset_stream_rows = bool(auto_reset), int(reset_stream_rows)
        if self._reset_stream_rows < 1:
            raise ValueError("reset_stream_rows must be >= 1")
        # eval_stats=True: every env keeps its episode return and success on the device, reduced by eval_stats()
        self._eval_stats = bool(eval_stats)
        # final_obs=True (with auto_reset): every step's info["final_observation"] holds the last observation of each
        # episode the step ended (see step())
        self._keep_final_obs = bool(final_obs)
        self._final_obs = None

    # ------------------------------------------------------------------ reference surface
    def get_task(self):
        return self._task

    def get_init_states(self):
        return self._initial_states['all_pairs']

    def get_next_goal(self):
        return self._goal_states[0]

    def reset_goal(self, goal=None):
        if goal is not None and not np.array_equal(np.asarray(goal, np.float64).reshape(23), self._goal_states[0]):
            raise NotImplementedError("Kitchen: custom goals are not built (the reference only ever sets goal_states[0])")

    def seed(self, seed=None):
        """env.seed(seed): environment i (global index) gets PCG64(SeedSequence(seed + i)); seed None = OS entropy."""
        self._env_seed = seed
        self._ensure()
        seeds = [None if seed is None else int(seed) + self._env_offset + i for i in range(self.num_envs)]
        st = np.ascontiguousarray(pcg64_states(seeds))
        _lib.check(_lib.lib().earl_mjk_seed(self._handle, st.ctypes.data))
        return [seed]

    # ------------------------------------------------------------------ construction
    def _configure(self, episode_horizon=None, lifelong=None, goal_change_frequency=None):
        if self._handle is not None:
            raise RuntimeError("wrappers must be applied before the env is first reset/stepped")
        if episode_horizon is not None:
            self._episode_horizon = int(episode_horizon)
        if lifelong is not None:
            self._lifelong = bool(lifelong)      # one goal: the periodic reset_goal() changes nothing, but the _get_obs() that
            # follows it draws a second noisy observation (lifelong_wrapper.py:36-42): done in the step kernel
        if goal_change_frequency is not None:
            self._goal_change_frequency = int(goal_change_frequency)

    def _ensure(self):
        if self._handle is not None:
            return
        cfg = MjkConfig()
        cfg.num_envs, cfg.device, cfg.frame_skip = self.num_envs, self.device.index or 0, FRAME_SKIP
        cfg.flags = (_lib.FLAG_LIFELONG if self._lifelong else 0) | (_lib.FLAG_AUTO_RESET if self._auto_reset else 0) | \
            (_lib.FLAG_EVAL_STATS if self._eval_stats else 0) | (_lib.FLAG_FINAL_OBS if self._keep_final_obs else 0)
        cfg.episode_horizon = self._episode_horizon
        cfg.goal_change_frequency = self._goal_change_frequency if self._lifelong else 0
        cfg.goal[:] = self.goal.tolist()
        cfg.init_qpos[:] = self.init_qpos.tolist()
        cfg.pos_noise_amp[:] = POS_NOISE_AMP.tolist()
        cfg.pos_bound[:] = POS_BOUND.reshape(-1).tolist()
        cfg.vel_bound[:] = VEL_BOUND.reshape(-1).tolist()
        cfg.midpoint[:], cfg.mocap_low[:], cfg.mocap_high[:] = MIDPOINT.tolist(), MOCAP_LOW.tolist(), MOCAP_HIGH.tolist()
        cfg.noise_ratio = NOISE_RATIO
        cfg.site[:] = [self.model.site_id(s) for s in REWARD_SITES]
        blob = self.model.to_blob()
        h = C.c_void_p()
        _lib.check(_lib.lib().earl_mjk_create(C.byref(cfg), blob, len(blob), C.byref(h)))
        self._handle = h
        n, dev = self.num_envs, self.device
        self._obs = torch.empty((n, OBS_DIM), dtype=torch.float64, device=dev)
        self._reward = torch.empty((n,), dtype=torch.float64, device=dev)
        self._done = torch.empty((n,), dtype=torch.uint8, device=dev)
        self._success = torch.empty((n,), dtype=torch.uint8, device=dev)
        if self._keep_final_obs:   # rows of envs that have not ended an episode yet hold NaN
            self._final_obs = torch.full((n, OBS_DIM), float("nan"), dtype=torch.float64, device=dev)
            _lib.check(_lib.lib().earl_mjk_set_final_obs(h, self._final_obs.data_ptr()))
        self.seed(self._env_seed)
        if self._auto_reset:
            config, table = reset_stream(self._seed, self._total_envs, self._env_offset, n, self._reset_stream_rows, self._task)
            config = np.ascontiguousarray(config)
            _lib.check(_lib.lib().earl_mjk_set_reset_stream(h, config.ctypes.data, self._reset_stream_rows, table.ctypes.data,
                                                            len(table)))

    def close(self):
        if self._handle is not None:
            _lib.lib().earl_mjk_destroy(self._handle)
            self._handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ------------------------------------------------------------------ reset / step
    def _draw_configs(self, count):
        """reset_model's np.random.randint(6) per environment, in environment order (kitchen.py:122-124)."""
        if self._task == 'all_pairs':
            k = self._initial_states['all_pairs'].shape[0]
            if count == self.num_envs:   # full reset: every shard consumes the global stream and keeps its slice (SURVEY 8e)
                idx = self._np_random.randint(k, self._total_envs)[self._env_offset:self._env_offset + self.num_envs]
            else:
                idx = self._np_random.randint(k, count)
            return self._initial_states['all_pairs'][idx, 9:], idx
        return np.tile(self._initial_states[self._task][9:], (count, 1)), np.zeros(count, np.int32)

    def reset(self, mask=None, config_index=None):
        """reset() of every env (or those in `mask`); `config_index` [count] overrides the random draw.  Returns the
        observation float64 [N,46] of all environments (rows of environments that were not reset hold their last one).
        On an auto_reset env the draw is each reset env's next entry of the pre-drawn reset stream, made on the device, and
        last_config_index is None."""
        self._ensure()
        if mask is None:
            ids, count = None, self.num_envs
        else:
            ids = torch.nonzero(torch.as_tensor(mask, device=self.device).reshape(-1)).to(torch.int32).reshape(-1).contiguous()
            count = int(ids.numel())
            if count == 0:
                return self._obs
        o = None
        if config_index is None and self._auto_reset:
            self.last_config_index = None
        else:
            if config_index is None:
                objs, self.last_config_index = self._draw_configs(count)
            else:
                self.last_config_index = np.asarray(config_index, np.int64).reshape(count)
                objs = self._initial_states['all_pairs'][self.last_config_index, 9:]
            o = torch.as_tensor(np.array(objs, np.float64, order="C", copy=True)).to(self.device)
        out = torch.empty((count, OBS_DIM), dtype=torch.float64, device=self.device)
        _lib.check(_lib.lib().earl_mjk_reset(self._handle, None if ids is None else ids.data_ptr(), count,
                                             None if o is None else o.data_ptr(), out.data_ptr(), _stream()))
        if ids is None:
            self._obs.copy_(out)
        else:
            self._obs[ids.long()] = out
        return self._obs

    def step(self, action, b=None):
        """CUDA float32 tensor [N,9] -> CUDA tensors (obs float64 [N,46], reward float64 [N], done bool [N], info); numpy
        in -> numpy out (copies through the device).  final_obs=True envs add info["final_observation"] float64 [N,46]:
        on rows where done is set, the observation the step reached before the auto-reset replaced it; other rows keep
        what an earlier step stored there (NaN before an env's first episode ends).  The env-owned tensor, valid until
        the next step; a numpy copy for numpy input."""
        self._ensure()
        host = not (isinstance(action, torch.Tensor) and action.is_cuda)
        a = torch.as_tensor(np.asarray(action, np.float32)).to(self.device) if host else action
        if a.dtype != torch.float32 or not a.is_contiguous():
            a = a.to(torch.float32).contiguous()
        if a.numel() != self.num_envs * ACT_DIM:
            raise ValueError(f"action must have shape [{self.num_envs},{ACT_DIM}]")
        _lib.check(_lib.lib().earl_mjk_step(self._handle, a.data_ptr(), self._obs.data_ptr(), self._reward.data_ptr(),
                                            self._done.data_ptr(), self._success.data_ptr(), _stream()))
        info = {"success": self._success.view(torch.bool)}
        if self._final_obs is not None:
            info["final_observation"] = self._final_obs
        if host:
            return self._obs.cpu().numpy(), self._reward.cpu().numpy(), self._done.cpu().numpy().view(np.bool_), \
                {k: v.cpu().numpy().view(np.bool_) if k == "success" else v.cpu().numpy() for k, v in info.items()}
        return self._obs, self._reward, self._done.view(torch.bool), info

    def _get_obs(self):
        return self._obs

    # ------------------------------------------------------------------ reward / success on caller-supplied observations
    def is_successful(self, obs=None):
        """||obs[9:23] - obs[32:46]|| <= 0.3 (kitchen.py:181-183)."""
        o = self._obs if obs is None else obs
        if isinstance(o, torch.Tensor):
            o = o.reshape(-1, OBS_DIM)
            return torch.linalg.norm(o[:, 9:23] - o[:, 32:46], dim=1) <= 0.3
        o = np.asarray(o).reshape(-1, OBS_DIM)
        return np.linalg.norm(o[:, 9:23] - o[:, 32:46], axis=1) <= 0.3

    def compute_reward(self, obs):
        """Kitchen._get_reward_n_score (kitchen.py:141-175) on caller-supplied observations [M,46] with the CURRENT mocap and
        site positions of the first M environments (cold path, numpy; the step kernel evaluates the same expressions)."""
        o = (obs.detach().cpu().numpy() if isinstance(obs, torch.Tensor) else np.asarray(obs)).reshape(-1, OBS_DIM)
        st = self.get_state()
        out = np.empty(len(o))
        keys = [k for k in component_to_state_idx if k != 'arm']
        for i, ob in enumerate(o):
            r = -10 * np.linalg.norm(ob[9:23] - ob[32:46])
            reaching = False
            for c, key in enumerate(keys):
                cur = np.array(component_to_state_idx[key])
                if np.linalg.norm(ob[cur] - ob[cur + 23]) < len(cur) * 0.01:
                    r += 1
                elif not reaching:
                    reaching = True
                    r += -0.5 * np.linalg.norm(st["mocap_pos"][i] - st["site_xpos"][i, c])
            out[i] = r
        return out

    # ------------------------------------------------------------------ counters / state
    def _counters(self, want_ll=False):
        self._ensure()
        total = C.c_int64()
        n = self.num_envs
        interv = torch.empty((n,), dtype=torch.int64, device=self.device)
        since = torch.empty((n,), dtype=torch.int32, device=self.device)
        ll = torch.empty((n,), dtype=torch.float64, device=self.device) if want_ll else None
        _lib.check(_lib.lib().earl_mjk_counters(self._handle, C.byref(total), interv.data_ptr(), since.data_ptr(),
                                                None if ll is None else ll.data_ptr(), _stream()))
        return total.value, interv, since, ll

    def eval_stats(self):
        """float64 CUDA tensor [4] = (sum of episode returns, #envs successful at their last step, #envs successful at any
        step of the episode, N), reduced on the device in the current stream; needs eval_stats=True.  A reset clears an
        env's statistics.  Sum it over shards with distributed.all_reduce_eval_stats."""
        self._ensure()
        out = torch.empty((4,), dtype=torch.float64, device=self.device)
        _lib.check(_lib.lib().earl_mjk_eval_stats(self._handle, out.data_ptr(), _stream()))
        return out

    def work_counters(self):
        self._ensure()
        out = np.zeros(7, np.uint64)
        _lib.check(_lib.lib().earl_mjk_work_counters(self._handle, out.ctypes.data))
        d = dict(zip(("env_steps", "substeps", "newton_iterations", "constraint_rows", "contacts", "bad_states", "overflow_states"),
                     (int(x) for x in out)))
        d["redone_states"] = int(_lib.lib().earl_mjk_redo_count(self._handle))
        return d

    def get_state(self):
        """dict(qpos, qvel, qacc_warmstart [N,23], mocap_pos [N,3], last_noisy_qp [N,9], site_xpos [N,8,3]) as host arrays."""
        self._ensure()
        n = self.num_envs
        q, v, w, mp, lq, st = np.zeros((n, 23)), np.zeros((n, 23)), np.zeros((n, 23)), np.zeros((n, 3)), np.zeros((n, 9)), np.zeros((n, 8, 3))
        _lib.check(_lib.lib().earl_mjk_get_state(self._handle, q.ctypes.data, v.ctypes.data, w.ctypes.data, mp.ctypes.data,
                                                 lq.ctypes.data, st.ctypes.data))
        return dict(qpos=q, qvel=v, qacc_warmstart=w, mocap_pos=mp, last_noisy_qp=lq, site_xpos=st)

    def set_state(self, qpos=None, qvel=None, qacc_warmstart=None, mocap_pos=None, last_noisy_qp=None):
        self._ensure()
        p = lambda a, sh: None if a is None else np.ascontiguousarray(np.asarray(a, np.float64).reshape(sh))  # noqa: E731
        n = self.num_envs
        arrs = [p(qpos, (n, 23)), p(qvel, (n, 23)), p(qacc_warmstart, (n, 23)), p(mocap_pos, (n, 3)), p(last_noisy_qp, (n, 9))]
        _lib.check(_lib.lib().earl_mjk_set_state(self._handle, *[None if a is None else a.ctypes.data for a in arrs]))
