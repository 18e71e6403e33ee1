"""Batched, device-resident `TabletopManipulation`.

Mirror of the reference class `earl_benchmark/envs/tabletop_manipulation.py:18-204` (same constructor
arguments, method names and semantics) with a leading environment dimension on every array.  All
arithmetic runs in the CUDA library (csrc/tabletop_kernels.cuh) through the C ABI; this file only
owns buffers and argument marshalling.  Without the CUDA library or a CUDA device it raises.

Differences from the reference that a caller can observe:
  * every array has a leading [N] dimension (N = num_envs), rewards / dones are arrays;
  * gym's constructor-time random `step()` (SURVEY.md App. A #1) is not replayed: call reset() first;
  * goals are rows of a goal table (the four `goal_states` + `initial_states[0]`, custom goals appended);
  * goal draws come from a per-env pre-drawn stream that replicates `random.seed(seed)` bit for bit in
    the order a Python loop over N reference envs would consume it (rng.py, include/earl_b200.h).
"""
import ctypes as C

import numpy as np
import torch

from .. import _lib, rng
from . import _hostio
from ._goals import goal_args
from ._hostio import HostBuffers
from ..spaces import Box

# reference module-level constants, earl_benchmark/envs/tabletop_manipulation.py:11-16
initial_states = np.array([[0.0, 0.0, 2.5, 0.0, -1., -1.]])
goal_states = np.array([[0.0, 0.0, -2.5, -1.0, -1., -1.],
                        [0.0, 0.0, -2.5, 1.0, -1., -1.],
                        [0.0, 0.0, 0.0, 2.0, -1., -1.],
                        [0.0, 0.0, 0.0, -2.0, -1., -1.],
                        ])

OBS_DIM, ACT_DIM = 12, 3
_NEVER = 1 << 62


def _ptr(t):
    return 0 if t is None else t.data_ptr()


def _stream():
    return torch.cuda.current_stream().cuda_stream


class TabletopManipulation:
    """N independent tabletop envs stepped by one kernel launch.

    Reference-compatible arguments: task_list, reward_type, reset_at_goal, wide_init_distr
    (tabletop_manipulation.py:24-28).  Batched extras: num_envs, device, seed, state_dtype ('float32' |
    'float64'), goal_stream_rows, auto_reset, eval_stats, env_offset/total_envs (this shard's slice of a
    larger job: the goal stream is drawn for `total_envs` envs and columns [env_offset, env_offset+N) kept),
    per_env_goals (every env keeps its own goal vector: set_goals() / get_goals()), final_obs (with auto_reset: every
    step's info["final_observation"] holds the last observation of each episode the step ended, see step()).
    """

    def __init__(self, task_list="rc_r-rc_k-rc_g-rc_b", reward_type="dense", reset_at_goal=False,
                 wide_init_distr=False, num_envs=1, device=None, seed=0, state_dtype="float32",
                 goal_stream_rows=64, auto_reset=False, eval_stats=False, env_offset=0, total_envs=None, host_io=False,
                 per_env_goals=False, final_obs=False):
        if final_obs and not auto_reset:
            raise ValueError("final_obs=True needs auto_reset=True: without it, the observation step() returns on done is the final one")
        if reward_type not in ("sparse", "dense"):
            raise ValueError(f"reward_type must be 'sparse' or 'dense', got {reward_type!r}")
        if state_dtype not in ("float32", "float64"):
            raise ValueError("state_dtype must be 'float32' or 'float64'")
        self._task_list = task_list
        self._reward_type = reward_type
        self._reset_at_goal = bool(reset_at_goal)
        self._wide_init_distr = bool(wide_init_distr)
        self.num_envs = int(num_envs)
        self._seed = int(seed)
        self._state_dtype = state_dtype
        self._goal_stream_rows = int(goal_stream_rows)
        self._auto_reset = bool(auto_reset)
        self._eval_stats = bool(eval_stats)
        self._per_env_goals = bool(per_env_goals)
        self._keep_final_obs = bool(final_obs)
        self._env_offset = int(env_offset)
        self._total_envs = int(total_envs) if total_envs is not None else self.num_envs + self._env_offset
        if device is None:
            device = torch.cuda.current_device() if torch.cuda.is_available() else 0
        self.device = torch.device(device if not isinstance(device, int) else f"cuda:{device}")
        if self.device.type != "cuda":
            raise ValueError("earl_benchmark_b200 environments live on a CUDA device; there is no CPU path")

        # reference attributes
        self.threshold = 0.4
        self.move_distance = 0.2
        self.initial_state = initial_states.copy()[0]
        self._goal_list = goal_states.copy()
        self.target_colors = ["r", "g", "b", "k"]
        self.action_space = Box(-1.0, 1.0, (ACT_DIM,), np.float32)
        self.observation_space = Box(-np.inf, np.inf, (OBS_DIM,), np.float32)

        # goal table: rows 0..3 = goal_states-derived goals, row 4 = the initial state (reverse demos)
        self._goal_table = [self._make_goal(r) for r in range(len(goal_states))] + [self.initial_state.copy()]
        self._task_to_row = self._parse_task_list(task_list)

        # wrapper configuration (set by PersistentStateWrapper / LifelongWrapper before first use)
        self._episode_horizon = _NEVER
        self._lifelong = False
        self._goal_change_frequency = 0
        self._handle = None
        self._np_random = rng.NumpyLegacyRandom(self._seed & 0xFFFFFFFF)  # np.random stream (wide-init resets)
        self._obs = self._reward = self._done = self._success = self._final_obs = None
        self._host_bufs = None
        self._host_mode = bool(host_io)   # host_io=True: reset() returns numpy like the numpy-driven step()

    # ------------------------------------------------------------------ construction helpers
    def _make_goal(self, row):
        g = self.initial_state.copy()
        g[2:4] = self._goal_list[row][2:4]  # get_next_goal(), tabletop_manipulation.py:62-76
        return g

    def _parse_task_list(self, task_list):
        rows = []
        for task in task_list.split("-"):
            parts = task.split("__")
            if len(parts) != 1 or parts[0][:2] != "rc":
                raise ValueError(f"unsupported task {task!r}: the single-object env only has the red cube ('rc_*')")
            rows.append(self.target_colors.index(parts[0].split("_")[1]))
        return np.array(rows, np.uint8)

    def _configure(self, episode_horizon=None, lifelong=None, goal_change_frequency=None):
        if self._handle is not None:
            raise RuntimeError("wrappers must be applied before the env is first reset/stepped")
        if episode_horizon is not None:
            self._episode_horizon = int(episode_horizon)
        if lifelong is not None:
            self._lifelong = bool(lifelong)
        if goal_change_frequency is not None:
            self._goal_change_frequency = int(goal_change_frequency)

    def _flags(self):
        f = 0
        if self._reward_type == "dense":
            f |= _lib.FLAG_DENSE_REWARD
        if self._wide_init_distr:
            f |= _lib.FLAG_WIDE_INIT
        if self._state_dtype == "float64":
            f |= _lib.FLAG_STATE_F64
        if self._lifelong:
            f |= _lib.FLAG_LIFELONG
        if self._auto_reset:
            f |= _lib.FLAG_AUTO_RESET
        if self._reset_at_goal:
            f |= _lib.FLAG_RESET_AT_GOAL
        if self._eval_stats:
            f |= _lib.FLAG_EVAL_STATS
        if self._per_env_goals:
            f |= _lib.FLAG_PER_ENV_GOALS
        if self._keep_final_obs:
            f |= _lib.FLAG_FINAL_OBS
        return f

    def _model_blob(self):
        m = _lib.TabletopModel()
        m.magic = _lib.TABLETOP_MAGIC
        m.num_goals = len(self._goal_table)
        m.threshold = self.threshold
        m.move_distance = self.move_distance
        m.clip = 2.8
        m.success_radius = 0.2
        for k in range(6):
            m.initial_state[k] = float(self.initial_state[k])
        for r, g in enumerate(self._goal_table):
            for k in range(6):
                m.goal_table[r][k] = float(g[k])
        return m

    def _ensure(self):
        if self._handle is not None:
            return
        L = _lib.lib()
        # the pre-drawn goal stream is a ring of `goal_stream_rows` draws per env: a lifelong run takes
        # horizon / goal_change_frequency of them (125 with the reference's defaults), so size it from the configuration
        # instead of letting the cursor wrap silently into a periodic goal sequence (ADVICE r1)
        if self._lifelong and self._goal_change_frequency > 0 and self._episode_horizon < _NEVER:
            need = -(-self._episode_horizon // self._goal_change_frequency) + 2
            if need > self._goal_stream_rows:
                if need * self._total_envs <= (1 << 28):
                    self._goal_stream_rows = int(need)
                else:
                    import warnings
                    warnings.warn(f"goal stream of {self._goal_stream_rows} draws per env wraps before the horizon "
                                  f"({need} needed); pass goal_stream_rows explicitly", RuntimeWarning)
        cfg = _lib.EarlConfig(_lib.ENV_TABLETOP, self.num_envs, self.device.index or 0, self._flags(),
                              self._episode_horizon, self._goal_change_frequency, self._goal_stream_rows, 0)
        blob = self._model_blob()
        h = C.c_void_p()
        _lib.check(L.earl_create(C.byref(cfg), C.byref(blob), C.sizeof(blob), C.byref(h)))
        self._handle = h
        zc = _hostio.host_zerocopy_default()
        if zc is not None:
            _lib.check(L.earl_set_host_zerocopy(h, zc))
        # goal stream: draw e of (global) env j = stream[e * total_envs + j]
        stream = rng.PyRandom(self._seed).tabletop_goal_rows(self._goal_stream_rows * self._total_envs,
                                                             self._task_to_row)
        rows = np.ascontiguousarray(
            stream.reshape(self._goal_stream_rows, self._total_envs)[:, self._env_offset:self._env_offset + self.num_envs])
        self._goal_stream = rows
        _lib.check(L.earl_set_goal_stream(h, rows.ctypes.data, self._goal_stream_rows))
        n, dev = self.num_envs, self.device
        self._obs = torch.empty((n, OBS_DIM), dtype=torch.float32, device=dev)
        self._reward = torch.empty((n,), dtype=torch.float32, device=dev)
        self._done = torch.empty((n,), dtype=torch.uint8, device=dev)
        self._success = torch.empty((n,), dtype=torch.uint8, device=dev)
        if self._keep_final_obs:   # rows of envs that have not ended an episode yet hold NaN
            self._final_obs = torch.full((n, OBS_DIM), float("nan"), dtype=torch.float32, device=dev)
            _lib.check(L.earl_set_final_obs(h, self._final_obs.data_ptr()))

    def close(self):
        if self._handle is not None:
            _lib.lib().earl_destroy(self._handle)
            self._handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ------------------------------------------------------------------ goals
    def _goal_rows_for(self, goal):
        """Map goal vector(s) [6] or [N,6] to goal-table rows, appending unseen goals."""
        g = np.asarray(goal.detach().cpu().numpy() if isinstance(goal, torch.Tensor) else goal, np.float64)
        g = np.broadcast_to(g.reshape(-1, 6) if g.ndim > 1 else g[None, :], (self.num_envs, 6))
        uniq, inv = np.unique(g, axis=0, return_inverse=True)
        rows = np.zeros(len(uniq), np.int32)
        for k, u in enumerate(uniq):
            for r, t in enumerate(self._goal_table):
                if np.array_equal(t, u):
                    rows[k] = r
                    break
            else:
                if len(self._goal_table) >= 256:
                    raise ValueError("goal table is full (256 distinct goals)")
                self._goal_table.append(u.copy())
                rows[k] = len(self._goal_table) - 1
                if self._handle is not None:
                    row = np.ascontiguousarray(u)
                    _lib.check(_lib.lib().earl_set_goal_table(self._handle, row.ctypes.data, int(rows[k]), 1))
        return rows[inv.reshape(-1)].astype(np.int32)

    def get_next_goal(self):
        """Draw the next goal of every env from its stream (advances it, like the reference consumes
        `random`), returning [N,6] float64.  Cold path: goes through a state snapshot."""
        self._ensure()
        snap = self.get_state()
        cur = snap["goal_cursor"]
        rows = self._goal_stream[cur % self._goal_stream_rows, np.arange(self.num_envs)]
        snap["goal_cursor"] = cur + 1
        self.set_state(snap)
        return np.stack([self._goal_table[r] for r in rows])

    def reset_goal(self, goal=None, mask=None):
        self._ensure()
        idx = None
        if goal is not None:
            idx = torch.from_numpy(self._goal_rows_for(goal)).to(self.device)
        m = self._mask(mask)
        _lib.check(_lib.lib().earl_set_goal(self._handle, _ptr(m), _ptr(idx), _stream()))

    @property
    def goal(self):
        """Current goals [N,6] float64 (reference attribute `self.goal`)."""
        if self._per_env_goals:
            return self.get_goals().cpu().numpy().astype(np.float64)
        snap = self.get_state()
        return np.stack([self._goal_table[r] for r in snap["goal_row"]])

    def set_goals(self, goals, mask=None):
        """reset_goal(goal) with any goal per env, effective at once (per_env_goals=True envs only).

        goals: CUDA float32 / float64 tensor [N,6], or [6] for every env; mask: CUDA bool / uint8 [N] or None (all envs).
        The masked envs pursue their new goal from now on: the returned observation [N,12] carries it (the other rows are
        the current observation) and the next step's reward, success, statistics and lifelong return are measured against
        it.  float64 goals are rounded to float32 as the goal table rounds them.  A later reset, reset_goal, lifelong goal
        swap or auto-reset gives the env the task's goal back.  One launch on the current stream, no synchronisation.
        host_io=True envs also take numpy / CPU input and return numpy."""
        if not self._per_env_goals:
            raise RuntimeError("set_goals needs an env built with per_env_goals=True")
        self._ensure()
        g, dtype, m = goal_args(goals, mask, self.num_envs, 6, self.device, self._host_mode)
        obs = torch.empty((self.num_envs, OBS_DIM), dtype=torch.float32, device=self.device)
        _lib.check(_lib.lib().earl_set_goals(self._handle, g.data_ptr(), dtype, _ptr(m), obs.data_ptr(), _stream()))
        return obs.cpu().numpy() if self._host_mode else obs

    def get_goals(self):
        """CUDA float32 [N,6]: the goal every env pursues now (per_env_goals=True envs only)."""
        if not self._per_env_goals:
            raise RuntimeError("get_goals needs an env built with per_env_goals=True")
        self._ensure()
        out = torch.empty((self.num_envs, 6), dtype=torch.float32, device=self.device)
        _lib.check(_lib.lib().earl_get_goals(self._handle, out.data_ptr(), _stream()))
        return out

    # ------------------------------------------------------------------ reset / step
    def _mask(self, mask):
        if mask is None:
            return None
        m = torch.as_tensor(mask, device=self.device)
        return m.to(torch.uint8).contiguous()

    def is_valid_init(self, state, goals):  # tabletop_manipulation.py:89-97
        if np.linalg.norm(state[0:2] - state[2:4]) < 1:
            return False
        for g in goals:
            if np.linalg.norm(state[2:4] - g[2:4]) < 1:
                return False
        return True

    def _wide_init_states(self, count):
        """np.random.uniform(-2.5, 2.5, 4) with rejection (tabletop_manipulation.py:114-117), one per env,
        drawn sequentially from this env's legacy-numpy stream."""
        out = np.empty((count, 4))
        for k in range(count):
            q = self._np_random.uniform(-2.5, 2.5, 4)
            while not self.is_valid_init(q, goal_states):
                q = self._np_random.uniform(-2.5, 2.5, 4)
            out[k] = q
        return out

    def reset(self, mask=None, goal_rows=None, init_qpos=None):
        """reset() of every env (or those in `mask`).  goal_rows / init_qpos override the draws."""
        self._ensure()
        m = self._mask(mask)
        if init_qpos is None and self._wide_init_distr and not self._reset_at_goal:
            q = np.zeros((self.num_envs, 4))
            if m is None:
                # a full reset of a sharded job draws for ALL envs of the global batch, in env order, and keeps its slice
                # (like the goal stream and the Sawyer / kitchen resets), so results do not depend on the number of GPUs
                # (ADVICE r1: every rank used to draw the same states from its own copy of the stream)
                q[:] = self._wide_init_states(self._total_envs)[self._env_offset:self._env_offset + self.num_envs]
            else:
                sel = m.cpu().numpy().astype(bool)
                q[sel] = self._wide_init_states(int(sel.sum()))
            init_qpos = q
        iq = None
        if init_qpos is not None:
            iq = torch.as_tensor(np.ascontiguousarray(init_qpos, np.float64)).to(self.device).reshape(self.num_envs, 4).contiguous()
        gi = None
        if goal_rows is not None:
            gi = torch.as_tensor(np.broadcast_to(np.asarray(goal_rows, np.int32), (self.num_envs,)).copy()).to(self.device)
        _lib.check(_lib.lib().earl_reset(self._handle, _ptr(m), _ptr(gi), _ptr(iq), 0, _stream()))
        obs = self._get_obs()
        return obs.cpu().numpy() if self._host_mode else obs   # numpy-driven env: numpy out, like its step()

    def step(self, action, out=None):
        """One step of every env.

        action: CUDA float32 tensor [N,3] -> returns CUDA tensors (obs [N,12], reward [N], done [N] bool, info);
                the tensors are owned by the env and valid until the next step (pass out=(obs, reward, done,
                success) to write elsewhere).
                numpy array / CPU tensor [N,3] -> host path (H2D copy, kernel, D2H copies inside the call),
                returns numpy arrays.
        final_obs=True envs add info["final_observation"] [N,12]: on rows where done is set, the observation the step
        reached before the auto-reset replaced it (obs holds the post-reset one); other rows keep what an earlier step
        stored there (NaN before an env's first episode ends).  The env-owned tensor, valid until the next step like obs;
        a numpy copy on the host path.
        """
        self._ensure()
        if isinstance(action, torch.Tensor) and action.is_cuda:
            a = action
            if a.dtype != torch.float32 or not a.is_contiguous():
                a = a.to(torch.float32).contiguous()
            if a.numel() != self.num_envs * ACT_DIM:
                raise ValueError(f"action must have shape [{self.num_envs},{ACT_DIM}]")
            obs, rew, done, succ = out if out is not None else (self._obs, self._reward, self._done, self._success)
            _lib.check(_lib.lib().earl_step(self._handle, a.data_ptr(), obs.data_ptr(), rew.data_ptr(), done.data_ptr(),
                                            _ptr(succ), _stream()))
            info = {"success": None if succ is None else succ.view(torch.bool)}
            if self._final_obs is not None:
                info["final_observation"] = self._final_obs
            return obs, rew, done.view(torch.bool), info
        return self._step_host(action)

    def _step_host(self, action):
        """numpy / CPU-tensor step: H2D copy, kernel, D2H copies inside one C call; returns numpy arrays that stay valid
        until the step after next (two alternating pinned output sets, envs/_hostio.py)."""
        if self._host_bufs is None:
            self._host_bufs = HostBuffers(self.num_envs, ACT_DIM, OBS_DIM)
        hb = self._host_bufs
        src = hb.stage(action)
        ho, hr, hd, hs = hb.next_outputs()
        _lib.check(_lib.lib().earl_step_host(self._handle, src.data_ptr(), ho.data_ptr(), hr.data_ptr(), hd.data_ptr(),
                   hs.data_ptr()))
        return HostBuffers.as_numpy(ho, hr, hd, hs, self._final_obs)

    def rollout_into(self, actions, num_steps, obs, reward, done, success=None):
        """`num_steps` back-to-back steps: step t reads actions[t % K], writes slot t % R of obs/reward/done
        (shapes [K,N,3]; [R,N,12], [R,N], [R,N]).  Not available on final_obs=True envs."""
        if self._keep_final_obs:
            raise RuntimeError("rollout_into does not keep final observations: step() a final_obs=True env")
        self._ensure()
        K, R = actions.shape[0], obs.shape[0]
        assert actions.is_cuda and actions.dtype == torch.float32 and actions.is_contiguous()
        assert obs.shape == (R, self.num_envs, OBS_DIM) and reward.shape == (R, self.num_envs) and done.shape == (R, self.num_envs)
        _lib.check(_lib.lib().earl_rollout(self._handle, actions.data_ptr(), K, int(num_steps), obs.data_ptr(),
                                           reward.data_ptr(), done.data_ptr(), _ptr(success), R, _stream()))

    # ------------------------------------------------------------------ observation / reward
    def _get_obs(self):
        self._ensure()
        obs = torch.empty((self.num_envs, OBS_DIM), dtype=torch.float32, device=self.device)
        _lib.check(_lib.lib().earl_get_obs(self._handle, obs.data_ptr(), _stream()))
        return obs

    def get_obs(self):
        return self._get_obs()

    def _reward_and_success(self, obs):
        self._ensure()
        host = not (isinstance(obs, torch.Tensor) and obs.is_cuda)
        o = torch.as_tensor(np.asarray(obs, np.float32) if host and not isinstance(obs, torch.Tensor) else obs)
        o = o.to(self.device, torch.float32).reshape(-1, OBS_DIM).contiguous()
        m = o.shape[0]
        rew = torch.empty((m,), dtype=torch.float32, device=self.device)
        suc = torch.empty((m,), dtype=torch.uint8, device=self.device)
        _lib.check(_lib.lib().earl_compute_reward(self._handle, o.data_ptr(), m, rew.data_ptr(), suc.data_ptr(), _stream()))
        if host:
            return rew.cpu().numpy(), suc.cpu().numpy().view(np.bool_)
        return rew, suc.view(torch.bool)

    def compute_reward(self, obs):
        return self._reward_and_success(obs)[0]

    def is_successful(self, obs=None):
        if obs is None:
            obs = self._get_obs()
        return self._reward_and_success(obs)[1]

    # ------------------------------------------------------------------ counters / stats / snapshots
    def _counters(self, want_ll=False):
        self._ensure()
        total = C.c_int64()
        n = self.num_envs
        interv = torch.empty((n,), dtype=torch.int64, device=self.device)
        since = torch.empty((n,), dtype=torch.int32, device=self.device)
        ll = torch.empty((n,), dtype=torch.float64, device=self.device) if want_ll else None
        _lib.check(_lib.lib().earl_counters(self._handle, C.byref(total), interv.data_ptr(), since.data_ptr(), _ptr(ll), _stream()))
        return total.value, interv, since, ll

    def eval_stats(self):
        """Device tensor [4] float64: (sum episode return, #success at last step, #success at any step, N)."""
        self._ensure()
        out = torch.empty((4,), dtype=torch.float64, device=self.device)
        _lib.check(_lib.lib().earl_eval_stats(self._handle, out.data_ptr(), _stream()))
        return out

    @property
    def launch_count(self):
        return 0 if self._handle is None else int(_lib.lib().earl_launch_count(self._handle))

    _SNAP_FIELDS = (("qpos", np.float64, 4), ("flags", np.uint32, 1), ("steps_since_reset", np.uint32, 1),
                    ("num_interventions", np.int64, 1), ("goal_cursor", np.uint32, 1),
                    ("steps_since_goal_change", np.uint32, 1), ("lifelong_return", np.float64, 1),
                    ("episode_return", np.float64, 1))

    def get_state(self):
        """Snapshot of all per-env state (host dict of numpy arrays; layout in DESIGN.md)."""
        self._ensure()
        torch.cuda.synchronize(self.device)
        L = _lib.lib()
        nb = L.earl_state_nbytes(self._handle)
        buf = np.empty(nb, np.uint8)
        _lib.check(L.earl_get_state(self._handle, buf.ctypes.data, nb))
        hdr = np.frombuffer(buf[:24].tobytes(), dtype=np.dtype([("magic", "<u4"), ("kind", "<i4"), ("n", "<i4"), ("flags", "<u4"), ("total", "<i8")]))[0]
        out = {"total_steps": int(hdr["total"])}
        off, n = 24, self.num_envs
        for name, dt, w in self._SNAP_FIELDS:
            cnt = n * w
            arr = np.frombuffer(buf[off:off + cnt * np.dtype(dt).itemsize].tobytes(), dtype=dt).copy()
            out[name] = arr.reshape(n, w) if w > 1 else arr
            off += cnt * np.dtype(dt).itemsize
        out["attached"] = (out["flags"] & 1).astype(bool)
        out["goal_row"] = ((out["flags"] >> 8) & 0xFF).astype(np.int32)
        return out

    def set_state(self, snap=None, qpos=None, attached=None, goal_row=None):
        """Restore a snapshot, or (reference `set_state(qpos)`) overwrite qpos [N,4] / attached / goal rows."""
        self._ensure()
        s = self.get_state() if snap is None else dict(snap)
        if qpos is not None:
            s["qpos"] = np.ascontiguousarray(np.broadcast_to(np.asarray(qpos, np.float64)[..., :4], (self.num_envs, 4)))
        flags = s["flags"].copy()
        if "attached" in s and snap is not None:
            flags = (flags & ~np.uint32(1)) | s["attached"].astype(np.uint32)
        if "goal_row" in s and snap is not None:
            flags = (flags & ~np.uint32(0xFF00)) | (s["goal_row"].astype(np.uint32) << 8)
        if attached is not None:
            flags = (flags & ~np.uint32(1)) | np.broadcast_to(np.asarray(attached), (self.num_envs,)).astype(np.uint32)
        if goal_row is not None:
            flags = (flags & ~np.uint32(0xFF00)) | (np.broadcast_to(np.asarray(goal_row), (self.num_envs,)).astype(np.uint32) << 8)
        s["flags"] = flags.astype(np.uint32)
        hdr = np.zeros(1, dtype=np.dtype([("magic", "<u4"), ("kind", "<i4"), ("n", "<i4"), ("flags", "<u4"), ("total", "<i8")]))
        hdr["magic"], hdr["kind"], hdr["n"], hdr["flags"], hdr["total"] = 0x45534E50, _lib.ENV_TABLETOP, self.num_envs, self._flags(), s["total_steps"]
        parts = [hdr.tobytes()]
        for name, dt, w in self._SNAP_FIELDS:
            parts.append(np.ascontiguousarray(s[name], dtype=dt).tobytes())
        raw = b"".join(parts)
        _lib.check(_lib.lib().earl_set_state(self._handle, raw, len(raw)))
