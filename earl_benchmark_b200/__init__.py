"""earl_benchmark_b200 -- B200-native batched implementation of EARL's environment step.

`EARLEnvs` keeps the surface of the reference loader (`earl_benchmark/__init__.py:83-247`):
    EARLEnvs(env_name, reward_type, reset_train_env_at_goal, setup_as_lifelong_learning, **kwargs)
        .get_envs() / .get_initial_states() / .get_goal_states() / .get_demonstrations() / .has_demos()
and adds the batched arguments `num_envs`, `device`, `seed`, `state_dtype`, `auto_reset` (with `reset_stream_rows` for
sawyer_door, sawyer_peg and kitchen), `eval_stats`,
`rank` / `world_size` (shard a global batch of `num_envs` across processes, one GPU each), and `per_env_goals`
(tabletop_manipulation, sawyer_door and sawyer_peg: the train and eval envs take a goal vector per env, effective at once,
through `set_goals(goals, mask=None)` and report them through `get_goals()`; kitchen raises), and `final_obs` (with
`auto_reset`: the train env's step() adds info["final_observation"], the last observation of every episode the step ended;
eval envs never auto-reset and do not take it).
"""
from . import demos
from .wrappers import lifelong_wrapper, persistent_state_wrapper

__all__ = ["EARLEnvs", "deployment_eval_config", "continuing_eval_config"]

# verbatim VALUES of the reference's two config tables (earl_benchmark/__init__.py:16-81)
deployment_eval_config = {
    'tabletop_manipulation': {'num_initial_state_samples': 1, 'num_goals': 4, 'train_horizon': int(2e5), 'eval_horizon': 200},
    'sawyer_door': {'num_initial_state_samples': 1, 'num_goals': 1, 'train_horizon': int(2e5), 'eval_horizon': 300},
    'sawyer_peg': {'num_initial_state_samples': 15, 'num_goals': 1, 'train_horizon': int(1e5), 'eval_horizon': 200},
    'kitchen': {'num_initial_state_samples': 1, 'train_horizon': int(1e5), 'eval_horizon': 400, 'task': 'all_pairs'},
    'minitaur': {'num_initial_state_samples': 1, 'num_goals': 4, 'train_horizon': int(1e5), 'eval_horizon': 1000},
}
continuing_eval_config = {
    'tabletop_manipulation': {'num_initial_state_samples': 1, 'num_goals': 4, 'train_horizon': int(5e4), 'goal_change_frequency': 400},
    'sawyer_door': {'num_initial_state_samples': 1, 'num_goals': 1, 'train_horizon': int(5e4), 'goal_change_frequency': 600},
    'sawyer_peg': {'num_initial_state_samples': 15, 'num_goals': 1, 'train_horizon': int(5e4), 'goal_change_frequency': 400},
    'kitchen': {'num_initial_state_samples': 1, 'train_horizon': int(5e4), 'goal_change_frequency': 800, 'task': 'all_pairs'},
    'minitaur': {'num_initial_state_samples': 1, 'num_goals': 4, 'train_horizon': int(1e5), 'goal_change_frequency': 2000},
}

_BUILT = ("tabletop_manipulation", "sawyer_door", "sawyer_peg", "kitchen")
_PER_ENV_GOALS = ("tabletop_manipulation", "sawyer_door", "sawyer_peg")


def shard_range(num_envs, rank, world_size):
    """Env-index range [lo, hi) of `rank` when `num_envs` envs are split across `world_size` GPUs."""
    base, rem = divmod(int(num_envs), int(world_size))
    lo = rank * base + min(rank, rem)
    return lo, lo + base + (1 if rank < rem else 0)


class EARLEnvs(object):
    def __init__(self,
                 env_name,
                 reward_type='sparse',
                 reset_train_env_at_goal=False,
                 setup_as_lifelong_learning=False,
                 **kwargs):
        self._env_name = env_name
        self._reward_type = reward_type
        self._reset_train_env_at_goal = reset_train_env_at_goal
        self._setup_as_lifelong_learning = setup_as_lifelong_learning
        self._kwargs = kwargs
        if kwargs.get('final_obs', False) and not kwargs.get('auto_reset', False):
            raise ValueError("final_obs=True needs auto_reset=True: without it, the observation step() returns on done is the final one")

        # batched / device arguments (not in the reference)
        self._num_envs = int(kwargs.get('num_envs', 1))
        self._rank = int(kwargs.get('rank', 0))
        self._world_size = int(kwargs.get('world_size', 1))
        self._lo, self._hi = shard_range(self._num_envs, self._rank, self._world_size)
        self._batched = dict(device=kwargs.get('device'), seed=int(kwargs.get('seed', 0)),
                             state_dtype=kwargs.get('state_dtype', 'float32'),
                             goal_stream_rows=int(kwargs.get('goal_stream_rows', 64)))
        if kwargs.get('per_env_goals', False):
            if env_name not in _PER_ENV_GOALS:
                raise NotImplementedError(f"{env_name}: per_env_goals is built for {', '.join(_PER_ENV_GOALS)} only")
            self._batched['per_env_goals'] = True

        # resolve to default parameters if not provided by the user (KeyError on unknown env, as the reference)
        if not self._setup_as_lifelong_learning:
            self._train_horizon = kwargs.get('train_horizon', deployment_eval_config[env_name]['train_horizon'])
            self._eval_horizon = kwargs.get('eval_horizon', deployment_eval_config[env_name]['eval_horizon'])
            self._num_initial_state_samples = kwargs.get('num_initial_state_samples', deployment_eval_config[env_name]['num_initial_state_samples'])

            self._train_env = self.get_train_env()
            self._eval_env = self.get_eval_env()
        else:
            self._train_horizon = kwargs.get('train_horizon', continuing_eval_config[env_name]['train_horizon'])
            self._num_initial_state_samples = kwargs.get('num_initial_state_samples', continuing_eval_config[env_name]['num_initial_state_samples'])
            self._goal_change_frequency = kwargs.get('goal_change_frequency', continuing_eval_config[env_name]['goal_change_frequency'])
            self._train_env = self.get_train_env(lifelong=True)

    def _shard_kwargs(self, seed_offset):
        b = dict(self._batched)
        b['seed'] = b['seed'] + seed_offset
        b.update(num_envs=self._hi - self._lo, env_offset=self._lo, total_envs=self._num_envs)
        return b

    def _auto_reset_kwargs(self):
        """train envs of the articulated-body tasks: reset in the step when the horizon fires (eval envs never do)"""
        return dict(auto_reset=bool(self._kwargs.get('auto_reset', False)),
                    reset_stream_rows=int(self._kwargs.get('reset_stream_rows', 64)),
                    final_obs=bool(self._kwargs.get('final_obs', False)))

    def _not_built(self):
        raise NotImplementedError(
            f"{self._env_name}: the batched CUDA step for this task is not built yet "
            f"(built: {', '.join(_BUILT)}); there is no CPU fallback")

    def get_train_env(self, lifelong=False):
        if self._env_name == 'tabletop_manipulation':
            from .envs import tabletop_manipulation
            train_env = tabletop_manipulation.TabletopManipulation(
                task_list='rc_r-rc_k-rc_g-rc_b',
                reward_type=self._reward_type,
                reset_at_goal=self._reset_train_env_at_goal,
                wide_init_distr=self._kwargs.get('wide_init_distr', False),
                auto_reset=self._kwargs.get('auto_reset', False),
                final_obs=self._kwargs.get('final_obs', False),
                eval_stats=False,
                **self._shard_kwargs(0))
        elif self._env_name == 'sawyer_door':
            from .envs import sawyer_door
            train_env = sawyer_door.SawyerDoorV2(reward_type=self._reward_type,
                                                 reset_at_goal=self._reset_train_env_at_goal,
                                                 eval_stats=False, **self._auto_reset_kwargs(), **self._shard_kwargs(0))
        elif self._env_name == 'sawyer_peg':
            from .envs import sawyer_peg
            train_env = sawyer_peg.SawyerPegV2(reward_type=self._reward_type,
                                               reset_at_goal=self._reset_train_env_at_goal,
                                               eval_stats=False, **self._auto_reset_kwargs(), **self._shard_kwargs(0))
        elif self._env_name == 'kitchen':
            from .envs import kitchen
            kitchen_task = self._kwargs.get('kitchen_task', deployment_eval_config[self._env_name]['task'])
            train_env = kitchen.Kitchen(task=kitchen_task, reward_type=self._reward_type, **self._auto_reset_kwargs(),
                                        **self._shard_kwargs(0))
        else:
            deployment_eval_config[self._env_name]  # KeyError for unknown names
            self._not_built()

        train_env = persistent_state_wrapper.PersistentStateWrapper(train_env, episode_horizon=self._train_horizon)
        if not lifelong:
            return train_env
        return lifelong_wrapper.LifelongWrapper(train_env, self._goal_change_frequency)

    def get_eval_env(self):
        if self._env_name == 'tabletop_manipulation':
            from .envs import tabletop_manipulation
            eval_env = tabletop_manipulation.TabletopManipulation(
                task_list='rc_r-rc_k-rc_g-rc_b',
                reward_type=self._reward_type,
                wide_init_distr=self._kwargs.get('wide_init_distr', False),
                eval_stats=self._kwargs.get('eval_stats', True),
                **self._shard_kwargs(1))
        elif self._env_name == 'sawyer_door':
            from .envs import sawyer_door
            eval_env = sawyer_door.SawyerDoorV2(reward_type=self._reward_type,
                                                eval_stats=self._kwargs.get('eval_stats', True), **self._shard_kwargs(1))
        elif self._env_name == 'sawyer_peg':
            from .envs import sawyer_peg
            eval_env = sawyer_peg.SawyerPegV2(reward_type=self._reward_type,
                                              eval_stats=self._kwargs.get('eval_stats', True), **self._shard_kwargs(1))
        elif self._env_name == 'kitchen':
            from .envs import kitchen
            kitchen_task = self._kwargs.get('kitchen_task', deployment_eval_config[self._env_name]['task'])
            eval_env = kitchen.Kitchen(task=kitchen_task, reward_type=self._reward_type,
                                       eval_stats=self._kwargs.get('eval_stats', True), **self._shard_kwargs(1))
        else:
            self._not_built()
        return persistent_state_wrapper.PersistentStateWrapper(eval_env, episode_horizon=self._eval_horizon)

    def has_demos(self):
        return self._env_name in ['tabletop_manipulation', 'sawyer_door', 'sawyer_peg']

    def get_envs(self):
        if not self._setup_as_lifelong_learning:
            return self._train_env, self._eval_env
        return self._train_env

    def get_initial_states(self, num_samples=None):
        '''Always returns initial states of the shape N x state_dim (reference :185-219).'''
        if self._env_name == 'tabletop_manipulation':
            from .envs import tabletop_manipulation
            return tabletop_manipulation.initial_states
        if self._env_name == 'sawyer_door':
            from .envs import sawyer_door
            return sawyer_door.initial_states
        if self._env_name == 'sawyer_peg':
            from .envs import sawyer_peg
            return sawyer_peg.initial_states
        if self._env_name == 'kitchen':
            from .envs import kitchen
            return kitchen.initial_states['all_pairs']      # reference :212-217 (get_init_states of a throw-away Kitchen)
        self._not_built()

    def get_goal_states(self):
        if self._env_name == 'tabletop_manipulation':
            from .envs import tabletop_manipulation
            return tabletop_manipulation.goal_states
        if self._env_name == 'sawyer_door':
            from .envs import sawyer_door
            return sawyer_door.goal_states
        if self._env_name == 'sawyer_peg':
            from .envs import sawyer_peg
            return sawyer_peg.goal_states
        if self._env_name == 'kitchen':
            from .envs import kitchen
            return kitchen.goal_states
        self._not_built()

    def get_demonstrations(self, device=None):
        """(forward, reverse) demonstration dicts (reference :238-247); `device` (batched extra) returns the numeric
        arrays as tensors on that device."""
        if demos.available(self._env_name):
            if device is not None:
                return demos.load_to_device(self._env_name, 'forward', device), demos.load_to_device(self._env_name, 'reverse', device)
            return demos.load(self._env_name, 'forward'), demos.load(self._env_name, 'reverse')
        print('please download the demonstrations corresponding to ', self._env_name)
