"""Single-environment facade with the reference's ``gym.Env`` contract
(gym_auv/environment.py:21-490), backed by a 1-env ``AUVVecEnv``.

    env = gym_auv_b200.make("MovingObstaclesNoRules-v0")      # like gym.make(id)
    obs = env.reset()
    obs, reward, done, info = env.step([0.5, 0.6])            # gym-0.21 4-tuple

Constructor signature, return types (``float`` reward, ``bool`` done, ``dict`` info with
the four reference keys), ``seed()``, spaces, and the attributes the reference's driver
reads (``history, last_episode, total_t_steps, episode, t_step, cumulative_reward,
config, obstacles, vessel, path, rewarder.params`` -- scripts/run.py:415-426) are kept.
A scenario plug-in overrides ``_generate()`` and returns a ``ScenarioSet`` (the batched
counterpart of setting ``self.vessel/self.path/self.obstacles``, environment.py:394-399)
holding one scenario -- or, via ``_generate_block(n)``, the scenarios of the next n episodes:
the facade keeps ONE AUVVecEnv (device tables, path bank, reset cache) alive for the whole
block and moves from scenario to scenario with ``reset_envs``; it is rebuilt only when the
block is used up.  Rendering is out of scope (SURVEY.md section 2 #14-15):
``renderer`` must be None.
"""
from __future__ import annotations

from types import SimpleNamespace
from typing import Optional, Union

import numpy as np

from . import scenarios as S
from .config import Config, effective_reference_config
from .spaces import Box, Dict as DictSpace

REWARDER_PARAMS = {  # rewarder.py:56-70, 143-159
    "colav": dict(gamma_theta=10.0, gamma_x=0.1, gamma_v_y=1.0, gamma_y_e=5.0, penalty_yawrate=10.0,
                  penalty_torque_change=0.0, penalty_slow=-2, cruise_speed=0.1, slow_speed=0.04,
                  neutral_speed=0.05, negative_multiplier=2.0, collision=-10000.0, **{"lambda": 0.5}, eta=0),
    "pathfollow": dict(gamma_theta=10.0, gamma_x=0.1, gamma_v_y=1.0, gamma_y_e=5.0, penalty_yawrate=10.0,
                       penalty_torque_change=0.0, cruise_speed=0.1, neutral_speed=0.05, negative_multiplier=2.0,
                       collision=-10000.0, **{"lambda": 0.5}, eta=0),
}


class AUVEnv:
    """Base class; subclasses provide ``_generate()`` (see ``scenario_env``)."""

    metadata = {"render.modes": []}
    scenario_name = ""
    block_size = 64  # episodes generated (and uploaded) at a time by families that implement _generate_block

    def __init__(
        self,
        env_config: Union[Config, dict, None] = None,
        test_mode: bool = False,
        renderer: Optional[str] = None,
        verbose: bool = False,
        device: str = "cuda:0",
    ):
        if isinstance(env_config, dict):  # RLlib-style {"config": Config} (environment.py:63-71)
            cfg = env_config["config"]
            assert isinstance(cfg, Config), f"Expected config attribute of env_config to be Config, got {type(cfg)}!"
        elif env_config is None:
            cfg = Config()
        else:
            assert isinstance(env_config, Config), f"Expected Config, got {type(env_config)}!"
            cfg = env_config
        if renderer not in (None, "none"):
            raise ValueError("rendering is outside the B200 step path; pass renderer=None")
        self.config = cfg
        self.test_mode = test_mode
        self.renderer = None
        self.verbose = verbose
        self.device = device
        self.episode = 0
        self.total_t_steps = 0
        self.history = []
        self.last_episode = None
        self.last_reward = 0
        self.rng = None
        self._seed_counter = 0
        self.seed()
        self._vec = None
        self._recycle = False
        self._block_pos = 0
        self._idx = 0
        self.vec_env_builds = 0  # how many times the backing AUVVecEnv was (re)built (diagnostic)
        n = cfg.vessel.dense_observation_size + (cfg.vessel.n_lidar_observations if cfg.vessel.use_lidar else 0)
        self.n_observations = n
        self._action_space = Box(low=np.array([-1, -0.15]), high=np.array([1, 0.15]), dtype=np.float32)
        if cfg.vessel.use_dict_observation:
            self._observation_space = DictSpace(
                {
                    "proprioceptive": Box(-1.0, 1.0, shape=(6,), dtype=np.float32),
                    "lidar": Box(-1.0, 1.0, shape=cfg.vessel.lidar_shape, dtype=np.float32),
                }
            )
        else:
            self._observation_space = Box(low=-np.ones(n), high=np.ones(n), dtype=np.float32)
        self.reset()

    # -- plug-in hook -------------------------------------------------------------
    def _generate(self) -> S.ScenarioSet:
        raise NotImplementedError

    def _generate_block(self, n: int):
        """-> (ScenarioSet, recycle).  The scenarios of the next episodes, in order; recycle=True means the
        set is the same every time (a deterministic scenario) and is simply replayed."""
        return self._generate(), False

    # -- gym contract -------------------------------------------------------------
    @property
    def action_space(self):
        return self._action_space

    @property
    def observation_space(self):
        return self._observation_space

    def seed(self, seed=None):
        if seed is None:
            seed = int(np.random.SeedSequence().entropy % (2**31))
        self.rng = np.random.RandomState(seed)
        return [seed]

    def reset(self, save_history: bool = True):
        from .vec_env import AUVVecEnv

        if self._vec is not None and self.t_step:
            self.save_latest_episode(save_history)
        self.episode += 1
        self.total_t_steps += self.t_step if self._vec is not None else 0
        self.last_reward = 0
        self._info = dict(collision=False, reached_goal=False, goal_distance=None, progress=0)
        if self._vec is None or (self._block_pos >= self.scenario.n_scenarios and not self._recycle):
            self.scenario, self._recycle = self._generate_block(self.block_size)
            self._vec = AUVVecEnv(self.scenario, 1, self.config, device=self.device, test_mode=self.test_mode,
                                  auto_reset=False, debug=True, count_ray_tests=False, record_tracks=1,
                                  track_capacity=max(1, int(self.config.episode.max_timesteps)))
            self.vec_env_builds += 1
            self.rewarder = SimpleNamespace(params=dict(REWARDER_PARAMS[self.scenario.rewarder]))
            self._block_pos, self._idx = 1, 0
            return self._format_obs(self._vec.reset())
        import torch

        self._idx = self._block_pos % self.scenario.n_scenarios
        self._block_pos += 1
        one = torch.ones(1, dtype=torch.uint8, device=self._vec.device)
        obs = self._vec.reset_envs(one, torch.tensor([self._idx], dtype=torch.int32, device=self._vec.device))
        self._vec.check_status()
        return self._format_obs(self._vec._fmt(obs))

    def step(self, action):
        import torch

        a = np.asarray(action, dtype=np.float32).reshape(1, 2)
        obs, reward, done, info = self._vec.step(torch.as_tensor(a, device=self._vec.device))
        reward = float(reward.item())
        done = bool(done.item())
        self.last_reward = reward
        self._info = dict(
            collision=bool(info["collision"].item()),
            reached_goal=bool(info["reached_goal"].item()),
            goal_distance=float(info["goal_distance"].item()),
            progress=float(info["progress"].item()),
        )
        return self._format_obs(obs), reward, done, dict(self._info)

    def observe(self):
        return self._format_obs(self._vec.observe(mode=1))

    def close(self):
        self._vec = None

    def render(self, mode="rgb_array", **kwargs):
        raise NotImplementedError("rendering is outside the B200 step path (SURVEY.md section 2 #14)")

    def _format_obs(self, obs):
        if isinstance(obs, dict):  # the batched env already split it (AUVVecEnv.observation_dict)
            return {k: v[0].detach().cpu().numpy().astype(np.float64) for k, v in obs.items()}
        o = obs[0].detach().cpu().numpy().astype(np.float64)
        if self.config.vessel.use_dict_observation:
            R = self.config.vessel.n_sensors
            return {"proprioceptive": o[:6], "lidar": o[6:].reshape(-1, R)}
        return o

    # -- attributes the reference driver reads -------------------------------------
    @property
    def t_step(self):
        return int(self._vec.get_attr("t_step").item()) if self._vec is not None else 0

    @property
    def cumulative_reward(self):
        return float(self._vec.get_attr("cumulative_reward").item()) if self._vec is not None else 0.0

    @property
    def collision(self):
        return self._info["collision"]

    @property
    def reached_goal(self):
        return self._info["reached_goal"]

    @property
    def progress(self):
        return self._info["progress"]

    @property
    def goal_distance(self):
        return self._info["goal_distance"]

    @property
    def vessel(self):
        st = self._vec.state[:, 0].cpu().numpy()
        d = self._vec.get_attr("lidar_dist")[0].cpu().numpy() if self.config.vessel.use_lidar else None
        return SimpleNamespace(position=st[0:2], heading=float(st[2]), velocity=st[3:5], yaw_rate=float(st[5]),
                               speed=float(np.linalg.norm(st[3:5])), width=self.config.vessel.vessel_width,
                               n_sensors=self.config.vessel.n_sensors, sensor_angles=self._vec.sensor_angles,
                               distance_measurements=d, max_speed=2,
                               progress=self.progress, max_progress=float(self._vec.get_attr("max_progress").item()))

    @property
    def path(self):
        return self.scenario.bank.tables[int(self.scenario.path_id[self._idx])]

    @property
    def obstacles(self):
        return self.scenario.describe(self._idx)

    def save_latest_episode(self, save_history=True):
        """environment.py:466-489.  ``path_taken`` and the obstacles' histories are the episode track the step
        kernel recorded (``AUVVecEnv.current_episode``: reset() saves whatever episode was running).  The track
        holds ``max_timesteps`` steps; a longer episode (``test_mode`` has no time limit) keeps its last
        ``max_timesteps`` rows: ``truncated`` is then True and ``step_index`` numbers the rows (row 0 is not
        the initial pose)."""
        rec = self._vec.current_episode(0)
        obstacles = dict(self.obstacles, moving_path_taken=rec["obstacles"]["moving_path_taken"])
        self.last_episode = {"path": self.path(np.linspace(0, self.path.length, 1000)), "path_taken": rec["path_taken"],
                             "heading_taken": rec["heading_taken"], "rewards": rec["rewards"], "obstacles": obstacles,
                             "truncated": rec["truncated"]}
        if rec["truncated"]:
            self.last_episode["step_index"] = rec["step_index"]
        if save_history:
            t = self.t_step
            self.history.append({
                "cross_track_error": float(self._vec._st["cte_sum"].item() / max(t, 1)),
                "reached_goal": int(self.reached_goal), "collision": int(self.collision),
                "reward": self.cumulative_reward, "timesteps": t,
                "duration": t * self.config.simulation.t_step_size, "progress": self.progress,
                "pathlength": self.path.length,
            })


def scenario_env(name: str, default_config=None):
    """Build the AUVEnv subclass for a registered scenario id."""
    builder = S.SCENARIOS[name]

    class _Env(AUVEnv):
        scenario_name = name

        def _generate(self):
            import inspect

            params = inspect.signature(builder).parameters
            if "seed" in params:
                return builder(seed=int(self.rng.randint(0, 2**31 - 1)))
            if "start_angle" in params:
                return builder(start_angle=float(self.rng.uniform(-np.deg2rad(5), np.deg2rad(5))))
            return builder()

        def _generate_block(self, n):
            import inspect

            params = inspect.signature(builder).parameters
            if "n" in params and "seed" in params:  # random families: the next n episodes in one set
                return builder(n=int(n), seed=int(self.rng.randint(0, 2**31 - 1))), False
            return self._generate(), not ({"seed", "start_angle"} & set(params))

    _Env.__name__ = name.split("-")[0]
    _Env.default_config = default_config
    return _Env


# scenario id -> effective config family (gym_auv/__init__.py:17-36)
_DEBUG_IDS = {"DebugScenario-v0", "EmptyScenario-v0"}


def make(env_id: str, env_config: Optional[Config] = None, **kwargs) -> AUVEnv:
    """``gym.make(id)`` for the ids of gym_auv/__init__.py:43-121.  Without an explicit
    config the *declared* defaults are used, except DEBUG_CONFIG scenarios which get
    t_step_size=0.5 / min_goal_distance=0.1 as registered by the reference."""
    if env_id not in S.SCENARIOS:
        raise KeyError(f"unknown scenario id {env_id!r}; known: {sorted(S.SCENARIOS)}")
    if env_config is None:
        env_config = effective_reference_config() if env_id in _DEBUG_IDS else Config()
    return scenario_env(env_id)(env_config, **kwargs)
