"""Consumer side of the step path: the VecEnv the reference's trainer drives and the report it
writes (SURVEY.md section 8 f-4).

``B200VecEnv`` has the surface ``scripts/run.py:278-475`` uses on ``SubprocVecEnv`` (stable-baselines
2.9): ``num_envs``, spaces, ``reset()``, ``step_async`` / ``step_wait`` / ``step`` with NumPy in / NumPy
out and a per-env info list, ``get_attr("history")`` / ``env_method`` / ``seed`` / ``close`` -- one object
for N envs on one GPU instead of N worker processes.  ``write_report`` is the text half of
``gym_auv/reporting.py:37-79`` (``report.txt``); the plots stay out of scope.
"""
from __future__ import annotations

import os
from typing import Dict, List, Optional, Sequence

import numpy as np

from .config import Config
from .scenarios import ScenarioSet

HISTORY_KEYS = ("reward", "timesteps", "progress", "collision", "reached_goal", "cross_track_error", "pathlength", "episode")


class InfoList:
    """The ``infos`` a VecEnv returns: list-like, one dict per env with the reference's keys
    (environment.py:336-340) plus stable-baselines' ``terminal_observation`` for finished envs.
    The dicts are built on access -- a Python loop over 65536 envs per step would cost more than the step."""

    def __init__(self, collision, reached_goal, goal_distance, progress, done, terminal):
        self._c, self._g, self._d, self._p, self._done, self._term = collision, reached_goal, goal_distance, progress, done, terminal

    def __len__(self):
        return len(self._c)

    def __getitem__(self, i):
        if isinstance(i, slice):
            return [self[k] for k in range(*i.indices(len(self)))]
        d = dict(collision=bool(self._c[i]), reached_goal=bool(self._g[i]), goal_distance=float(self._d[i]),
                 progress=float(self._p[i]))
        if self._done[i] and self._term is not None:
            d["terminal_observation"] = self._term()[i]
        return d

    def __iter__(self):
        return (self[i] for i in range(len(self)))


class B200VecEnv:
    """N gym-auv envs behind the stable-baselines ``VecEnv`` surface.

    ``scenarios`` is a pool (``gym_auv_b200.scenarios``) -- e.g. ``moving_obstacles_template(2 * n, 17, 11,
    path_period=n)`` with ``fresh_scenarios=True`` draws a new MovingObstacles scenario for every episode on
    the GPU, as the reference's ``_generate()`` does at every ``reset()``.  ``record_history`` keeps the
    per-episode entries of ``env.history`` (environment.py:476-489) for ``get_attr("history")`` / the report.
    ``record_tracks`` envs (spread evenly, ``impl.tracked_envs``) record their episodes on the GPU, up to
    ``track_capacity`` steps each: ``get_attr("last_episode")`` returns the ``save_latest_episode`` dict of each
    one's most recent finished episode (None for the other envs, and before a tracked env finished one).
    """

    def __init__(self, scenarios: ScenarioSet, num_envs: int, config: Optional[Config] = None, device="cuda:0",
                 test_mode: bool = False, fresh_scenarios: bool = False, refresh_every: int = 8, seed: int = 0,
                 record_history: bool = True, history_limit: int = 100000, record_tracks: int = 0,
                 track_capacity: int = 2048, **vec_kw):
        from .vec_env import AUVVecEnv

        self.impl = AUVVecEnv(scenarios, num_envs, config, device=device, test_mode=test_mode, auto_reset=True,
                              record_tracks=record_tracks, track_capacity=track_capacity, **vec_kw)
        self.num_envs = int(num_envs)
        self.observation_space = self.impl.observation_space
        self.action_space = self.impl.action_space
        self.config = self.impl.config
        self.fresh_scenarios = bool(fresh_scenarios)
        self.refresh_every = int(refresh_every)
        self._seed = int(seed)
        self._steps = 0
        self.record_history = bool(record_history)
        self.history: List[Dict[str, float]] = []
        self._history_limit = int(history_limit)
        if self.fresh_scenarios:
            self.impl.regenerate_scenarios(seed=self._seed, epoch=1)

    # ------------------------------------------------------------------ VecEnv
    def seed(self, seed=None):
        if seed is not None:
            self._seed = int(seed)
            if self.fresh_scenarios:
                self.impl.regenerate_scenarios(seed=self._seed, epoch=1)
        return [self._seed + i for i in range(self.num_envs)]

    def reset(self):
        return self.impl.reset().cpu().numpy()

    def step_async(self, actions):
        self.impl.step_async(np.asarray(actions, dtype=np.float32).reshape(self.num_envs, 2))

    def step_wait(self):
        import torch

        obs, rew, done = self.impl.step_wait()
        done = done.astype(bool)
        self._steps += 1
        o = self.impl._out
        n_done = int(done.sum())
        if n_done and self.record_history:
            rows = o["episode_out"][torch.as_tensor(np.nonzero(done)[0], device=self.impl.device)].cpu().numpy()
            for r in rows:
                e = dict(zip(HISTORY_KEYS, (float(v) for v in r)))
                e["duration"] = e["timesteps"] * float(self.config.simulation.t_step_size)
                self.history.append(e)
            if len(self.history) > self._history_limit:
                del self.history[: len(self.history) - self._history_limit]
        # info arrays cross the link only when some env finished (terminal_observation) or on access
        host = {k: o[k].cpu().numpy() for k in ("collision", "reached_goal", "goal_distance", "progress")}
        infos = InfoList(host["collision"], host["reached_goal"], host["goal_distance"], host["progress"], done,
                         (lambda: o["terminal_obs"].cpu().numpy()) if n_done else None)
        if self.fresh_scenarios and self._steps % self.refresh_every == 0:
            with torch.cuda.stream(self.impl._async_stream):
                self.impl.refresh_finished_device(seed=self._seed)
        return obs, rew, done, infos

    def step(self, actions):
        self.step_async(actions)
        return self.step_wait()

    def get_attr(self, attr_name: str, indices: Optional[Sequence[int]] = None):
        """``SubprocVecEnv.get_attr`` (scripts/run.py:415-426 reads ``history``, ``total_t_steps``, ...)."""
        idx = range(self.num_envs) if indices is None else ([indices] if isinstance(indices, int) else indices)
        if attr_name == "history":
            return [self.history for _ in idx]  # one shared history: every env reports the pool's episodes
        if attr_name == "total_t_steps":
            return [self._steps for _ in idx]
        if attr_name == "config":
            return [self.config for _ in idx]
        if attr_name == "last_episode":  # reporting.plot_trajectory / plot_scenario input, per env
            return [self.impl.last_episode(i) for i in idx]
        vals = self.impl.get_attr(attr_name).cpu().numpy()
        return [vals[i] for i in idx]

    def env_method(self, method_name: str, *args, indices=None, **kwargs):
        if method_name == "seed":
            return self.seed(*args, **kwargs)
        raise AttributeError(f"B200VecEnv has no per-env method {method_name!r}")

    def get_images(self, indices: Optional[Sequence[int]] = None, half_width: Optional[float] = None) -> List[np.ndarray]:
        """``VecEnv.get_images``: one ``np.uint8`` (400, 400, 3) top-down frame per env (``AUVVecEnv.render``;
        ``half_width`` defaults to ``config.vessel.render_distance`` and must be given when that is not a number).
        The default is the first ``min(num_envs, 16)`` envs, not all of them: video recorders call this every
        step, and frames of 65536 envs would be 31 GB; a 4 x 4 grid is what a person can look at."""
        idx = list(range(min(self.num_envs, 16))) if indices is None else ([indices] if isinstance(indices, int) else list(indices))
        frames = self.impl.render(idx, half_width=half_width).cpu().numpy()
        return [f for f in frames]

    def render(self, mode: str = "rgb_array", indices: Optional[Sequence[int]] = None,
               half_width: Optional[float] = None) -> np.ndarray:
        """``VecEnv.render``: the ``get_images`` frames tiled into one image, ``ceil(sqrt(n))`` columns, row by
        row, black where the grid has no frame.  Only ``"rgb_array"``: there is no window."""
        if mode != "rgb_array":
            raise NotImplementedError(f"render mode {mode!r}: only 'rgb_array' is supported (there is no window)")
        imgs = self.get_images(indices, half_width=half_width)
        n = len(imgs)
        cols = int(np.ceil(np.sqrt(n)))
        rows = (n + cols - 1) // cols
        h, w, _ = imgs[0].shape
        out = np.zeros((rows * h, cols * w, 3), dtype=np.uint8)
        for k, img in enumerate(imgs):
            r, c = divmod(k, cols)
            out[r * h:(r + 1) * h, c * w:(c + 1) * w] = img
        return out

    def episode_stats(self, reduce: bool = True):
        return self.impl.episode_stats(reduce=reduce)

    def close(self):
        self.impl.close()


def write_report(history: Sequence[Dict[str, float]], report_dir: str, lastn: int = 100) -> str:
    """``report.txt`` of gym_auv/reporting.py:37-79: averages over the last ``lastn`` episodes of an
    ``env.history`` list (entries with the keys of environment.py:476-489).  Returns the file's path."""
    os.makedirs(report_dir, exist_ok=True)
    rel = list(history[-min(lastn, len(history)):]) if lastn > -1 else list(history)
    if not rel:
        raise ValueError("empty history")
    col = lambda k: np.array([h[k] for h in rel], dtype=np.float64)
    collisions, pathlengths, duration = col("collision"), col("pathlength"), col("duration")
    with np.errstate(divide="ignore", invalid="ignore"):
        speeds = np.where(duration > 0, pathlengths / duration, np.nan)
    path = os.path.join(report_dir, "report.txt")
    with open(path, "w") as f:
        f.write("# PERFORMANCE METRICS (LAST {} EPISODES AVG.)\n".format(lastn))
        f.write("{:<30}{:<30}\n".format("Episodes", len(pathlengths)))
        f.write("{:<30}{:<30.2f}\n".format("Avg. Reward", col("reward").mean()))
        f.write("{:<30}{:<30.2f}\n".format("Std. Reward", col("reward").std()))
        f.write("{:<30}{:<30.2%}\n".format("Avg. Progress", col("progress").mean()))
        f.write("{:<30}{:<30.2f}\n".format("Avg. Collisions", collisions.mean()))
        f.write("{:<30}{:<30.2%}\n".format("No Collisions", (collisions == 0).mean()))
        f.write("{:<30}{:<30.2f}\n".format("Avg. Cross-Track Error", col("cross_track_error").mean()))
        f.write("{:<30}{:<30.2f}\n".format("Avg. Timesteps", col("timesteps").mean()))
        f.write("{:<30}{:<30.2f}\n".format("Avg. Duration", duration.mean()))
        f.write("{:<30}{:<30.2f}\n".format("Avg. Pathlength", pathlengths.mean()))
        f.write("{:<30}{:<30.2f}\n".format("Avg. Speed", speeds.mean()))
    return path
