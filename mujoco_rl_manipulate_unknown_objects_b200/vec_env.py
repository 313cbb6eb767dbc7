"""BatchedRobotVecEnv — drop-in for `DummyVecEnv([lambda: Monitor(RobotEnv(config))])` (reference train_agent.py:17-23)
holding thousands of RobotEnv instances on one GPU.

Follows the stable-baselines3 VecEnv protocol (reset / step_async / step_wait / step, auto-reset with
infos[i]["terminal_observation"], Monitor's infos[i]["episode"], optional "TimeLimit.truncated", get_attr / set_attr /
env_method / env_is_wrapped / seed / close).  stable-baselines3 and gym are not importable in the build image, so the
class subclasses SB3's VecEnv only when it is present and otherwise duck-types the same methods; spaces fall back to
small stand-ins with the attributes SB3 reads (shape, dtype, low, high, spaces).

`infos` is a lazy sequence: a 4 096-element list of 16-key dicts per step would dominate the wall time
(SURVEY.md §8b), so the per-env dict (same keys as robot_env.py:226-241) is built on first access.
"""
import time
from collections.abc import Sequence
from enum import Enum

import numpy as np

from ._native import INFO
from .config import make_config
from .sim import GripperSim

try:  # pragma: no cover - not installed in the build image
    from stable_baselines3.common.vec_env import VecEnv as _VecEnvBase
except Exception:  # noqa: BLE001
    _VecEnvBase = object

try:  # pragma: no cover
    from gym import spaces as _spaces
except Exception:  # noqa: BLE001
    try:
        from gymnasium import spaces as _spaces
    except Exception:  # noqa: BLE001
        _spaces = None


class _Box:
    def __init__(self, low, high, shape, dtype):
        self.shape, self.dtype = tuple(shape), np.dtype(dtype)
        self.low = np.full(self.shape, low, dtype=self.dtype)
        self.high = np.full(self.shape, high, dtype=self.dtype)

    def sample(self):
        if self.dtype == np.uint8:
            return np.random.randint(0, 256, self.shape).astype(np.uint8)
        return np.random.uniform(-1, 1, self.shape).astype(self.dtype)

    def contains(self, x):
        x = np.asarray(x)
        return x.shape == self.shape and bool(np.all(x >= self.low) and np.all(x <= self.high))


class _Dict(dict):
    def __init__(self, spaces):
        super().__init__(spaces)
        self.spaces = spaces


def _box(low, high, shape, dtype):
    if _spaces is not None:
        return _spaces.Box(low=low, high=high, shape=shape, dtype=dtype)
    return _Box(low, high, shape, dtype)


def make_spaces(config):
    """sensor.py:12-54 (observation) and actuator.py:217-247 (action)."""
    c = 5 if config.full_observation else 4
    d = {"observation": _box(0, 255, (c, config.height_capture, config.width_capture), np.uint8),
         "achieved_goal": _box(-np.inf, np.inf, (2,), np.float32),
         "desired_goal": _box(-np.inf, np.inf, (2,), np.float32)}
    obs = _spaces.Dict(d) if _spaces is not None else _Dict(d)
    act = _box(-1.0, 1.0, (6 if config.include_roll else 5,), np.float32)
    return obs, act


def target_direction(direction):
    """robot_env.py:30-33: 0 -> [1, 0], 45 -> [1, 1] (not normalised).  Any other angle in degrees gives the unit vector of the
    reference's disabled `_get_direction` (robot_env.py:46-54; theta rounded to 2 decimals)."""
    if direction == 0:
        return np.array([1, 0])
    if direction == 45:
        return np.array([1, 1])
    theta = np.round(np.deg2rad(direction), 2)
    return np.array([np.cos(theta), np.sin(theta)])


class Status(Enum):
    """RobotEnv.Status (robot_env.py:19-22): same member names and values, so `info["status"].value` / `.name` work."""
    RUNNING = 0
    FAIL = 1
    TIME_LIMIT = 2


STATUS_NAMES = tuple(m.name for m in Status)


def intrinsic_reward(old_obs, new_obs, full_observation=True):
    """IntrinsicReward.intrinsic_reward (reward.py:57-77) for one stored transition: KL(old || new) between the 256-bin
    histograms of the grey image (cv2.COLOR_BGR2GRAY applied to RGB-ordered data, i.e. channel 0 takes the blue weight:
    (c0*3735 + c1*19235 + c2*9798 + 16384) >> 15) and, with the depth channel, the mean of both terms.  float32 pdfs as
    utils.make_pdf; terms with a zero bin on either side contribute nothing (rel_entr's inf is zeroed at reward.py:67)."""
    def pdf(img):
        h = np.bincount(img.reshape(-1), minlength=256).astype(np.float32)
        return h / np.float32(img.size)

    def kl(p, q):
        m = (p > 0) & (q > 0)
        return float(np.sum(p[m] * np.log(p[m] / q[m])))

    def grey(o):
        c = o[:3].astype(np.uint32)
        return ((c[0] * 3735 + c[1] * 19235 + c[2] * 9798 + 16384) >> 15).astype(np.uint8)

    old_obs, new_obs = np.asarray(old_obs), np.asarray(new_obs)
    r = kl(pdf(grey(old_obs)), pdf(grey(new_obs)))
    if full_observation:
        r = (r + kl(pdf(old_obs[3]), pdf(new_obs[3]))) / 2
    return float(r)


class LazyInfos(Sequence):
    """infos of one vectorised step; infos[i] (the 16 keys of robot_env.py:226-241 plus the VecEnv / Monitor extras) is built
    on demand from the packed info rows.  The image-valued keys are views into the environment's pinned host buffers: they
    stay valid until the next-but-one step() (the buffers flip every step); copy what has to live longer."""

    def __init__(self, rows, dones, terminal_obs, target_dir, t_start, extra=None, obs=None, prev_obs=None, episode_rewards=None,
                 finished_rewards=None, truncation_key=False, object_key=False):
        self._rows, self._dones, self._tobs, self._dir, self._t0 = rows, dones, terminal_obs, target_dir, t_start
        self._object_key = object_key
        self._cache = {}
        self._extra = extra or {}
        self._obs, self._prev_obs, self._ep_rew, self._fin_rew, self._trunc = obs, prev_obs, episode_rewards, finished_rewards or {}, truncation_key

    def __len__(self):
        return len(self._rows)

    def __getitem__(self, i):
        if isinstance(i, slice):
            return [self[k] for k in range(*i.indices(len(self)))]
        if i < 0:
            i += len(self)
        if i in self._cache:
            return self._cache[i]
        r = self._rows[i]
        I = INFO
        status = int(r[I["STATUS"]])
        done = bool(self._dones[i])
        tob = self._tobs.get(i) if (done and self._tobs is not None) else None
        d = {"old_obs": None if self._prev_obs is None else self._prev_obs[i],
             "new_obs": tob if tob is not None else (None if self._obs is None else self._obs[i]),
             "init_obj_pos": r[I["INIT_OBJ_POS"]:I["INIT_OBJ_POS"] + 3].astype(np.float64),
             "final_obj_pos": r[I["FINAL_OBJ_POS"]:I["FINAL_OBJ_POS"] + 3].astype(np.float64),
             "target_dir": self._dir,
             "gripper_open": bool(r[I["GRIPPER_OPEN"]]),
             "controls": np.zeros(2),  # ctrl[5:7] is always zero when step() returns (robot_env.py:149,168)
             "object_grasped": int(r[I["OBJECT_GRASPED"]]),
             "episode_step": int(r[I["EPISODE_STEP"]]),
             # robot_env.py:199,232: the episode's reward array, filled up to this step (the reference hands out its live array)
             "episode_rewards": self._fin_rew[i] if i in self._fin_rew else (None if self._ep_rew is None else self._ep_rew[i]),
             "status": Status(status),
             "gripper_position": r[I["GRIPPER_POS"]:I["GRIPPER_POS"] + 3].astype(np.float64),
             "object_position": r[I["FINAL_OBJ_POS"]:I["FINAL_OBJ_POS"] + 3].astype(np.float64),
             "position_reached": {"target": bool(r[I["REACHED_TARGET"]]), "initial": bool(r[I["REACHED_INITIAL"]]), "fail": bool(r[I["FAIL"]])},
             "total_distance": float(r[I["TOTAL_DISTANCE"]]),
             "line_distance": float(r[I["LINE_DISTANCE"]]),
             # extras (not in the reference's dict)
             "substeps": int(r[I["NSUB_A"]] + r[I["NSUB_B"]] + r[I["NSUB_C"]]),
             "achieved_goal": r[I["ACHIEVED"]:I["ACHIEVED"] + 2].copy(),
             "desired_goal": r[I["DESIRED"]:I["DESIRED"] + 2].copy()}
        if self._object_key:  # mixed simulator: the variant (index into sim.scenes) of the episode the step belongs to
            d["object_id"] = int(r[I["OBJECT"]])
        if done:
            if self._trunc:
                d["TimeLimit.truncated"] = status == 2
            if tob is not None:
                d["terminal_observation"] = {"observation": tob, "achieved_goal": d["achieved_goal"], "desired_goal": d["desired_goal"]}
            d["episode"] = {"r": float(r[I["EPISODE_RETURN"]]), "l": int(r[I["EPISODE_STEP"]]), "t": round(time.time() - self._t0, 6)}
        for k, v in self._extra.items():
            d[k] = v[i]
        self._cache[i] = d
        return d


class _HostBuffers:
    """One set of pinned host arrays a step writes into."""

    def __init__(self, pin, N, obs_shape, adim):
        import torch
        C, H, W = obs_shape
        self.obs = pin((N, C, H, W), torch.uint8)
        self.ag, self.dg = pin((N, 2), torch.float32), pin((N, 2), torch.float32)
        self.rew, self.done = pin((N,), torch.float32), pin((N,), torch.uint8)
        self.info = pin((N, INFO["STRIDE"]), torch.float32)


class BatchedRobotVecEnv(_VecEnvBase):
    """VecEnv of `num_envs` RobotEnv instances (reference simulation/environment/robot_env.py) on one GPU.

    Host-side cost per step is O(1) in python: the simulator stores observations straight into PINNED host arrays while the
    kernel runs (C-ABI grs_step_host), and step() returns VIEWS of those arrays.  Two buffer sets alternate, so what one
    step returned stays intact during the next step (SB3 keeps `_last_obs` exactly that long) and is overwritten by the one
    after; pass copy_outputs=True to get private copies instead (one 20 KB memcpy per environment and step).
    """

    metadata = {"render.modes": ["rgb_array", "depth_array"]}
    Status = Status

    def __init__(self, config=None, num_envs=1, device=0, monitor_file=None, copy_outputs=False, truncation_as_timeout=False, _sim=None, **overrides):
        """monitor_file: directory or file prefix of a stable-baselines3 `monitor.csv` (train_agent.py:22 wraps the
        environment in `Monitor(env, log_dir)`); one `r,l,t` row is appended per finished episode.
        truncation_as_timeout: add infos[i]["TimeLimit.truncated"] when an episode ends at time_horizon.  The reference never
        wraps RobotEnv in gym's TimeLimit (train_agent.py:17-23), so the key does not exist there and SB3 treats the time
        horizon as a terminal state; off by default to keep the reference's training targets."""
        if config is None:
            config = make_config(**overrides)
        self.config = config
        self._monitor = None
        if monitor_file is not None:
            from .sb3_io import MonitorWriter
            self._monitor = MonitorWriter(monitor_file)
        # _sim: wrap an existing simulator (created with auto_reset=True) instead of building one; close() then leaves it open
        self._own_sim = _sim is None
        self.sim = GripperSim(config, num_envs=num_envs, device=device, auto_reset=True) if _sim is None else _sim
        if self.sim.num_envs != int(num_envs):
            raise ValueError("num_envs does not match the simulator")
        self.observation_space, self.action_space = make_spaces(config)
        if _VecEnvBase is not object:  # pragma: no cover
            super().__init__(num_envs, self.observation_space, self.action_space)
        self.num_envs = int(num_envs)
        self.target_direction = target_direction(config.direction)
        self._t_start = time.time()
        self._actions = None
        self._copy, self._trunc = bool(copy_outputs), bool(truncation_as_timeout)
        import torch
        N = self.num_envs
        pin = lambda shape, dt: torch.empty(shape, dtype=dt).pin_memory().numpy()  # noqa: E731
        self._h_act = pin((N, self.sim.action_dim), torch.float32)
        self._bufs = [_HostBuffers(pin, N, self.sim.obs_shape, self.sim.action_dim) for _ in range(2)]
        self._cur = 0  # buffer set holding the most recent observation
        self._h_tobs = pin((N,) + tuple(self.sim.obs_shape), torch.uint8)  # rows are written for finished episodes only
        # robot_env.py:68,199: per-episode reward array of every environment (host mirror, one scatter per step)
        self._ep_rewards = np.zeros((N, int(config.time_horizon)), np.float64)
        self._ep_pos = np.zeros(N, np.int64)
        self._rows = np.arange(N)

    # ------------------------------------------------------------------ VecEnv protocol
    def reset(self):
        b = self._bufs[self._cur]
        self.sim.reset_host(b.obs, b.ag, b.dg)
        self._ep_rewards[...] = 0
        self._ep_pos[...] = 0
        return self._obs_dict(b)

    def step_async(self, actions):
        a = np.asarray(actions, dtype=np.float32)
        if a.shape != self._h_act.shape:
            raise ValueError("actions must have shape %s, got %s" % (self._h_act.shape, a.shape))
        np.clip(a, -1.0, 1.0, out=self._h_act)
        self._actions = self._h_act

    def step_wait(self):
        if self._actions is None:
            raise RuntimeError("step_wait() called without step_async()")
        prev = self._bufs[self._cur]
        self._cur ^= 1
        b = self._bufs[self._cur]
        self.sim.step_host(self._actions, b.obs, b.ag, b.dg, b.rew, b.done, b.info, self._h_tobs)
        self._actions = None
        dones = b.done.view(np.bool_)
        # episode reward arrays (robot_env.py:199): reward of this step at the episode step it was taken at
        T = self._ep_rewards.shape[1]
        self._ep_rewards[self._rows, np.minimum(self._ep_pos, T - 1)] = b.rew
        self._ep_pos += 1
        tobs, finished = None, None
        if dones.any():
            idx = np.flatnonzero(dones)
            tobs = {int(i): self._h_tobs[i].copy() for i in idx}  # the shared terminal buffer is rewritten by later episodes
            finished = {int(i): self._ep_rewards[i].copy() for i in idx}
            self._ep_rewards[idx] = 0
            self._ep_pos[idx] = 0
        infos = LazyInfos(b.info.copy() if self._copy else b.info, dones.copy() if self._copy else dones, tobs, self.target_direction, self._t_start,
                          obs=b.obs, prev_obs=prev.obs, episode_rewards=self._ep_rewards, finished_rewards=finished, truncation_key=self._trunc,
                          object_key=len(self.sim.scenes) > 1)
        if self._monitor is not None and tobs is not None:
            self._monitor.write_step(dones, infos)
        return self._obs_dict(b), (b.rew.copy() if self._copy else b.rew), (dones.copy() if self._copy else dones), infos

    def step(self, actions):
        self.step_async(actions)
        return self.step_wait()

    def _obs_dict(self, b):
        if self._copy:
            return {"observation": b.obs.copy(), "achieved_goal": b.ag.copy(), "desired_goal": b.dg.copy()}
        return {"observation": b.obs, "achieved_goal": b.ag, "desired_goal": b.dg}

    # zero-copy device path (rollouts that keep the policy on the GPU): tensors alias the simulator's buffers
    def step_tensors(self, actions):
        self.sim.step(actions)
        s = self.sim
        return {"observation": s.obs, "achieved_goal": s.achieved_goal, "desired_goal": s.desired_goal}, s.reward, s.done, s.info

    @property
    def last_info_rows(self):
        """Packed info records [N, INFO.STRIDE] of the most recent step (a view of the pinned array; layout in _native.INFO)."""
        return self._bufs[self._cur].info

    def close(self):
        if self._monitor is not None:
            self._monitor.close()
        if self._own_sim:
            self.sim.close()

    def seed(self, seed=None):
        # the reference creates np_random but never consumes it (robot_env.py:28,46): resets are deterministic
        return [seed] * self.num_envs

    def get_attr(self, attr_name, indices=None):
        n = len(self._indices(indices))
        if attr_name in ("target_direction",):
            return [self.target_direction] * n
        if attr_name == "config":
            return [self.config] * n
        if attr_name in ("episode_step", "gripper_open", "status"):
            f = self.sim.get_state()["flags"]
            col = {"gripper_open": 0, "episode_step": 1, "status": 2}[attr_name]
            vals = f[self._indices(indices), col]
            if attr_name == "gripper_open":
                return [bool(v) for v in vals]
            if attr_name == "status":
                return [Status(int(v)) for v in vals]
            return [int(v) for v in vals]
        if hasattr(self, attr_name):
            return [getattr(self, attr_name)] * n
        raise AttributeError(attr_name)

    def set_attr(self, attr_name, value, indices=None):
        raise AttributeError("environment attributes are fixed at construction (scene, direction and config are compiled into the simulator)")

    def env_method(self, method_name, *method_args, indices=None, **method_kwargs):
        idx = self._indices(indices)
        if method_name == "compute_reward":
            r = self.compute_reward(*method_args, **method_kwargs)
            return [r] if np.ndim(r) == 0 else list(np.atleast_1d(r))
        if method_name == "seed":
            return [None] * len(idx)
        raise AttributeError("env_method(%r) is not supported by the batched environment" % method_name)

    def env_is_wrapped(self, wrapper_class, indices=None):
        return [False] * len(self._indices(indices))

    def _indices(self, indices):
        if indices is None:
            return list(range(self.num_envs))
        if isinstance(indices, int):
            return [indices]
        return list(indices)

    def get_images(self):
        rgb, _ = self.sim.render(camera_id=2, width=self.config.width_capture, height=self.config.height_capture)
        return list(rgb.cpu().numpy())

    def render(self, mode="rgb_array", camera_id=None, width=640, height=480, env_index=0):
        """RobotEnv.render (robot_env.py:302-340): camera_id 0-2 = one camera, 3 = cameras 0-2 side by side."""
        cid = self.config.camera_id if camera_id is None else camera_id
        cams = [cid] if cid in (0, 1, 2) else list(range(cid))
        out = []
        for c in cams:
            rgb, depth = self.sim.render(camera_id=c, width=width, height=height)
            out.append((depth if mode == "depth_array" else rgb)[env_index].cpu().numpy())
        return np.hstack(out)

    # ------------------------------------------------------------------ HER support
    def compute_reward(self, achieved_goal, desired_goal, info):
        """RobotEnv.compute_reward (robot_env.py:243-273) for stored transitions: progress reward from the recorded object
        positions, + the intrinsic KL term between info["old_obs"] and info["new_obs"] when config.im_reward
        (reward.py:45-77), + the HER goal term when config.her_buffer.  `info` may be one dict or a sequence/array of dicts."""
        infos = [info] if isinstance(info, dict) else list(info)
        ag = np.atleast_2d(np.asarray(achieved_goal, dtype=np.float32))
        dg = np.atleast_2d(np.asarray(desired_goal, dtype=np.float32))
        out = np.zeros(len(infos), np.float64)
        d = self.target_direction.astype(np.float64)
        for k, inf in enumerate(infos):
            ip, fp = np.asarray(inf["init_obj_pos"], np.float64), np.asarray(inf["final_obj_pos"], np.float64)
            pi, pf = ip[:2] @ d / (d @ d), fp[:2] @ d / (d @ d)
            lat, trav = np.linalg.norm(pf * d - fp[:2]), pf - pi
            r = 0.0
            if 0.0 < trav < 0.1 and lat < 0.1:
                r = trav
                ctr = np.asarray(inf.get("controls", (0.0, 0.0)))
                if (not inf["gripper_open"]) and bool(np.all(ctr) != 0) and inf["object_grasped"] == 3:
                    r *= 2
                    if fp[2] > 0:
                        r *= 1.5
            out[k] = r * 30
            if self.config.im_reward:
                if inf.get("old_obs") is None or inf.get("new_obs") is None:
                    raise KeyError("compute_reward with im_reward needs info['old_obs'] and info['new_obs'] (robot_env.py:250-251)")
                out[k] += intrinsic_reward(inf["old_obs"], inf["new_obs"], bool(self.config.full_observation))
            if self.config.her_buffer:
                out[k] += 1.0 / np.exp(np.linalg.norm(dg[min(k, len(dg) - 1)] - ag[min(k, len(ag) - 1)]))
        return out if not isinstance(info, dict) else float(out[0])
