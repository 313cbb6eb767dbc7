"""GripperSim — Python face of the C-ABI (include/b200_gripper_sim.h).

Device buffers are exposed as torch tensors that ALIAS the library's memory (zero copy, through
__cuda_array_interface__); torch is used for nothing else here.  All compute happens in the CUDA library; if it
cannot be loaded, or there is no GPU, construction fails — there is no CPU path.
"""
import ctypes as C

import numpy as np

from . import _native
from ._native import INFO, DBG, GrsConfig
from .config import make_config, scene_path

NQ, NV, NU = 14, 13, 7


class NativeError(RuntimeError):
    pass


def _check(rc):
    if rc != 0:
        raise NativeError(_native.last_error())


class _DevArray:
    """Minimal __cuda_array_interface__ carrier for a raw device pointer."""

    def __init__(self, ptr, shape, typestr):
        self.__cuda_array_interface__ = dict(shape=tuple(shape), typestr=typestr, data=(int(ptr), False), version=2)


class CompiledModel:
    """Compiled scene (the mjModel-like constants).  Works without a GPU (grs_compile_only)."""

    def __init__(self, xml_path=None, _handle=None):
        self._lib = _native.load()
        self._own = _handle is None
        if _handle is None:
            _handle = self._lib.grs_compile_only(str(xml_path).encode())
            if not _handle:
                raise NativeError(_native.last_error())
        self._h = _handle

    def get(self, name):
        n = self._lib.grs_model_get(self._h, name.encode(), None, 0)
        if n < 0:
            m = self._lib.grs_model_get_int(self._h, name.encode(), None, 0)
            if m < 0:
                raise KeyError(name)
            out = np.zeros(m, np.int32)
            self._lib.grs_model_get_int(self._h, name.encode(), out.ctypes.data, m)
            return out
        out = np.zeros(n, np.float64)
        self._lib.grs_model_get(self._h, name.encode(), out.ctypes.data, n)
        return out

    def names(self, kind):
        n = self._lib.grs_model_names(self._h, kind.encode(), None, 0)
        if n < 0:
            raise KeyError(kind)
        buf = C.create_string_buffer(int(n))
        self._lib.grs_model_names(self._h, kind.encode(), buf, n)
        s = buf.value.decode()
        return s.split("\n") if s else []

    @property
    def sizes(self):
        k = ("nbody", "njnt", "nq", "nv", "nu", "ngeom", "nmesh", "npair", "ncam", "nlight")
        return dict(zip(k, self.get("sizes").tolist()))

    def close(self):
        if self._h and self._own:
            self._lib.grs_destroy(self._h)
        self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def compile_model(sim_env):
    return CompiledModel(scene_path(sim_env))


def _grs_config(config, auto_reset):
    c = GrsConfig()
    c.max_steps, c.time_horizon = int(config.max_steps), int(config.time_horizon)
    c.include_roll, c.full_observation = int(bool(config.include_roll)), int(bool(config.full_observation))
    c.im_reward, c.her_buffer = int(bool(config.im_reward)), int(bool(config.her_buffer))
    c.direction = int(config.direction)
    c.width, c.height = int(config.width_capture), int(config.height_capture)
    c.auto_reset = int(bool(auto_reset))
    c.pos_tolerance, c.grasp_tolerance = float(config.pos_tolerance), float(config.grasp_tolerance)
    c.max_translation, c.max_rotation = float(config.max_translation), float(config.max_rotation)
    c.reset_noise_xy, c.reset_noise_yaw = float(getattr(config, "reset_noise_xy", 0.0)), float(getattr(config, "reset_noise_yaw", 0.0))
    c.seed = int(getattr(config, "seed", 0)) & 0xFFFFFFFF
    return c


class GripperSim(CompiledModel):
    """num_envs instances of the reference's RobotEnv (simulation/environment/robot_env.py) on one GPU.

    config: Namespace as produced by the reference's BaseConfig (or make_config()); `direction` is 0 or 45 as in the reference, or any other angle in degrees
    (robot_env.py:30-33).  auto_reset=True gives SB3 VecEnv semantics (an environment is reset inside the step
    that ends its episode; the terminal observation is kept in `terminal_obs`).
    """

    def __init__(self, config=None, num_envs=1, device=0, auto_reset=True, **overrides):
        import torch
        if config is None:
            config = make_config(**overrides)
        elif overrides:
            raise TypeError("pass either a config or keyword overrides")
        if not torch.cuda.is_available():
            raise NativeError("no CUDA device: the simulator has no CPU fallback")
        self._torch = torch
        self.config = config
        self.device_index = int(device)
        self.device = torch.device("cuda", self.device_index)
        lib = _native.load()
        cfg = _grs_config(config, auto_reset)
        h = lib.grs_create(scene_path(config.sim_env).encode(), int(num_envs), C.byref(cfg), self.device_index)
        if not h:
            raise NativeError(_native.last_error())
        super().__init__(_handle=h)
        self._own = True
        self.num_envs = int(num_envs)
        self.action_dim = lib.grs_action_dim(h)
        chw = (C.c_int32 * 3)()
        lib.grs_obs_shape(h, chw)
        self.obs_shape = tuple(chw)
        N, (Cc, H, W) = self.num_envs, self.obs_shape
        self.obs = self._tensor("obs", (N, Cc, H, W), "|u1")
        self.terminal_obs = self._tensor("terminal_obs", (N, Cc, H, W), "|u1")
        self.reset_obs = self._tensor("reset_obs", (Cc, H, W), "|u1")
        self.reward = self._tensor("reward", (N,), "<f4")
        self.done = self._tensor("done", (N,), "|u1")
        self.achieved_goal = self._tensor("achieved", (N, 2), "<f4")
        self.desired_goal = self._tensor("desired", (N, 2), "<f4")
        self.info = self._tensor("info", (N, INFO["STRIDE"]), "<f4")
        self.state = self._tensor("state", (N, _native.STATE_STRIDE), "<f4")
        self.render_state = self._tensor("render_state", (N, _native.RENDER_STATE_STRIDE), "<f4")
        self.debug = self._tensor("debug", (N, _native.DEBUG_STRIDE), "<f4")

    # ------------------------------------------------------------------ plumbing
    def _tensor(self, name, shape, typestr):
        p, sz = C.c_void_p(), C.c_uint64()
        _check(self._lib.grs_buffer(self._h, name.encode(), C.byref(p), C.byref(sz)))
        with self._torch.cuda.device(self.device):
            return self._torch.as_tensor(_DevArray(p.value, shape, typestr), device=self.device)

    def _stream(self):
        # torch's default stream is the legacy NULL stream; the C-ABI reads NULL as "the handle's own stream",
        # so name the legacy stream explicitly (cudaStreamLegacy == 0x1)
        return C.c_void_p(self._torch.cuda.current_stream(self.device).cuda_stream or 1)

    # ------------------------------------------------------------------ RobotEnv surface, batched
    def reset(self, mask=None):
        """RobotEnv.reset (robot_env.py:56-75) for the environments selected by `mask` (uint8/bool tensor on the
        device; None = all).  Results are in .obs / .achieved_goal / .desired_goal."""
        mp = None
        if mask is not None:
            mask = mask.to(device=self.device, dtype=self._torch.uint8).contiguous()
            mp = C.c_void_p(mask.data_ptr())
        _check(self._lib.grs_reset(self._h, mp, self._stream()))

    def step(self, actions):
        """RobotEnv.step (robot_env.py:77-241) for every environment; `actions` float32 [N, A] on the device.
        Runs on torch's current stream.  Results are in .obs/.reward/.done/.achieved_goal/.desired_goal/.info."""
        t = self._torch
        if actions.device != self.device or actions.dtype != t.float32 or not actions.is_contiguous():
            actions = actions.to(device=self.device, dtype=t.float32).contiguous()
        if tuple(actions.shape) != (self.num_envs, self.action_dim):
            raise ValueError("actions must have shape (%d, %d), got %s" % (self.num_envs, self.action_dim, tuple(actions.shape)))
        _check(self._lib.grs_step(self._h, C.c_void_p(actions.data_ptr()), self._stream()))

    def step_host(self, actions, obs=None, achieved=None, desired=None, reward=None, done=None, info=None, terminal_obs=None):
        """The same through HOST numpy buffers (H2D of the actions, the step, D2H of whatever is not None, sync)."""
        a = np.ascontiguousarray(actions, dtype=np.float32)
        if a.shape != (self.num_envs, self.action_dim):
            raise ValueError("actions must have shape (%d, %d), got %s" % (self.num_envs, self.action_dim, a.shape))
        ptr = lambda x: None if x is None else C.c_void_p(x.ctypes.data)  # noqa: E731
        _check(self._lib.grs_step_host(self._h, ptr(a), ptr(obs), ptr(achieved), ptr(desired), ptr(reward), ptr(done), ptr(info), ptr(terminal_obs)))

    def reset_host(self, obs=None, achieved=None, desired=None):
        ptr = lambda x: None if x is None else C.c_void_p(x.ctypes.data)  # noqa: E731
        _check(self._lib.grs_reset_host(self._h, ptr(obs), ptr(achieved), ptr(desired)))

    def substep(self, n=1):
        """n x physics.step() with the controls currently in the state (robot_env.py:100)."""
        _check(self._lib.grs_substep(self._h, int(n), self._stream()))

    def synchronize(self):
        self._torch.cuda.current_stream(self.device).synchronize()
        self._torch.cuda.synchronize(self.device)

    # ------------------------------------------------------------------ state access (parity tests, checkpoints)
    def get_state(self):
        N = self.num_envs
        out = dict(qpos=np.zeros((N, NQ), np.float32), qvel=np.zeros((N, NV), np.float32), ctrl=np.zeros((N, NU), np.float32),
                   warmstart=np.zeros((N, NV), np.float32), flags=np.zeros((N, 3), np.int32), xfrc_z=np.zeros(N, np.float32))
        self.synchronize()
        _check(self._lib.grs_get_state(self._h, *[C.c_void_p(out[k].ctypes.data) for k in ("qpos", "qvel", "ctrl", "warmstart", "flags", "xfrc_z")]))
        return out

    def set_state(self, qpos=None, qvel=None, ctrl=None, warmstart=None, flags=None, xfrc_z=None):
        N = self.num_envs

        def prep(x, shape, dt):
            if x is None:
                return None
            a = np.ascontiguousarray(np.broadcast_to(np.asarray(x, dtype=dt), shape))
            return a
        arrs = [prep(qpos, (N, NQ), np.float32), prep(qvel, (N, NV), np.float32), prep(ctrl, (N, NU), np.float32),
                prep(warmstart, (N, NV), np.float32), prep(flags, (N, 3), np.int32), prep(xfrc_z, (N,), np.float32)]
        self.synchronize()
        _check(self._lib.grs_set_state(self._h, *[None if a is None else C.c_void_p(a.ctypes.data) for a in arrs]))

    def contacts(self):
        """physics.data.ncon / contact[i] at the current state: dict of numpy arrays, K = max contacts."""
        N, K = self.num_envs, self._lib.grs_max_contacts()
        out = dict(ncon=np.zeros(N, np.int32), geom=np.zeros((N, K, 2), np.int32), dist=np.zeros((N, K), np.float32),
                   pos=np.zeros((N, K, 3), np.float32), frame=np.zeros((N, K, 9), np.float32))
        self.synchronize()
        _check(self._lib.grs_get_contacts(self._h, *[C.c_void_p(out[k].ctypes.data) for k in ("ncon", "geom", "dist", "pos", "frame")]))
        return out

    def debug_step(self):
        """One physics.step() with the intermediate quantities dumped; returns a dict of numpy arrays per env."""
        self.synchronize()
        _check(self._lib.grs_debug_step(self._h))
        d = self.debug.cpu().numpy()
        N = self.num_envs
        ne = d[:, DBG["NEFC"]].astype(int)
        out = dict(M=d[:, DBG["M"]:DBG["M"] + 169].reshape(N, 13, 13), qfrc_bias=d[:, DBG["BIAS"]:DBG["BIAS"] + 13],
                   qfrc_smooth=d[:, DBG["FSMOOTH"]:DBG["FSMOOTH"] + 13], qacc_smooth=d[:, DBG["ASMOOTH"]:DBG["ASMOOTH"] + 13],
                   ncon=d[:, DBG["NCON"]].astype(int), nefc=ne, nlim=d[:, DBG["NLIM"]].astype(int), iters=d[:, DBG["ITERS"]].astype(int),
                   qacc=d[:, DBG["QACC"]:DBG["QACC"] + 13], qfrc_constraint=d[:, DBG["FCON"]:DBG["FCON"] + 13],
                   efc_D=d[:, DBG["D"]:DBG["D"] + 55], efc_aref=d[:, DBG["AREF"]:DBG["AREF"] + 55], efc_force=d[:, DBG["FORCE"]:DBG["FORCE"] + 55],
                   efc_J=d[:, DBG["J"]:DBG["J"] + 715].reshape(N, 55, 13), contact=d[:, DBG["CONTACT"]:DBG["CONTACT"] + 180].reshape(N, 12, 15),
                   mu=d[:, DBG["MU"]:DBG["MU"] + 12])
        return out

    def render(self, camera_id=2, width=64, height=64):
        """physics.render(camera_id, width, height) and the depth=True variant (sensor.py:64-73) for every
        environment: returns (rgb uint8 [N,h,w,3], depth float32 [N,h,w] metres) torch tensors on the device."""
        t = self._torch
        rgb = t.empty((self.num_envs, height, width, 3), dtype=t.uint8, device=self.device)
        depth = t.empty((self.num_envs, height, width), dtype=t.float32, device=self.device)
        _check(self._lib.grs_render(self._h, int(camera_id), int(width), int(height), C.c_void_p(rgb.data_ptr()), C.c_void_p(depth.data_ptr()), self._stream()))
        return rgb, depth

    @property
    def actions(self):
        """float32 [N, action_dim] view of the library's action buffer: the actions AsyncGripperEnv.send stored for each
        environment (row id), unchanged until the environment is sent again.  The synchronous step() need not write it."""
        N, a = self.num_envs, self.action_dim
        return self._tensor("actions", (N * 6,), "<f4")[:N * a].view(N, a)  # allocated N x 6, written with stride action_dim

    @property
    def launch_count(self):
        return int(self._lib.grs_launch_count(self._h))

    def step_kernel_ms(self, reset=True):
        return float(self._lib.grs_step_kernel_ms(self._h, int(reset)))
