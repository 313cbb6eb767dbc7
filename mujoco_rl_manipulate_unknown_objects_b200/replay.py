"""DeviceReplayBuffer — Python face of the device-resident HER replay buffer (grl_replay_* in include/b200_gripper_sim.h,
csrc/replay_kernels.cu).

Replaces SB3's HerReplayBuffer (train_agent.py:61-88) for the batched environments: transitions are written straight from the
simulator's device buffers and sampled, with "future" goal relabelling and the reward recomputed on the device, into device
tensors.  Differs from SB3 2.x in one respect: SB3 samples only from finished episodes, here every complete transition can be
sampled (a 400-step episode does not fit a 128-slot ring); a goal drawn for a running episode comes from its stored part.

Two write modes, fixed by the first begin call: lock-step (`begin` / `add`, every environment in every call) and indexed
(`begin_indexed` / `add_indexed`, the environments an AsyncGripperEnv.recv returned, each with its own count on the device).
"""
import ctypes as C

from . import _native
from ._native import INFO


class DeviceReplayBuffer:
    """`capacity` transitions per environment for `num_envs` environments, on one GPU.

    Storage views (torch tensors aliasing the library's memory, slot-major [capacity + 1, num_envs, ...]): obs, next_obs,
    actions, reward, done, info; `added` int64[num_envs] counts each environment's complete transitions in indexed mode.
    Calls run on torch's current stream."""

    def __init__(self, capacity, num_envs, obs_shape=(5, 64, 64), action_dim=6, her_reward=False, seed=0, device=0):
        import torch
        from .sim import NativeError
        self._torch = torch
        self._lib = _native.load()
        c, h, w = (int(x) for x in obs_shape)
        self._h = self._lib.grl_replay_create(int(capacity), int(num_envs), c, h, w, int(action_dim), int(bool(her_reward)),
                                              int(seed) & 0xFFFFFFFF, int(device))
        if not self._h:
            raise NativeError(self._lib.grl_last_error().decode())
        self.capacity, self.num_envs, self.obs_shape, self.action_dim = int(capacity), int(num_envs), (c, h, w), int(action_dim)
        self.her_reward, self.seed = bool(her_reward), int(seed)
        self.device = torch.device("cuda", int(device))
        self.begun = False  # begin() or begin_indexed() was called
        self.indexed = False  # the buffer is in indexed write mode
        self.draw = 0  # counter of sample() calls: the batch is a pure function of the buffer, seed, draw, size and her_ratio
        S, N = self.capacity + 1, self.num_envs
        self.obs = self._view("obs", (S, N, c, h, w), torch.uint8)
        self.next_obs = self._view("next_obs", (S, N, c, h, w), torch.uint8)
        self.actions = self._view("actions", (S, N, self.action_dim), torch.float32)
        self.reward = self._view("reward", (S, N), torch.float32)
        self.done = self._view("done", (S, N), torch.uint8)
        self.info = self._view("info", (S, N, INFO["STRIDE"]), torch.float32)
        self.added = self._view("added", (N,), torch.int64)
        self.nbytes = sum(t.numel() * t.element_size() for t in (self.obs, self.next_obs, self.actions, self.reward, self.done, self.info))

    def _check(self, rc):
        if rc != 0:
            from .sim import NativeError
            raise NativeError(self._lib.grl_last_error().decode())

    def _view(self, name, shape, dtype):
        from .sim import _DevArray
        p, sz = C.c_void_p(), C.c_uint64()
        self._check(self._lib.grl_replay_buffer(self._h, name.encode(), C.byref(p), C.byref(sz)))
        t = self._torch
        with t.cuda.device(self.device):
            raw = t.as_tensor(_DevArray(p.value, (int(sz.value),), "|u1"), device=self.device)
        return raw.view(dtype).reshape(shape)

    def _stream(self):
        return C.c_void_p(self._torch.cuda.current_stream(self.device).cuda_stream or 1)  # legacy default stream = 0x1

    def _ptr(self, x, dtype, shape):
        if x.device != self.device or x.dtype != dtype or not x.is_contiguous() or tuple(x.shape) != tuple(shape):
            raise ValueError("expected a contiguous %s tensor of shape %s on %s, got %s %s on %s" % (dtype, tuple(shape), self.device, x.dtype,
                                                                                                    tuple(x.shape), x.device))
        return C.c_void_p(x.data_ptr())

    # ------------------------------------------------------------------ filling
    def begin(self, obs):
        """Records obs u8[N, C, H, W], the observations the next actions are taken on: once before the first add() and after
        every explicit reset of the environments (which closes their open episodes)."""
        self._check(self._lib.grl_replay_begin(self._h, self._ptr(obs, self._torch.uint8, (self.num_envs,) + self.obs_shape), self._stream()))
        self.begun = True

    def begin_indexed(self):
        """Enters indexed write mode, for an asynchronous pool, after every AsyncGripperEnv.async_reset: closes the open
        episodes and disarms every environment, whose next listing in add_indexed() then records its observation."""
        self._check(self._lib.grl_replay_begin_indexed(self._h, self._stream()))
        self.begun = self.indexed = True

    def add(self, actions, reward, done, info, obs, terminal_obs):
        """One vectorised step, from the simulator's buffers after its step (GripperSim.actions / reward / done / info / obs /
        terminal_obs)."""
        t, N = self._torch, self.num_envs
        img = (N,) + self.obs_shape
        self._check(self._lib.grl_replay_add(self._h, self._ptr(actions, t.float32, (N, self.action_dim)), self._ptr(reward, t.float32, (N,)),
                                             self._ptr(done, t.uint8, (N,)), self._ptr(info, t.float32, (N, INFO["STRIDE"])),
                                             self._ptr(obs, t.uint8, img), self._ptr(terminal_obs, t.uint8, img), self._stream()))

    def add_indexed(self, env_ids, actions, reward, done, info, obs, terminal_obs):
        """The environments env_ids (int32 [n], an AsyncGripperEnv.recv batch; -1 entries are skipped) from the simulator's
        full per-environment buffers [N, ...] (GripperSim.actions / reward / done / info / obs / terminal_obs, read at row id).
        Out-of-range and duplicated ids are reported by status()."""
        t, N = self._torch, self.num_envs
        img = (N,) + self.obs_shape
        if env_ids.device != self.device or env_ids.dtype != t.int32 or not env_ids.is_contiguous() or env_ids.dim() != 1:
            raise ValueError("env_ids must be a contiguous 1-d int32 tensor on %s" % self.device)
        self._check(self._lib.grl_replay_add_indexed(self._h, C.c_void_p(env_ids.data_ptr()), env_ids.numel(),
                                                     self._ptr(actions, t.float32, (N, self.action_dim)), self._ptr(reward, t.float32, (N,)),
                                                     self._ptr(done, t.uint8, (N,)), self._ptr(info, t.float32, (N, INFO["STRIDE"])),
                                                     self._ptr(obs, t.uint8, img), self._ptr(terminal_obs, t.uint8, img), self._stream()))

    def status(self):
        """Synchronises and returns the complete transitions stored over all environments; raises NativeError if an indexed
        add or sample met a bad id or an empty buffer since the last call (the error is cleared by reporting it)."""
        n = C.c_int64()
        self._check(self._lib.grl_replay_status(self._h, C.byref(n)))
        return int(n.value)

    @property
    def transitions_per_env(self):
        """Lock-step mode only (raises in indexed mode, where the counts differ)."""
        n = int(self._lib.grl_replay_size(self._h))
        if n < 0:
            self._check(n)
        return n

    def __len__(self):
        """Complete transitions stored over all environments (synchronises in indexed mode)."""
        if self.indexed:
            return int(self.added.clamp(max=self.capacity).sum())
        return self.transitions_per_env * self.num_envs

    # ------------------------------------------------------------------ sampling
    def sample(self, batch_size, her_ratio=0.0, draw=None):
        """`batch_size` transitions as a dict of device tensors: obs, next_obs u8[B, C, H, W], actions f32[B, A], reward f32[B],
        done u8[B], desired_goal, achieved_goal f32[B, 2], info f32[B, 40], index i64[B] (flat slot * N + env into the storage
        views) and goal_index i64[B] (flat index of the transition the relabelled goal comes from, -1 if not relabelled).
        In indexed mode an empty buffer is not seen on the host: every row gets index -1 and status() raises.
        her_ratio: probability of "future" relabelling (SB3's n_sampled_goal=4 is 0.8).  draw: the sampling counter to use
        (default: the next one)."""
        t = self._torch
        B = int(batch_size)
        if draw is None:
            draw, self.draw = self.draw, self.draw + 1
        dev, n = self.device, max(B, 0)  # B <= 0 reaches the library, which rejects it
        out = dict(obs=t.empty((n,) + self.obs_shape, dtype=t.uint8, device=dev), next_obs=t.empty((n,) + self.obs_shape, dtype=t.uint8, device=dev),
                   actions=t.empty((n, self.action_dim), dtype=t.float32, device=dev), reward=t.empty(n, dtype=t.float32, device=dev),
                   done=t.empty(n, dtype=t.uint8, device=dev), desired_goal=t.empty((n, 2), dtype=t.float32, device=dev),
                   achieved_goal=t.empty((n, 2), dtype=t.float32, device=dev), info=t.empty((n, INFO["STRIDE"]), dtype=t.float32, device=dev),
                   index=t.empty(n, dtype=t.int64, device=dev), goal_index=t.empty(n, dtype=t.int64, device=dev))
        p = lambda k: C.c_void_p(out[k].data_ptr())  # noqa: E731
        self._check(self._lib.grl_replay_sample(self._h, B, float(her_ratio), int(draw), p("obs"), p("next_obs"), p("actions"), p("reward"), p("done"),
                                                p("desired_goal"), p("achieved_goal"), p("info"), p("index"), p("goal_index"), self._stream()))
        return out

    def close(self):
        if getattr(self, "_h", None):
            self._lib.grl_replay_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:  # noqa: BLE001
            pass
