"""GripperPolicy — Python face of the tensor-core policy forward (grp_* in include/b200_gripper_sim.h).

Replaces, for a whole batch of observations, the per-step `model.predict(obs, deterministic=True)` of the reference
(eval_agent.py:57): SB3 `preprocess_obs` (/255) -> `AugmentedNatureCNN` (models/feature_extractor.py:19-49) -> SAC actor
`latent_pi` [256, 256] (train_agent.py:18-20) -> `mu` / `log_std` -> tanh.  The parameters keep the torch / SB3
`state_dict` names and shapes, so a trained `best_model.zip` policy loads without conversion (`load_state_dict`).

All arithmetic happens in the CUDA library (tcgen05 / TMEM kernels); torch only carries device memory and streams.
"""
import ctypes as C
import math

import numpy as np

from . import _native

# (state_dict suffix, shape builder) in the flat order of grp_set_params
def param_spec(channels=5, action_dim=6, n_flatten=1024):
    cin = channels - 1
    return [("features_extractor.cnn.0.weight", (32, cin, 8, 8)), ("features_extractor.cnn.0.bias", (32,)),
            ("features_extractor.cnn.2.weight", (64, 32, 4, 4)), ("features_extractor.cnn.2.bias", (64,)),
            ("features_extractor.cnn.4.weight", (64, 64, 3, 3)), ("features_extractor.cnn.4.bias", (64,)),
            ("features_extractor.linear.0.weight", (512, n_flatten)), ("features_extractor.linear.0.bias", (512,)),
            ("latent_pi.0.weight", (256, 514)), ("latent_pi.0.bias", (256,)),
            ("latent_pi.2.weight", (256, 256)), ("latent_pi.2.bias", (256,)),
            ("mu.weight", (action_dim, 256)), ("mu.bias", (action_dim,)),
            ("log_std.weight", (action_dim, 256)), ("log_std.bias", (action_dim,))]


def init_params(channels=5, action_dim=6, n_flatten=1024, seed=0):
    """Random initialisation with torch's default nn.Conv2d / nn.Linear scheme (kaiming-uniform(a=sqrt 5) weights,
    U(-1/sqrt(fan_in), 1/sqrt(fan_in)) biases) — what SB3's SAC uses (no orthogonal init).  numpy only."""
    rng = np.random.default_rng(seed)
    out = {}
    for name, shape in param_spec(channels, action_dim, n_flatten):
        if name.endswith("weight"):
            fan_in = int(np.prod(shape[1:]))
            last_fan_in = fan_in
        bound = 1.0 / math.sqrt(last_fan_in)
        out[name] = rng.uniform(-bound, bound, shape).astype(np.float32)
    return out


class GripperPolicy:
    """Actor of the reference's SAC `MultiInputPolicy` with the AugmentedNatureCNN extractor, batched on one GPU."""

    def __init__(self, max_envs, obs_shape=(5, 64, 64), action_dim=6, device=0, params=None, seed=0):
        import torch
        if not torch.cuda.is_available():
            raise RuntimeError("no CUDA device: the policy forward has no CPU fallback")
        self._torch = torch
        self._lib = _native.load()
        self.device_index = int(device)
        self.device = torch.device("cuda", self.device_index)
        c, h, w = (int(x) for x in obs_shape)
        self._h = self._lib.grp_create(int(max_envs), c, h, w, int(action_dim), self.device_index)
        if not self._h:
            raise RuntimeError(self._lib.grp_last_error().decode())
        self.max_envs, self.obs_shape, self.action_dim = int(max_envs), (c, h, w), int(action_dim)
        sh = (C.c_int32 * 10)()
        self._lib.grp_shape(self._h, sh)
        self.n_flatten = 64 * sh[7] * sh[8]
        self.spec = param_spec(c, self.action_dim, self.n_flatten)
        assert sum(int(np.prod(s)) for _, s in self.spec) == self._lib.grp_num_params(self._h)
        self.mu = self._tensor("mu", (self.max_envs, self.action_dim), torch.float32)
        self.log_std = self._tensor("log_std", (self.max_envs, self.action_dim), torch.float32)
        self.features = self._tensor("features", (self.max_envs, 576), torch.bfloat16)
        self.load_state_dict(params if params is not None else init_params(c, self.action_dim, self.n_flatten, seed))

    def _check(self, rc):
        if rc != 0:
            raise RuntimeError(self._lib.grp_last_error().decode())

    def _tensor(self, name, shape, dtype):
        from .sim import _DevArray
        p, sz = C.c_void_p(), C.c_uint64()
        self._check(self._lib.grp_buffer(self._h, name.encode(), C.byref(p), C.byref(sz)))
        t = self._torch
        with t.cuda.device(self.device):
            raw = t.as_tensor(_DevArray(p.value, (int(sz.value),), "|u1"), device=self.device)
        return raw.view(dtype).reshape(shape)

    def buffer(self, name, shape, dtype):
        """Intermediate activation of the last forward ("act1", "act2", "act3": bf16 NHWC) as a torch tensor (tests)."""
        return self._tensor(name, shape, dtype)

    # ------------------------------------------------------------------ parameters
    def load_state_dict(self, sd, prefix=None):
        """`sd`: mapping name -> array/tensor.  Names may carry the SB3 prefix ('actor.'): the first prefix under which
        every parameter is found is used."""
        def get(name):
            for pre in ((prefix,) if prefix is not None else ("", "actor.", "policy.actor.")):
                if pre + name in sd:
                    return sd[pre + name]
            raise KeyError("parameter %r not found in the state dict" % name)
        flat = []
        for name, shape in self.spec:
            v = get(name)
            v = v.detach().cpu().numpy() if hasattr(v, "detach") else np.asarray(v)
            if tuple(v.shape) != tuple(shape):
                raise ValueError("parameter %s has shape %s, expected %s" % (name, tuple(v.shape), tuple(shape)))
            flat.append(np.ascontiguousarray(v, dtype=np.float32).ravel())
        flat = np.concatenate(flat)
        self._check(self._lib.grp_set_params(self._h, C.c_void_p(flat.ctypes.data), flat.size))

    def load_sb3_zip(self, path):
        """Loads the actor of a stable-baselines3 SAC archive (reference eval_agent.py:34-48: `SAC.load(best_model, ...)`)."""
        from .sb3_io import read_sb3_zip
        sd, data = read_sb3_zip(path)
        self.load_state_dict(sd, prefix="actor.")
        return data

    def save_sb3_zip(self, path, data=None):
        """Writes the actor's parameters as a stable-baselines3 archive (policy.pth with 'actor.*' names)."""
        from .sb3_io import write_sb3_zip
        return write_sb3_zip(path, self.state_dict(), data=data)

    def state_dict(self):
        n = self._lib.grp_num_params(self._h)
        flat = np.zeros(n, np.float32)
        self._check(self._lib.grp_get_params(self._h, C.c_void_p(flat.ctypes.data), n))
        out, o = {}, 0
        for name, shape in self.spec:
            k = int(np.prod(shape))
            out[name] = flat[o:o + k].reshape(shape).copy()
            o += k
        return out

    # ------------------------------------------------------------------ forward
    def forward(self, obs, deterministic=True, noise=None, out=None):
        """obs: uint8 [n, C, H, W] on the device.  Returns actions float32 [n, A] in [-1, 1] (device).
        deterministic=False draws noise ~ N(0, 1) with torch unless `noise` [n, A] is given."""
        t = self._torch
        if obs.dtype != t.uint8 or obs.device != self.device or not obs.is_contiguous():
            raise ValueError("obs must be a contiguous uint8 tensor on %s" % self.device)
        n = obs.shape[0]
        if tuple(obs.shape[1:]) != self.obs_shape:
            raise ValueError("obs must have shape (n, %d, %d, %d)" % self.obs_shape)
        if out is None:
            out = t.empty((n, self.action_dim), dtype=t.float32, device=self.device)
        if not deterministic and noise is None:
            noise = t.randn((n, self.action_dim), dtype=t.float32, device=self.device)
        npx = None
        if noise is not None:
            noise = noise.to(device=self.device, dtype=t.float32).contiguous()
            npx = C.c_void_p(noise.data_ptr())
        stream = C.c_void_p(t.cuda.current_stream(self.device).cuda_stream or 1)
        self._check(self._lib.grp_forward(self._h, C.c_void_p(obs.data_ptr()), C.c_void_p(out.data_ptr()), npx, int(n), stream))
        return out

    __call__ = forward

    def predict(self, obs, deterministic=True):
        """SB3 `predict`-style convenience for host observations: numpy uint8 [n, C, H, W] (or the VecEnv obs dict) ->
        numpy actions [n, A]."""
        t = self._torch
        if isinstance(obs, dict):
            obs = obs["observation"]
        o = t.as_tensor(np.ascontiguousarray(obs), device=self.device)
        return self.forward(o, deterministic=deterministic).cpu().numpy(), None

    @property
    def launch_count(self):
        return int(self._lib.grp_launch_count(self._h))

    def close(self):
        if getattr(self, "_h", None):
            self._lib.grp_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:  # noqa: BLE001
            pass
