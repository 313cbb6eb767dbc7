"""Device-resident rollouts and the multi-GPU plumbing around them (SURVEY.md §8e, §8f-N1).

Environments are independent, so they shard across ranks with no data-path collective: rank r of W owns the global
environment indices [r*N, (r+1)*N) and seeds its generators with seed + r.  torch.distributed (NCCL on the GPUs, gloo in the
CPU tests) carries only
  * the rollout statistics — one small SUM all-reduce per rollout, and
  * the policy gradient — one flat fp32 bucket (~1.0 M parameters = 4 MB) per optimiser step.

`RolloutWorker` keeps the whole loop on the GPU: tensor-core policy forward (GripperPolicy) -> fused environment step
(GripperSim) -> observation, with no host copy.  `PPOLearner` is the minimal learner BASELINE.json's config 4 asks for
("full PPO rollout loop ... with NCCL gradient allreduce"); the reference itself trains with SB3's SAC on one environment
(train_agent.py:61-88), so the learner has no reference counterpart and uses torch autograd for the backward pass — only the
rollout forward is on the hand-written kernels.
"""
import numpy as np

from ._native import INFO

STAT_NAMES = ("transitions", "substeps", "reward_sum", "episodes", "episode_return_sum", "episode_length_sum", "fails",
              "line_distance_sum", "total_distance_sum", "grasps")


# ---------------------------------------------------------------------------------------------- sharding
def shard_range(total_envs, rank, world):
    """Contiguous, balanced split of `total_envs` global environment indices: returns (start, stop) for `rank`."""
    if world <= 0 or not 0 <= rank < world:
        raise ValueError("rank %r outside world %r" % (rank, world))
    base, extra = divmod(int(total_envs), world)
    start = rank * base + min(rank, extra)
    return start, start + base + (1 if rank < extra else 0)


def rank_seed(seed, rank):
    return int(seed) + int(rank)


def dist_info():
    """(rank, world, local_rank) from torch.distributed when initialised, else from the torchrun environment."""
    import os
    try:
        import torch.distributed as dist
        if dist.is_available() and dist.is_initialized():
            return dist.get_rank(), dist.get_world_size(), int(os.environ.get("LOCAL_RANK", "0"))
    except Exception:  # noqa: BLE001
        pass
    return int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1")), int(os.environ.get("LOCAL_RANK", "0"))


# ---------------------------------------------------------------------------------------------- statistics
class RolloutStats:
    """Running sums of the per-step info records, kept on the device the records live on (float64)."""

    def __init__(self, device):
        import torch
        self._t = torch
        self.v = torch.zeros(len(STAT_NAMES), dtype=torch.float64, device=device)

    def update(self, info, reward, done, weight=None):
        """info f32[N, 40] (GRS_INFO_* layout), reward f32[N], done u8/bool[N] of one vectorised step.  weight (optional,
        [N]): each row counts weight times (0 leaves a row out without boolean indexing, which would synchronise)."""
        t, I = self._t, INFO
        if weight is not None:
            w = weight.to(t.float64)
            d = done.to(t.float64) * w
            n = w.sum()
            total = lambda x: (x.to(t.float64) * w).sum()  # noqa: E731
            nsub = total(info[:, I["NSUB_A"]:I["NSUB_A"] + 3].sum(1, dtype=t.float64))
        else:
            d = done.to(t.float64)
            n = t.tensor(float(info.shape[0]), dtype=t.float64, device=info.device)
            total = lambda x: x.sum(dtype=t.float64)  # noqa: E731
            nsub = info[:, I["NSUB_A"]:I["NSUB_A"] + 3].sum(dtype=t.float64)
        row = t.stack([
            n, nsub, total(reward), d.sum(),
            (info[:, I["EPISODE_RETURN"]].to(t.float64) * d).sum(), (info[:, I["EPISODE_STEP"]].to(t.float64) * d).sum(),
            ((info[:, I["STATUS"]] == 1).to(t.float64) * d).sum(), total(info[:, I["LINE_DISTANCE"]]),
            total(info[:, I["TOTAL_DISTANCE"]]), total(info[:, I["GRASP"]] == 3)])
        self.v += row

    def all_reduce(self):
        """SUM over ranks (no-op without an initialised process group).  Returns self."""
        import torch.distributed as dist
        if dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1:
            dist.all_reduce(self.v, op=dist.ReduceOp.SUM)
        return self

    def as_dict(self):
        v = self.v.detach().cpu().numpy()
        d = dict(zip(STAT_NAMES, v.tolist()))
        ep = max(d["episodes"], 1.0)
        d["mean_episode_return"] = d["episode_return_sum"] / ep
        d["mean_episode_length"] = d["episode_length_sum"] / ep
        d["mean_reward"] = d["reward_sum"] / max(d["transitions"], 1.0)
        d["substeps_per_transition"] = d["substeps"] / max(d["transitions"], 1.0)
        return d


def allreduce_flat_(tensors, average=True):
    """One collective for a list of tensors (gradients): flatten into a single bucket, SUM all-reduce, scatter back."""
    import torch
    import torch.distributed as dist
    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size() == 1 or not tensors:
        return
    flat = torch.cat([t.reshape(-1) for t in tensors])
    dist.all_reduce(flat, op=dist.ReduceOp.SUM)
    if average:
        flat /= dist.get_world_size()
    o = 0
    for t in tensors:
        n = t.numel()
        t.copy_(flat[o:o + n].view_as(t))
        o += n


# ---------------------------------------------------------------------------------------------- rollout worker
class RolloutWorker:
    """This rank's shard of the environments plus the policy, everything resident on one GPU."""

    def __init__(self, config, envs_per_gpu, device=0, seed=0, policy_params=None, total_envs=None):
        import torch
        from .policy import GripperPolicy
        from .sim import GripperSim
        rank, world, _ = dist_info()
        self.rank, self.world = rank, world
        self.global_range = shard_range(total_envs, rank, world) if total_envs is not None else (rank * envs_per_gpu, (rank + 1) * envs_per_gpu)
        n = self.global_range[1] - self.global_range[0]
        self.sim = GripperSim(config, num_envs=n, device=device, auto_reset=True)
        self.policy = GripperPolicy(max_envs=n, obs_shape=self.sim.obs_shape, action_dim=self.sim.action_dim, device=device, params=policy_params, seed=seed)
        self.device = self.sim.device
        self.gen = torch.Generator(device=self.device).manual_seed(rank_seed(seed, rank))
        self.actions = torch.zeros((n, self.sim.action_dim), dtype=torch.float32, device=self.device)
        self.noise = torch.zeros_like(self.actions)
        self.sim.reset()

    def collect(self, n_steps, deterministic=False, storage=None, random_actions=False, replay=None):
        """n_steps vectorised transitions.  storage (optional dict of preallocated tensors [T, N, ...]: obs, actions, rewards,
        dones, mu, log_std, noise) receives the trajectory.  replay (optional DeviceReplayBuffer over this worker's
        environments) receives every transition right after the step; a buffer not yet begun records the current observations
        first (replay.begin()).  Returns RolloutStats (local; call .all_reduce())."""
        t = self.sim._torch
        stats = RolloutStats(self.device)
        if replay is not None and not replay.begun:
            replay.begin(self.sim.obs)
        for k in range(n_steps):
            if storage is not None:
                storage["obs"][k].copy_(self.sim.obs)
            if random_actions:
                self.actions.copy_(t.rand(self.actions.shape, device=self.device, generator=self.gen) * 2 - 1)
            else:
                if not deterministic:
                    self.noise.normal_(generator=self.gen)
                self.policy.forward(self.sim.obs, deterministic=deterministic, noise=None if deterministic else self.noise, out=self.actions)
            self.sim.step(self.actions)
            if replay is not None:
                s = self.sim
                replay.add(self.actions, s.reward, s.done, s.info, s.obs, s.terminal_obs)
            stats.update(self.sim.info, self.sim.reward, self.sim.done)
            if storage is not None:
                storage["actions"][k].copy_(self.actions)
                storage["rewards"][k].copy_(self.sim.reward)
                storage["dones"][k].copy_(self.sim.done)
                if not random_actions:
                    n = self.actions.shape[0]
                    storage["mu"][k].copy_(self.policy.mu[:n])
                    storage["log_std"][k].copy_(self.policy.log_std[:n])
                    storage["noise"][k].copy_(self.noise)
        return stats

    def start_async(self, batch_size, replay=None):
        """Switches the worker to an asynchronous pool over its simulator (AsyncGripperEnv, batch `batch_size`): resets every
        environment and, with a replay buffer, enters its indexed write mode (DeviceReplayBuffer.begin_indexed)."""
        from .async_env import AsyncGripperEnv
        t = self.sim._torch
        if getattr(self, "pool", None) is not None:
            self.pool.async_end()  # a restart needs every environment received first
        self.pool = AsyncGripperEnv(self.sim, batch_size)
        self.pool.async_reset()
        if replay is not None:
            replay.begin_indexed()
        # stepped[n]: environment n has completed an agent step since async_reset (its first return is the reset observation);
        # entry N takes the -1 ids of a short recv
        self._stepped = t.zeros(self.sim.num_envs + 1, dtype=t.bool, device=self.device)

    def collect_async(self, n_recv, deterministic=False, replay=None):
        """n_recv rounds of the pool started by start_async: recv the next batch, add it to `replay` (optional, indexed mode)
        straight from the simulator's per-environment buffers, count it, run the policy on its observations and send the
        actions.  No host synchronisation.  The statistics cover the returned rows that end an agent step, not the first
        return of each environment after start_async.  Returns RolloutStats (local; call .all_reduce())."""
        t, s = self.sim._torch, self.sim
        stats = RolloutStats(self.device)
        B = self.pool.batch_size
        for _ in range(n_recv):
            r = self.pool.recv()
            ids = r["env_id"]
            if replay is not None:
                replay.add_indexed(ids, s.actions, s.reward, s.done, s.info, s.obs, s.terminal_obs)
            slot = t.where(ids >= 0, ids.long(), s.num_envs)
            stats.update(r["info"], r["reward"], r["done"], weight=self._stepped[slot] & (ids >= 0))
            self._stepped[slot] = True
            act, noise = self.actions[:B], self.noise[:B]
            if not deterministic:
                noise.normal_(generator=self.gen)
            self.policy.forward(r["obs"], deterministic=deterministic, noise=None if deterministic else noise, out=act)
            self.pool.send(act, ids)
        return stats

    def make_storage(self, n_steps):
        t = self.sim._torch
        n, a = self.actions.shape
        f = lambda *s: t.zeros(s, dtype=t.float32, device=self.device)  # noqa: E731
        return dict(obs=t.zeros((n_steps, n) + tuple(self.sim.obs_shape), dtype=t.uint8, device=self.device), actions=f(n_steps, n, a),
                    rewards=f(n_steps, n), dones=t.zeros((n_steps, n), dtype=t.uint8, device=self.device), mu=f(n_steps, n, a),
                    log_std=f(n_steps, n, a), noise=f(n_steps, n, a))

    def close(self):
        self.policy.close()
        self.sim.close()


# ---------------------------------------------------------------------------------------------- minimal PPO learner
def build_actor_critic(channels=5, action_dim=6, n_flatten=1024):
    """torch twin of the rollout policy (same parameter names as GripperPolicy.spec) plus a value head; used for the
    backward pass only."""
    import torch
    from torch import nn

    class ActorCritic(nn.Module):
        def __init__(self):
            super().__init__()
            ext = nn.Module()
            ext.cnn = nn.Sequential(nn.Conv2d(channels - 1, 32, 8, 4), nn.ReLU(), nn.Conv2d(32, 64, 4, 2), nn.ReLU(), nn.Conv2d(64, 64, 3, 1), nn.ReLU(), nn.Flatten())
            ext.linear = nn.Sequential(nn.Linear(n_flatten, 512), nn.ReLU())
            self.features_extractor = ext
            self.latent_pi = nn.Sequential(nn.Linear(514, 256), nn.ReLU(), nn.Linear(256, 256), nn.ReLU())
            self.mu = nn.Linear(256, action_dim)
            self.log_std = nn.Linear(256, action_dim)
            self.value = nn.Sequential(nn.Linear(514, 256), nn.ReLU(), nn.Linear(256, 1))

        def forward(self, obs_u8):
            x = obs_u8.float() / 255.0
            f = self.features_extractor.linear(self.features_extractor.cnn(x[:, :-1]))
            f = torch.cat((f, x[:, -1, 0, :2]), dim=1)
            h = self.latent_pi(f)
            return self.mu(h), torch.clamp(self.log_std(h), -20.0, 2.0), self.value(f).squeeze(-1)

    return ActorCritic()


def gae_device(rewards, dones, values, gamma, lam, stream=None, want_moments=True):
    """GAE + returns by the library kernel grl_gae (csrc/train_kernels.cu).  rewards f32[T,N], dones u8[T,N], values f32[T+1,N]
    CUDA tensors -> (adv f32[T,N], ret f32[T,N], moments f64[2] = sum(adv), sum(adv^2))."""
    import ctypes as C
    import torch
    from . import _native
    T, N = rewards.shape
    assert rewards.is_cuda and rewards.dtype == torch.float32 and rewards.is_contiguous()
    assert dones.dtype == torch.uint8 and dones.is_contiguous() and tuple(dones.shape) == (T, N)
    assert values.dtype == torch.float32 and values.is_contiguous() and tuple(values.shape) == (T + 1, N)
    adv, ret = torch.empty_like(rewards), torch.empty_like(rewards)
    mom = torch.zeros(2, dtype=torch.float64, device=rewards.device) if want_moments else None
    st = stream if stream is not None else (torch.cuda.current_stream(rewards.device).cuda_stream or 1)
    L = _native.load()
    rc = L.grl_gae(C.c_void_p(rewards.data_ptr()), C.c_void_p(dones.data_ptr()), C.c_void_p(values.data_ptr()), C.c_void_p(adv.data_ptr()),
                   C.c_void_p(ret.data_ptr()), C.c_void_p(mom.data_ptr()) if mom is not None else None, T, N, float(gamma), float(lam), C.c_void_p(st))
    if rc != 0:
        raise RuntimeError(L.grl_last_error().decode())
    return adv, ret, mom


class FlatAdam:
    """Adam over ONE flat fp32 bucket.  The module's parameters and gradients are re-pointed at views of two flat CUDA arrays, so
    that (1) autograd accumulates straight into the bucket NCCL all-reduces — no concatenate before, no scatter after — and
    (2) the optimiser step is one fused kernel (grl_adam_step, csrc/train_kernels.cu) that also applies the 1/world averaging."""

    def __init__(self, module, lr=3e-4, betas=(0.9, 0.999), eps=1e-8, weight_decay=0.0):
        import torch
        params = [p for p in module.parameters() if p.requires_grad]
        dev = params[0].device
        sizes = [(p.numel() + 3) // 4 * 4 for p in params]  # every view starts 16-byte aligned
        total = sum(sizes)
        self.flat = torch.zeros(total, dtype=torch.float32, device=dev)
        self.grad = torch.zeros(total, dtype=torch.float32, device=dev)
        self.exp_avg, self.exp_avg_sq = torch.zeros_like(self.flat), torch.zeros_like(self.flat)
        o = 0
        for p, n in zip(params, sizes):
            self.flat[o:o + p.numel()].copy_(p.data.reshape(-1))
            p.data = self.flat[o:o + p.numel()].view_as(p.data)
            p.grad = self.grad[o:o + p.numel()].view_as(p.data)
            o += n
        self.params, self.count, self.step_count = params, total, 0
        self.lr, self.betas, self.eps, self.weight_decay = lr, betas, eps, weight_decay
        self.allreduce_ms = []  # device time of every gradient all-reduce (CUDA events on the launching stream)

    def zero_grad(self):
        self.grad.zero_()  # in place: the parameters keep their gradient views

    def all_reduce(self):
        """SUM all-reduce of the gradient bucket (one collective per optimiser step).  Returns the world size."""
        import torch
        import torch.distributed as dist
        if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size() == 1:
            return 1
        if self.grad.is_cuda:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            dist.all_reduce(self.grad, op=dist.ReduceOp.SUM)
            e1.record()
            self._pending = getattr(self, "_pending", []) + [(e0, e1)]
        else:
            dist.all_reduce(self.grad, op=dist.ReduceOp.SUM)
        return dist.get_world_size()

    def harvest_timings(self):
        import torch
        if getattr(self, "_pending", None):
            torch.cuda.synchronize(self.grad.device)
            self.allreduce_ms += [a.elapsed_time(b) for a, b in self._pending]
            self._pending = []
        return self.allreduce_ms

    def step(self, world=1):
        import ctypes as C
        import torch
        from . import _native
        for p in self.params:  # autograd must have accumulated in place
            assert p.grad is not None and p.grad.data_ptr() >= self.grad.data_ptr() and p.grad.data_ptr() < self.grad.data_ptr() + 4 * self.count, \
                "a parameter's gradient left the flat bucket (zero_grad(set_to_none=True) was called?)"
        self.step_count += 1
        L = _native.load()
        st = torch.cuda.current_stream(self.flat.device).cuda_stream or 1
        rc = L.grl_adam_step(C.c_void_p(self.flat.data_ptr()), C.c_void_p(self.grad.data_ptr()), C.c_void_p(self.exp_avg.data_ptr()),
                             C.c_void_p(self.exp_avg_sq.data_ptr()), self.count, self.step_count, float(self.lr), float(self.betas[0]), float(self.betas[1]),
                             float(self.eps), 1.0 / float(world), float(self.weight_decay), C.c_void_p(st))
        if rc != 0:
            raise RuntimeError(L.grl_last_error().decode())


class PPOLearner:
    """Clipped-surrogate PPO on trajectories collected by RolloutWorker (squashed-Gaussian policy; log-probabilities are taken
    on the pre-tanh sample, the tanh Jacobian cancels in the ratio).  Gradients are averaged over ranks in one flat bucket."""

    def __init__(self, worker, lr=3e-4, gamma=0.99, lam=0.95, clip=0.2, vf_coef=0.5, minibatch=2048, seed=0):
        import torch
        self.t, self.w = torch, worker
        torch.manual_seed(seed)  # identical initial weights on every rank
        c = worker.sim.obs_shape[0]
        self.net = build_actor_critic(c, worker.sim.action_dim, worker.policy.n_flatten).to(worker.device)
        self.opt = FlatAdam(self.net, lr=lr)  # flat parameter / gradient buckets + fused Adam kernel
        self.gamma, self.lam, self.clip, self.vf_coef, self.minibatch = gamma, lam, clip, vf_coef, minibatch
        self.sync_policy()

    def sync_policy(self):
        sd = {k: v for k, v in self.net.state_dict().items() if not k.startswith("value.")}
        self.w.policy.load_state_dict(sd)

    def update(self, storage, last_obs, epochs=1):
        t = self.t
        T, N = storage["rewards"].shape
        with t.no_grad():
            values = t.stack([self._values(storage["obs"][k]) for k in range(T)] + [self._values(last_obs)]).contiguous()
            # GAE + returns + the advantage moments in one kernel over the rollout storage (csrc/train_kernels.cu : k_gae)
            adv, ret, mom = gae_device(storage["rewards"], storage["dones"], values, self.gamma, self.lam)
            pre = storage["mu"] + t.exp(storage["log_std"]) * storage["noise"]
            logp_old = self._logp(storage["mu"], storage["log_std"], pre)
            cnt = float(T * N)
            mean = mom[0] / cnt
            std = t.sqrt(t.clamp(mom[1] - cnt * mean * mean, min=0.0) / max(cnt - 1.0, 1.0))  # unbiased, as torch.std
            adv = ((adv - mean.float()) / (std.float() + 1e-8))
        obs = storage["obs"].reshape((T * N,) + tuple(storage["obs"].shape[2:]))
        pre, logp_old, adv, ret = pre.reshape(T * N, -1), logp_old.reshape(-1), adv.reshape(-1), ret.reshape(-1)
        losses = []
        for _ in range(epochs):
            perm = t.randperm(T * N, device=obs.device)
            for s in range(0, T * N, self.minibatch):
                idx = perm[s:s + self.minibatch]
                mu, ls, v = self.net(obs[idx])
                ratio = t.exp(self._logp(mu, ls, pre[idx]) - logp_old[idx])
                pg = -t.min(ratio * adv[idx], t.clamp(ratio, 1 - self.clip, 1 + self.clip) * adv[idx]).mean()
                vf = ((v - ret[idx]) ** 2).mean()
                loss = pg + self.vf_coef * vf
                self.opt.zero_grad()
                loss.backward()                      # accumulates into the flat gradient bucket
                world = self.opt.all_reduce()        # ONE collective on that bucket (NCCL SUM)
                self.opt.step(world)                 # fused Adam, 1/world folded in
                losses.append(float(loss.detach()))
        self.sync_policy()
        return float(np.mean(losses)) if losses else 0.0

    def _values(self, obs):
        out = []
        for s in range(0, obs.shape[0], 4096):
            out.append(self.net(obs[s:s + 4096])[2])
        return self.t.cat(out)

    @staticmethod
    def _logp(mu, log_std, pre):
        return (-0.5 * ((pre - mu) / log_std.exp()) ** 2 - log_std - 0.9189385332046727).sum(-1)
