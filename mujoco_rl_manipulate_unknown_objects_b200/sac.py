"""SACLearner — SB3's `SAC.train` (train_agent.py:61-88: batch 256, lr 3e-4, gamma 0.99, tau 0.005, automatic entropy
coefficient) on batches drawn from a DeviceReplayBuffer, with the rollouts on the tensor-core actor of RolloutWorker.

The networks follow SB3's `SACPolicy` as this project records it in the archive meta (sb3_io.write_sb3_zip): the actor is the
torch twin of GripperPolicy (policy.param_spec names: AugmentedNatureCNN features extractor -> latent_pi [256, 256] -> mu /
log_std), the critic is two Q networks `qf0` / `qf1` (514 features + action -> 256 -> 256 -> 1), and the features extractor is
shared with `share_features_extractor=True` semantics: the critic reads the actor's features without gradient, so the critic
loss does not update the extractor, while `critic_target` keeps its own polyak-averaged copy.  The reference's actual
`policy_kwargs` (train_agent.py:18-20) are not available to this project; net_arch [256, 256] and the shared extractor are
what its saved-archive meta states.

The backward pass is torch autograd (as in PPOLearner).  Actor, critic and entropy coefficient each have one FlatAdam (one
flat parameter / gradient bucket, one gradient all-reduce per gradient step, the fused grl_adam_step kernel), so on several
ranks the learners stay identical while every rank samples its own environments' buffer.
"""
from .rollout import FlatAdam, rank_seed


def build_sac_modules(channels=5, action_dim=6, n_flatten=1024):
    """(actor, critic, critic_target) torch modules with SB3's state-dict names (under the 'actor.', 'critic.' and
    'critic_target.' prefixes).  critic holds qf0 / qf1 only: its features come from the actor's extractor."""
    import math
    import torch
    from torch import nn

    def extractor():
        ext = nn.Module()
        ext.cnn = nn.Sequential(nn.Conv2d(channels - 1, 32, 8, 4), nn.ReLU(), nn.Conv2d(32, 64, 4, 2), nn.ReLU(), nn.Conv2d(64, 64, 3, 1), nn.ReLU(), nn.Flatten())
        ext.linear = nn.Sequential(nn.Linear(n_flatten, 512), nn.ReLU())
        return ext

    def q_net():
        return nn.Sequential(nn.Linear(514 + action_dim, 256), nn.ReLU(), nn.Linear(256, 256), nn.ReLU(), nn.Linear(256, 1))

    def features(ext, obs_u8):
        x = obs_u8.float() / 255.0
        return torch.cat((ext.linear(ext.cnn(x[:, :-1])), x[:, -1, 0, :2]), dim=1)

    class Actor(nn.Module):
        def __init__(self):
            super().__init__()
            self.features_extractor = extractor()
            self.latent_pi = nn.Sequential(nn.Linear(514, 256), nn.ReLU(), nn.Linear(256, 256), nn.ReLU())
            self.mu = nn.Linear(256, action_dim)
            self.log_std = nn.Linear(256, action_dim)

        def features(self, obs_u8):
            return features(self.features_extractor, obs_u8)

        def action_log_prob(self, feats, eps):
            """SquashedDiagGaussianDistribution.log_prob_from_params with the standard-normal sample `eps` given."""
            h = self.latent_pi(feats)
            mu, log_std = self.mu(h), torch.clamp(self.log_std(h), -20.0, 2.0)
            std = log_std.exp()
            g = mu + eps * std
            a = torch.tanh(g)
            logp = (-((g - mu) ** 2) / (2 * std ** 2) - std.log() - math.log(math.sqrt(2 * math.pi))).sum(dim=1)
            return a, logp - torch.log(1 - a ** 2 + 1e-6).sum(dim=1)

    class Critic(nn.Module):
        def __init__(self):
            super().__init__()
            self.qf0, self.qf1 = q_net(), q_net()

        def forward(self, feats, actions):
            x = torch.cat((feats, actions), dim=1)
            return self.qf0(x), self.qf1(x)

    class CriticTarget(Critic):
        def __init__(self):
            super().__init__()
            self.features_extractor = extractor()

        def forward(self, obs_u8, actions):
            return super().forward(features(self.features_extractor, obs_u8), actions)

    return Actor(), Critic(), CriticTarget()


class SACLearner:
    """SAC gradient steps for `worker`'s tensor-core actor on batches from `replay` (a DeviceReplayBuffer)."""

    def __init__(self, worker, replay, lr=3e-4, gamma=0.99, tau=0.005, batch_size=256, her_ratio=0.8, seed=0):
        import torch
        self.t, self.w, self.replay = torch, worker, replay
        torch.manual_seed(seed)  # identical initial weights on every rank
        dev = worker.device
        self.actor, self.critic, self.critic_target = (m.to(dev) for m in build_sac_modules(worker.sim.obs_shape[0], worker.sim.action_dim,
                                                                                                worker.policy.n_flatten))
        self.critic_target.features_extractor.load_state_dict(self.actor.features_extractor.state_dict())
        self.critic_target.qf0.load_state_dict(self.critic.qf0.state_dict())
        self.critic_target.qf1.load_state_dict(self.critic.qf1.state_dict())
        self.critic_target.requires_grad_(False)
        self.ent = torch.nn.Module()
        self.ent.log_ent_coef = torch.nn.Parameter(torch.zeros(1, device=dev))  # ent_coef "auto": initial value 1.0
        self.target_entropy = -float(worker.sim.action_dim)
        self.actor_opt, self.critic_opt, self.ent_opt = FlatAdam(self.actor, lr=lr), FlatAdam(self.critic, lr=lr), FlatAdam(self.ent, lr=lr)
        # polyak pairs in the order of zip(critic.parameters(), critic_target.parameters()) in SB3: the shared extractor first
        self._online = list(self.actor.features_extractor.parameters()) + list(self.critic.parameters())
        self._target = list(self.critic_target.features_extractor.parameters()) + list(self.critic_target.qf0.parameters()) + \
            list(self.critic_target.qf1.parameters())
        self.gamma, self.tau, self.batch_size, self.her_ratio = gamma, tau, batch_size, her_ratio
        self.gen = torch.Generator(device=dev).manual_seed(rank_seed(seed, worker.rank))
        self.sync_policy()

    @property
    def log_ent_coef(self):
        return self.ent.log_ent_coef

    def sync_policy(self):
        """The tensor-core rollout policy takes the actor's current weights."""
        self.w.policy.load_state_dict(self.actor.state_dict())

    def gradient_step(self, batch, noise=None):
        """One gradient step of SAC.train on `batch` (a DeviceReplayBuffer.sample dict).  noise: (eps_pi, eps_next), the
        standard-normal samples f32[B, A] of the reparametrised actions for obs and next_obs; drawn from the learner's
        generator when None.  Returns the detached losses (actor, critic, entropy coefficient) and the entropy coefficient."""
        t = self.t
        obs, next_obs = batch["obs"], batch["next_obs"]
        B, A = batch["actions"].shape
        if noise is None:
            noise = (t.randn((B, A), device=obs.device, generator=self.gen), t.randn((B, A), device=obs.device, generator=self.gen))
        eps_pi, eps_next = noise
        reward, done = batch["reward"].reshape(-1, 1), batch["done"].float().reshape(-1, 1)
        feats = self.actor.features(obs)
        actions_pi, log_prob = self.actor.action_log_prob(feats, eps_pi)
        log_prob = log_prob.reshape(-1, 1)
        ent_coef = t.exp(self.log_ent_coef.detach())
        ent_coef_loss = -(self.log_ent_coef * (log_prob + self.target_entropy).detach()).mean()
        self.ent_opt.zero_grad()
        ent_coef_loss.backward()
        self.ent_opt.step(self.ent_opt.all_reduce())
        with t.no_grad():
            next_actions, next_log_prob = self.actor.action_log_prob(self.actor.features(next_obs), eps_next)
            next_q = t.min(t.cat(self.critic_target(next_obs, next_actions), dim=1), dim=1, keepdim=True)[0]
            next_q = next_q - ent_coef * next_log_prob.reshape(-1, 1)
            target_q = reward + (1 - done) * self.gamma * next_q
        feats = feats.detach()  # share_features_extractor: the critic sees the actor's features without gradient
        critic_loss = 0.5 * sum(t.nn.functional.mse_loss(q, target_q) for q in self.critic(feats, batch["actions"]))
        self.critic_opt.zero_grad()
        critic_loss.backward()
        self.critic_opt.step(self.critic_opt.all_reduce())
        min_qf_pi = t.min(t.cat(self.critic(feats, actions_pi), dim=1), dim=1, keepdim=True)[0]
        actor_loss = (ent_coef * log_prob - min_qf_pi).mean()
        self.actor_opt.zero_grad()
        actor_loss.backward()
        self.actor_opt.step(self.actor_opt.all_reduce())
        with t.no_grad():
            t._foreach_mul_(self._target, 1.0 - self.tau)
            t._foreach_add_(self._target, self._online, alpha=self.tau)
        return t.stack([actor_loss.detach(), critic_loss.detach(), ent_coef_loss.detach(), ent_coef.reshape(())])

    def update(self, gradient_steps):
        """`gradient_steps` SAC gradient steps on fresh batches (batch_size, her_ratio) from the replay buffer, then the rollout
        policy takes the new actor.  Returns the mean losses."""
        out = [self.gradient_step(self.replay.sample(self.batch_size, self.her_ratio)) for _ in range(int(gradient_steps))]
        self.sync_policy()
        if not out:
            return {}
        m = self.t.stack(out).mean(dim=0).tolist()
        return dict(actor_loss=m[0], critic_loss=m[1], ent_coef_loss=m[2], ent_coef=m[3])

    def q_values(self, obs, actions):
        """(qf0, qf1) of the critic on u8 observations and actions (no gradient)."""
        with self.t.no_grad():
            return self.critic(self.actor.features(obs), actions)

    # ------------------------------------------------------------------ SB3 archives
    def sb3_state_dict(self):
        """The policy state dict under SB3's names: actor.*, critic.* (the shared extractor appears as
        critic.features_extractor.*) and critic_target.*."""
        cpu = lambda m, pre: {pre + k: v.detach().cpu() for k, v in m.state_dict().items()}  # noqa: E731
        sd = cpu(self.actor, "actor.")
        sd.update(cpu(self.actor.features_extractor, "critic.features_extractor."))
        sd.update(cpu(self.critic, "critic."))
        sd.update(cpu(self.critic_target, "critic_target."))
        return sd

    def save_sb3_zip(self, path, data=None):
        """Writes actor.*, critic.* and critic_target.* as a stable-baselines3 archive.  The entropy coefficient and the
        optimiser moments are not part of it."""
        from .sb3_io import write_sb3_zip
        sd = self.sb3_state_dict()
        actor = {k[len("actor."):]: v.numpy() for k, v in sd.items() if k.startswith("actor.")}
        return write_sb3_zip(path, actor, data=data, extra_state={k: v.numpy() for k, v in sd.items() if not k.startswith("actor.")})

    def load_sb3_zip(self, path):
        """Restores actor, critic and critic_target from an archive written by save_sb3_zip (or SB3's SAC with this
        architecture) into the optimisers' buckets, then syncs the rollout policy.  Returns the archive's data dict."""
        from .sb3_io import read_sb3_zip
        sd, data = read_sb3_zip(path)
        for m, pre in ((self.actor, "actor."), (self.critic, "critic."), (self.critic_target, "critic_target.")):
            m.load_state_dict({k: sd[pre + k] for k in m.state_dict()})  # copies into the existing (bucket-view) parameters
        self.sync_policy()
        return data

    def checksum(self):
        """float64 sum of every learner parameter (equal on all ranks while the ranks stay in step)."""
        parts = [self.actor_opt.flat, self.critic_opt.flat, self.ent_opt.flat] + [p.reshape(-1) for p in self.critic_target.parameters()]
        return float(sum(p.double().sum() for p in parts))
