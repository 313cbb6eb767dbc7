"""Device-resident HER replay buffer (csrc/replay_kernels.cu, replay.DeviceReplayBuffer) and the SAC learner on top of it
(sac.SACLearner).  Storage is checked bit-exactly against the same rollout recorded in torch, sampled batches against torch
indexing of the storage views, relabelled rewards against BatchedRobotVecEnv.compute_reward, and one learner step against
SB3's SAC.train restated here with plain torch tensors and torch.optim.Adam."""
import math

import numpy as np
import pytest

N, CAP, STEPS = 64, 16, 40  # 40 steps wrap a 16-transition ring; time_horizon 6 ends several episodes per environment


def test_create_rejects_bad_sizes_and_needs_a_device():
    from mujoco_rl_manipulate_unknown_objects_b200 import _native
    L = _native.load()
    assert L.grl_replay_create(0, 4, 5, 64, 64, 6, 0, 0, 0) is None and b"capacity" in L.grl_last_error()
    assert L.grl_replay_create(4, 4, 3, 5, 5, 6, 0, 0, 0) is None and b"multiple of 16" in L.grl_last_error()
    assert L.grl_replay_sample(None, 8, 0.0, 0, *([None] * 10), None) != 0 and b"null" in L.grl_last_error()
    import torch
    if torch.cuda.is_available():
        return
    assert L.grl_replay_create(16, 64, 5, 64, 64, 6, 0, 0, 0) is None and b"CUDA" in L.grl_last_error()
    from mujoco_rl_manipulate_unknown_objects_b200.replay import DeviceReplayBuffer
    with pytest.raises(RuntimeError):
        DeviceReplayBuffer(16, 64)


def _rollout(her_buffer=True, im_reward=False, steps=STEPS, seed=3):
    """RolloutWorker with random actions feeding a DeviceReplayBuffer through collect(replay=...); every step also recorded in
    torch: obs the action was taken on, action, reward, done, info, next_obs and the post-step achieved_goal buffer."""
    import torch
    from mujoco_rl_manipulate_unknown_objects_b200 import make_config
    from mujoco_rl_manipulate_unknown_objects_b200.replay import DeviceReplayBuffer
    from mujoco_rl_manipulate_unknown_objects_b200.rollout import RolloutWorker
    # reset noise: every episode starts from its own object pose, so goals differ between episodes
    cfg = make_config(sim_env="/xmls/sugar_cube_env.xml", time_horizon=6, her_buffer=her_buffer, im_reward=im_reward, reset_noise_xy=0.02,
                      reset_noise_yaw=0.3, seed=seed)
    w = RolloutWorker(cfg, envs_per_gpu=N, seed=seed)
    rb = DeviceReplayBuffer(CAP, N, w.sim.obs_shape, w.sim.action_dim, her_reward=her_buffer, seed=7)
    rec = {k: [] for k in ("obs", "actions", "reward", "done", "info", "next_obs", "achieved_after")}
    for _ in range(steps):
        _record_step(w, rb, rec)
    return w, rb, rec


def _record_step(w, rb, rec):
    import torch
    before = w.sim.obs.clone()
    w.collect(1, random_actions=True, replay=rb)
    s = w.sim
    rec["obs"].append(before)
    rec["actions"].append(w.actions.clone())
    rec["reward"].append(s.reward.clone())
    rec["done"].append(s.done.clone())
    rec["info"].append(s.info.clone())
    rec["next_obs"].append(torch.where(s.done.bool()[:, None, None, None], s.terminal_obs, s.obs))
    rec["achieved_after"].append(s.achieved_goal.clone())


def _flat(rb):
    S = rb.capacity + 1
    return dict(obs=rb.obs.reshape(S * N, *rb.obs_shape), next_obs=rb.next_obs.reshape(S * N, *rb.obs_shape), actions=rb.actions.reshape(S * N, -1),
                reward=rb.reward.reshape(-1), done=rb.done.reshape(-1), info=rb.info.reshape(S * N, -1))


def _t_of(index, added):
    """Transition number of flat storage indices (slot * N + env) among the complete ones [added - CAP, added)."""
    slot = index // N
    S = CAP + 1
    base = added - CAP
    return base + (slot - base % S) % S


@pytest.mark.gpu
def test_storage_matches_the_recorded_rollout():
    import torch
    from mujoco_rl_manipulate_unknown_objects_b200._native import INFO
    w, rb, rec = _rollout()
    S = CAP + 1
    assert rb.transitions_per_env == CAP and len(rb) == CAP * N
    assert int(torch.stack(rec["done"]).sum(0).min()) >= 4  # every environment finished several episodes
    for t in range(STEPS - CAP, STEPS):
        s = t % S
        assert torch.equal(rb.obs[s], rec["obs"][t]), t
        assert torch.equal(rb.next_obs[s], rec["next_obs"][t]), t
        assert torch.equal(rb.actions[s], rec["actions"][t]) and torch.equal(rb.reward[s], rec["reward"][t])
        assert torch.equal(rb.done[s], rec["done"][t]) and torch.equal(rb.info[s], rec["info"][t])
    assert torch.equal(rb.obs[STEPS % S], w.sim.obs)  # the pending observation (its transition's action is not taken yet)
    # next_obs is the terminal observation on done, which differs from the reset observation the simulator returns
    d = torch.stack(rec["done"]).bool()
    assert all(not torch.equal(rec["next_obs"][t][d[t]], rec["obs"][t + 1][d[t]]) for t in range(STEPS - 1) if d[t].any())
    # the achieved goal is the transition's own (info), not the post-reset state of the simulator's achieved buffer
    ag_info = torch.stack(rec["info"])[..., INFO["ACHIEVED"]:INFO["ACHIEVED"] + 2]
    ag_after = torch.stack(rec["achieved_after"])
    assert (ag_info[d] != ag_after[d]).any(dim=-1).float().mean() > 0.9
    b = rb.sample(8192, 0.8)
    slot = b["index"] // N
    assert not (slot == STEPS % S).any() and not (b["goal_index"] // N == STEPS % S).any()  # the pending slot is never returned
    t_s = _t_of(b["index"], STEPS)
    ref_info = torch.stack(rec["info"])[t_s, b["index"] % N]
    assert torch.equal(b["info"], ref_info) and torch.equal(b["achieved_goal"], ref_info[:, INFO["ACHIEVED"]:INFO["ACHIEVED"] + 2])
    assert int(t_s.min()) == STEPS - CAP  # overwritten transitions are gone, the oldest complete one is still there
    w.close()
    rb.close()


@pytest.mark.gpu
def test_sampling_gathers_relabels_and_is_reproducible():
    import torch
    from mujoco_rl_manipulate_unknown_objects_b200._native import INFO
    w, rb, rec = _rollout()
    f = _flat(rb)
    A, D = INFO["ACHIEVED"], INFO["DESIRED"]
    b = rb.sample(4096, 0.8, draw=11)
    idx, gi = b["index"], b["goal_index"]
    for k in ("obs", "next_obs", "actions", "done", "info"):
        assert torch.equal(b[k], f[k][idx]), k
    rel = gi >= 0
    assert torch.equal(b["achieved_goal"], f["info"][idx, A:A + 2])
    assert torch.equal(b["desired_goal"][rel], f["info"][gi[rel], A:A + 2])
    assert torch.equal(b["desired_goal"][~rel], f["info"][idx[~rel], D:D + 2])
    assert torch.equal(b["reward"][~rel], f["reward"][idx[~rel]])
    # a pure function of (buffer, seed, draw, B, her_ratio)
    again = rb.sample(4096, 0.8, draw=11)
    assert all(torch.equal(b[k], again[k]) for k in b)
    assert not torch.equal(rb.sample(4096, 0.8, draw=12)["index"], idx)
    assert rb.draw == 0 and torch.equal(rb.sample(4096, 0.8)["index"], rb.sample(4096, 0.8, draw=0)["index"]) and rb.draw == 1
    # relabelled fraction within 5 sigma of her_ratio
    B = 16384
    for p in (0.0, 0.8, 1.0):
        s = rb.sample(B, p, draw=100)
        ok = (s["info"][:, INFO["FLAGS"]].int() & 2) == 0  # a step whose state went non-finite is never relabelled
        frac = float((s["goal_index"][ok] >= 0).float().mean())
        assert abs(frac - p) <= 5 * math.sqrt(p * (1 - p) / int(ok.sum())) + 1e-9, (p, frac)
        assert torch.isfinite(s["desired_goal"][ok]).all()
    # uniform environments and slots: loose chi-square bounds
    b = rb.sample(B, 0.8, draw=200)
    env_counts = torch.bincount(b["index"] % N, minlength=N).double()
    t_counts = torch.bincount(_t_of(b["index"], STEPS) - (STEPS - CAP), minlength=CAP).double()
    for c in (env_counts, t_counts):
        e = B / len(c)
        chi2, dof = float(((c - e) ** 2 / e).sum()), len(c) - 1
        assert chi2 < dof + 8 * math.sqrt(2 * dof), (chi2, dof)
    # goal source: same environment, same episode, at or after the sample, no later than the episode's done / newest transition
    idx, gi = b["index"], b["goal_index"]
    rel = gi >= 0
    assert torch.equal(gi[rel] % N, idx[rel] % N)
    t_s, t_g = _t_of(idx[rel], STEPS), _t_of(gi[rel], STEPS)
    assert (t_g >= t_s).all() and (t_g <= STEPS - 1).all()
    done = torch.stack(rec["done"]).long()  # [T, N]
    cs = torch.cat([torch.zeros((1, N), dtype=torch.long, device=done.device), done.cumsum(0)])  # dones strictly before t: cs[t]
    env = idx[rel] % N
    assert (cs[t_g, env] - cs[t_s, env] == 0).all()  # no done in [t_s, t_g)
    assert (t_g > t_s).any() and (done[t_g, env] == 1).any() and (done[t_g, env] == 0).any()
    w.close()
    rb.close()


@pytest.mark.gpu
def test_explicit_reset_closes_episodes_at_the_newest_transition():
    import torch
    w, rb, rec = _rollout(steps=20)
    w.sim.reset()
    rb.begin(w.sim.obs)
    for _ in range(3):
        _record_step(w, rb, rec)
    added = 23
    b = rb.sample(16384, 1.0, draw=5)
    rel = b["goal_index"] >= 0
    t_s, t_g = _t_of(b["index"][rel], added), _t_of(b["goal_index"][rel], added)
    old = t_s <= 19
    assert old.any() and (~old).any()
    assert (t_g[old] <= 19).all()  # an episode cut by the reset ends at the last transition before it
    assert (t_g[~old] >= 20).all()
    assert torch.equal(rb.obs[20 % (CAP + 1)], rec["obs"][20])  # the reset observation opened the new episode
    w.close()
    rb.close()


@pytest.mark.gpu
@pytest.mark.parametrize("her_buffer,im_reward", [(0, 0), (1, 0), (0, 1), (1, 1)])
def test_sampled_reward_equals_compute_reward(her_buffer, im_reward):
    import torch
    from mujoco_rl_manipulate_unknown_objects_b200 import BatchedRobotVecEnv
    from mujoco_rl_manipulate_unknown_objects_b200._native import INFO
    from mujoco_rl_manipulate_unknown_objects_b200.vec_env import LazyInfos
    w, rb, _ = _rollout(her_buffer=bool(her_buffer), im_reward=bool(im_reward), steps=20)
    env = BatchedRobotVecEnv(w.sim.config, num_envs=N, _sim=w.sim)
    b = {k: v.cpu().numpy() for k, v in rb.sample(512, 0.8, draw=3).items()}
    infos = LazyInfos(b["info"], b["done"].astype(bool), None, env.target_direction, 0.0, obs=b["next_obs"], prev_obs=b["obs"])
    ref = env.compute_reward(b["achieved_goal"], b["desired_goal"], infos)
    bad = (b["info"][:, INFO["FLAGS"]].astype(np.int32) & 2) != 0
    assert (b["reward"][bad] == 0).all()
    err = np.abs(ref - b["reward"])[~bad] / np.maximum(1.0, np.abs(ref[~bad]))
    assert err.max() <= 1e-5, (err.max(), int(np.argmax(err)))
    if her_buffer:  # relabelling changed some rewards
        rel = b["goal_index"] >= 0
        assert (b["desired_goal"][rel] != b["info"][rel, INFO["DESIRED"]:INFO["DESIRED"] + 2]).any()
    env.close()
    w.close()
    rb.close()


@pytest.mark.gpu
def test_bad_arguments_raise():
    import torch
    from mujoco_rl_manipulate_unknown_objects_b200.replay import DeviceReplayBuffer
    rb = DeviceReplayBuffer(4, 8)
    with pytest.raises(RuntimeError, match="no complete transition"):
        rb.sample(4)
    z = torch.zeros
    with pytest.raises(RuntimeError, match="begin"):
        rb.add(z((8, 6), device="cuda"), z(8, device="cuda"), z(8, dtype=torch.uint8, device="cuda"), z((8, 40), device="cuda"),
               z((8, 5, 64, 64), dtype=torch.uint8, device="cuda"), z((8, 5, 64, 64), dtype=torch.uint8, device="cuda"))
    obs = torch.zeros((8, 5, 64, 64), dtype=torch.uint8, device="cuda")
    rb.begin(obs)
    rb.add(z((8, 6), device="cuda"), z(8, device="cuda"), z(8, dtype=torch.uint8, device="cuda"), z((8, 40), device="cuda"), obs, obs)
    assert len(rb) == 8
    for B, p in ((0, 0.0), (-3, 0.0), (4, 1.5), (4, -0.1), (4, float("nan"))):
        with pytest.raises(RuntimeError):
            rb.sample(B, p)
    with pytest.raises(ValueError):
        rb.begin(obs[:4])
    rb.close()


# ---------------------------------------------------------------------------------------------------------------- learner
def _ref_features(p, pre, obs):
    import torch
    import torch.nn.functional as F
    x = obs.float() / 255.0
    h = x[:, :-1]
    for i, s in ((0, 4), (2, 2), (4, 1)):
        h = F.relu(F.conv2d(h, p[pre + "cnn.%d.weight" % i], p[pre + "cnn.%d.bias" % i], stride=s))
    h = F.relu(F.linear(h.flatten(1), p[pre + "linear.0.weight"], p[pre + "linear.0.bias"]))
    return torch.cat((h, x[:, -1, 0, :2]), dim=1)


def _ref_mlp(p, pre, x, layers):
    import torch.nn.functional as F
    for i in range(layers):
        x = F.linear(x, p[pre + "%d.weight" % (2 * i)], p[pre + "%d.bias" % (2 * i)])
        if i < layers - 1:
            x = F.relu(x)
    return x


def _ref_actor(p, feats, eps):
    """SB3 Actor.action_log_prob: SquashedDiagGaussianDistribution over the latent_pi head, sample mean + eps * std."""
    import torch
    import torch.nn.functional as F
    h = F.relu(_ref_mlp(p, "actor.latent_pi.", feats, 2))
    mean = F.linear(h, p["actor.mu.weight"], p["actor.mu.bias"])
    log_std = torch.clamp(F.linear(h, p["actor.log_std.weight"], p["actor.log_std.bias"]), -20, 2)
    dist = torch.distributions.Normal(mean, log_std.exp())
    g = mean + eps * log_std.exp()
    a = torch.tanh(g)
    return a, dist.log_prob(g).sum(dim=1) - torch.log(1 - a ** 2 + 1e-6).sum(dim=1)


def _ref_q(p, pre, feats, actions):
    x = __import__("torch").cat((feats, actions), dim=1)
    return [_ref_mlp(p, pre + "qf%d." % k, x, 3) for k in (0, 1)]


@pytest.mark.gpu
def test_sac_learner_step_matches_sb3_train_in_torch(tmp_path):
    import torch
    import torch.nn.functional as F
    from mujoco_rl_manipulate_unknown_objects_b200.policy import GripperPolicy
    from mujoco_rl_manipulate_unknown_objects_b200.sac import SACLearner
    from mujoco_rl_manipulate_unknown_objects_b200.sb3_io import read_sb3_zip
    w, rb, _ = _rollout(steps=10)
    # the two sides must see the same gradients: cuDNN's default weight-gradient algorithms sum in a varying order, and Adam's
    # first step (lr * g / (|g| + eps)) magnifies the last bits of the near-zero gradients of the first convolution
    torch.backends.cudnn.deterministic, torch.backends.cudnn.benchmark = True, False
    learner = SACLearner(w, rb, batch_size=64, seed=1)
    gamma, tau, lr, A = 0.99, 0.005, 3e-4, w.sim.action_dim
    p = {k: v.cuda().clone().requires_grad_(not k.startswith("critic_target.")) for k, v in learner.sb3_state_dict().items()}
    actor_keys = [k for k in p if k.startswith("actor.")]
    critic_keys = [k for k in p if k.startswith("critic.qf")]
    log_ent = torch.zeros(1, device="cuda", requires_grad=True)
    opt_a, opt_c, opt_e = (torch.optim.Adam([p[k] for k in actor_keys], lr=lr), torch.optim.Adam([p[k] for k in critic_keys], lr=lr),
                           torch.optim.Adam([log_ent], lr=lr))
    batch = rb.sample(64, 0.8, draw=9)
    g = torch.Generator(device="cuda").manual_seed(4)
    noise = (torch.randn((64, A), device="cuda", generator=g), torch.randn((64, A), device="cuda", generator=g))
    old_target = {k: v.detach().clone() for k, v in p.items() if k.startswith("critic_target.")}
    # --- SAC.train, one gradient step (stable_baselines3/sac/sac.py), share_features_extractor=True
    obs, nobs = batch["obs"], batch["next_obs"]
    rew, done = batch["reward"].reshape(-1, 1), batch["done"].float().reshape(-1, 1)
    actions_pi, log_prob = _ref_actor(p, _ref_features(p, "actor.features_extractor.", obs), noise[0])
    log_prob = log_prob.reshape(-1, 1)
    ent_coef = torch.exp(log_ent.detach())
    ent_loss = -(log_ent * (log_prob + (-A)).detach()).mean()
    opt_e.zero_grad(); ent_loss.backward(); opt_e.step()
    with torch.no_grad():
        na, nlp = _ref_actor(p, _ref_features(p, "actor.features_extractor.", nobs), noise[1])
        nq = torch.min(torch.cat(_ref_q(p, "critic_target.", _ref_features(p, "critic_target.features_extractor.", nobs), na), dim=1), dim=1, keepdim=True)[0]
        target_q = rew + (1 - done) * gamma * (nq - ent_coef * nlp.reshape(-1, 1))
    with torch.no_grad():
        feats = _ref_features(p, "actor.features_extractor.", obs)
    critic_loss = 0.5 * sum(F.mse_loss(q, target_q) for q in _ref_q(p, "critic.", feats, batch["actions"]))
    opt_c.zero_grad(); critic_loss.backward(); opt_c.step()
    min_qf_pi = torch.min(torch.cat(_ref_q(p, "critic.", feats, actions_pi), dim=1), dim=1, keepdim=True)[0]
    actor_loss = (ent_coef * log_prob - min_qf_pi).mean()
    opt_a.zero_grad(); actor_loss.backward(); opt_a.step()
    with torch.no_grad():
        for k in old_target:
            src = "actor." + k[len("critic_target."):] if ".features_extractor." in k else "critic." + k[len("critic_target."):]
            p[k].mul_(1 - tau).add_(p[src], alpha=tau)
    # --- the learner's step on the same batch and noise
    losses = learner.gradient_step(batch, noise=noise).tolist()
    ref_losses = [float(actor_loss.detach()), float(critic_loss.detach()), float(ent_loss.detach()), 1.0]
    assert np.allclose(losses, ref_losses, rtol=1e-5, atol=1e-6), (losses, ref_losses)
    got = learner.sb3_state_dict()
    for k, v in p.items():
        if k.startswith("critic.features_extractor."):
            continue  # the shared extractor: the same tensors as actor.features_extractor.*
        ref = v.detach().cpu()
        assert float((got[k] - ref).abs().max()) <= 1e-5 * max(1.0, float(ref.abs().max())), k
    assert abs(float(learner.log_ent_coef.detach()) - float(log_ent)) <= 1e-5 * max(1.0, abs(float(log_ent)))
    assert float(log_ent) != 0.0
    # polyak: critic_target = (1 - tau) old + tau critic, the critic's extractor being the actor's
    for k, old in old_target.items():
        src = ("actor." + k[len("critic_target."):]) if ".features_extractor." in k else ("critic." + k[len("critic_target."):])
        assert torch.allclose(got[k], (old * (1 - tau)).cpu() + tau * got[src], rtol=0, atol=1e-7), k
    # update() syncs the tensor-core actor with the torch actor
    out = learner.update(2)
    assert set(out) == {"actor_loss", "critic_loss", "ent_coef_loss", "ent_coef"} and all(np.isfinite(v) for v in out.values())
    with torch.no_grad():
        mu_t = learner.actor.mu(learner.actor.latent_pi(learner.actor.features(w.sim.obs)))
    w.policy.forward(w.sim.obs)
    assert (w.policy.mu[:N] - mu_t).abs().max().item() < 2e-2
    # SB3 archive round trip: a fresh learner restores identical Q values; the actor part loads into GripperPolicy
    path = learner.save_sb3_zip(str(tmp_path / "sac_model"))
    sd, _ = read_sb3_zip(path)
    assert {k.split(".")[0] for k in sd} == {"actor", "critic", "critic_target"}
    assert any(k.startswith("critic.features_extractor.") for k in sd) and any(k.startswith("critic_target.qf1.") for k in sd)
    fresh = SACLearner(w, rb, batch_size=64, seed=5)
    b = rb.sample(64, 0.0, draw=1)
    assert not torch.equal(fresh.q_values(b["obs"], b["actions"])[0], learner.q_values(b["obs"], b["actions"])[0])
    fresh.load_sb3_zip(path)
    for q_new, q_old in zip(fresh.q_values(b["obs"], b["actions"]), learner.q_values(b["obs"], b["actions"])):
        assert torch.equal(q_new, q_old)
    tgt = [torch.equal(a, c) for a, c in zip(fresh.critic_target(b["next_obs"], b["actions"]), learner.critic_target(b["next_obs"], b["actions"]))]
    assert all(tgt)
    pol = GripperPolicy(max_envs=N, obs_shape=w.sim.obs_shape, action_dim=A)
    pol.load_sb3_zip(path)
    a_file = pol.forward(w.sim.obs).clone()
    learner.sync_policy()
    assert torch.equal(a_file, w.policy.forward(w.sim.obs))
    pol.close()
    w.close()
    rb.close()
