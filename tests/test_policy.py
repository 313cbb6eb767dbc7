"""Policy forward (tcgen05 / TMEM kernels, grp_* C-ABI) against the fp32 torch oracle (oracle/policy_ref.py) and the golden
vectors produced by the reference's own AugmentedNatureCNN class (tests/golden/policy_vectors.npz).

Tolerances (SURVEY.md §8 a-R, bf16 operands with fp32 accumulation vs fp32): |mu - mu_ref| <= 2e-2 (pre-tanh),
|action - action_ref| <= 1e-2, features within 2e-2."""
import os

import numpy as np
import pytest

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "policy_vectors.npz")
TOL_MU, TOL_ACTION, TOL_FEAT = 2e-2, 1e-2, 2e-2


def _params(C, seed):
    from mujoco_rl_manipulate_unknown_objects_b200.policy import init_params
    return init_params(channels=C, action_dim=6, n_flatten=1024, seed=seed)


# ------------------------------------------------------------------------------------------------ CPU: oracle pinned
@pytest.mark.parametrize("tag,C", [("full", 5), ("nodepth", 4)])
def test_oracle_reproduces_the_reference_feature_extractor(tag, C):
    import torch
    from oracle import policy_ref
    g = np.load(GOLD)
    params = _params(C, int(g[tag + "_seed"]))
    with torch.no_grad():
        o = policy_ref.actor(params, g[tag + "_obs"])
        s = policy_ref.actor(params, g[tag + "_obs"], g[tag + "_noise"])
    assert np.abs(o["features"].numpy() - g[tag + "_features"]).max() < 1e-5   # the reference class's own output
    assert np.abs(o["mu"].numpy() - g[tag + "_mu"]).max() < 1e-5
    assert np.abs(o["action"].numpy() - g[tag + "_action"]).max() < 1e-5
    assert np.abs(s["action"].numpy() - g[tag + "_action_stochastic"]).max() < 1e-5
    # the two direct features are the padding-channel scalars / 255 (feature_extractor.py:42)
    assert np.allclose(g[tag + "_features"][:, 512:], g[tag + "_obs"][:, -1, 0, :2] / 255.0, atol=1e-7)


def test_parameter_layout_matches_the_state_dict_names():
    from mujoco_rl_manipulate_unknown_objects_b200.policy import param_spec
    spec = param_spec(5, 6, 1024)
    n = sum(int(np.prod(s)) for _, s in spec)
    # extractor 602 784 parameters (SURVEY.md §3.4) + actor 514*256+256 + 256*256+256 + 2*(6*256+6)
    assert sum(int(np.prod(s)) for k, s in spec if k.startswith("features_extractor.")) == 602784
    assert n == 602784 + 514 * 256 + 256 + 256 * 256 + 256 + 2 * (6 * 256 + 6)


# ------------------------------------------------------------------------------------------------ GPU: kernels vs oracle
@pytest.mark.gpu
@pytest.mark.parametrize("tag,C", [("full", 5), ("nodepth", 4)])
def test_cuda_policy_matches_golden(tag, C):
    import torch
    from mujoco_rl_manipulate_unknown_objects_b200.policy import GripperPolicy
    g = np.load(GOLD)
    pol = GripperPolicy(max_envs=8, obs_shape=(C, 64, 64), action_dim=6, params=_params(C, int(g[tag + "_seed"])))
    obs = torch.as_tensor(g[tag + "_obs"], device="cuda")
    n = obs.shape[0]
    act = pol(obs).cpu().numpy()
    feat = pol.features[:n, :514].float().cpu().numpy()
    mu = pol.mu[:n].cpu().numpy()
    print("[%s] max err: features %.2e mu %.2e action %.2e" % (tag, np.abs(feat - g[tag + "_features"]).max(), np.abs(mu - g[tag + "_mu"]).max(),
                                                               np.abs(act - g[tag + "_action"]).max()))
    assert np.abs(feat - g[tag + "_features"]).max() <= TOL_FEAT
    assert np.all(pol.features[:n, 514:].float().cpu().numpy() == 0)
    assert np.abs(mu - g[tag + "_mu"]).max() <= TOL_MU
    assert np.abs(act - g[tag + "_action"]).max() <= TOL_ACTION
    sto = pol(obs, deterministic=False, noise=torch.as_tensor(g[tag + "_noise"], device="cuda")).cpu().numpy()
    assert np.abs(sto - g[tag + "_action_stochastic"]).max() <= 2 * TOL_ACTION
    assert pol.launch_count == 10  # 5 kernels per forward: conv1, conv2, conv3, linear (+ direct features), fused actor MLP
    pol.close()


@pytest.mark.gpu
@pytest.mark.parametrize("n", [1, 37, 300, 1025])
@pytest.mark.parametrize("C", [5, 4])
def test_cuda_policy_layers_match_oracle_at_ragged_batch_sizes(C, n):
    """Row counts that are not multiples of the 128-row tile (n*225, n*36, n*16, n) and every intermediate activation, for both
    conv chains: C = 5 (4 image planes) runs the descriptor-addressed kernels, C = 4 (3 image planes) the generic k_layer."""
    import torch
    import torch.nn.functional as F
    from mujoco_rl_manipulate_unknown_objects_b200.policy import GripperPolicy
    params = _params(C, 3)
    pol = GripperPolicy(max_envs=n, obs_shape=(C, 64, 64), action_dim=6, params=params)
    gen = torch.Generator().manual_seed(n)
    obs = torch.randint(0, 256, (n, C, 64, 64), dtype=torch.uint8, generator=gen)
    obs[:, C - 1] = 0
    obs[:, C - 1, 0, :2] = torch.randint(0, 4, (n, 2), dtype=torch.uint8, generator=gen)
    act = pol(obs.cuda()).cpu()
    tp = {k: torch.as_tensor(v) for k, v in params.items()}
    with torch.no_grad():
        x = obs.float()[:, :C - 1] / 255.0
        a1 = F.relu(F.conv2d(x, tp["features_extractor.cnn.0.weight"], tp["features_extractor.cnn.0.bias"], stride=4))
        a2 = F.relu(F.conv2d(a1, tp["features_extractor.cnn.2.weight"], tp["features_extractor.cnn.2.bias"], stride=2))
        a3 = F.relu(F.conv2d(a2, tp["features_extractor.cnn.4.weight"], tp["features_extractor.cnn.4.bias"], stride=1))
        from oracle import policy_ref
        ref = policy_ref.actor(params, obs)
    g1 = pol.buffer("act1", (n, 15, 15, 32), torch.bfloat16).float().cpu().permute(0, 3, 1, 2)
    g2 = pol.buffer("act2", (n, 6, 6, 64), torch.bfloat16).float().cpu().permute(0, 3, 1, 2)
    g3 = pol.buffer("act3", (n, 4, 4, 64), torch.bfloat16).float().cpu().permute(0, 3, 1, 2)
    e1, e2, e3 = (g1 - a1).abs().max().item(), (g2 - a2).abs().max().item(), (g3 - a3).abs().max().item()
    ef = (pol.features[:n, :514].float().cpu() - ref["features"]).abs().max().item()
    em = (pol.mu[:n].cpu() - ref["mu"]).abs().max().item()
    ea = (act - ref["action"]).abs().max().item()
    print("[C=%d n=%d] conv1 %.2e conv2 %.2e conv3 %.2e features %.2e mu %.2e action %.2e" % (C, n, e1, e2, e3, ef, em, ea))
    assert e1 <= 1e-2 and e2 <= 2e-2 and e3 <= 2e-2 and ef <= TOL_FEAT
    assert em <= TOL_MU and ea <= TOL_ACTION
    pol.close()


@pytest.mark.gpu
def test_cuda_policy_full_batch_properties():
    """BASELINE size (4 096 envs): row independence — a batch element's action does not depend on its neighbours or on its
    position in the batch — and determinism."""
    import torch
    from mujoco_rl_manipulate_unknown_objects_b200.policy import GripperPolicy
    N = 4096
    pol = GripperPolicy(max_envs=N, obs_shape=(5, 64, 64), action_dim=6, seed=11)
    gen = torch.Generator(device="cuda").manual_seed(5)
    obs = torch.randint(0, 256, (N, 5, 64, 64), dtype=torch.uint8, device="cuda", generator=gen)
    a = pol(obs).clone()
    b = pol(obs).clone()
    assert torch.equal(a, b)
    perm = torch.randperm(N, device="cuda", generator=gen)
    c = pol(obs[perm].contiguous())
    assert torch.equal(c, a[perm])
    small = pol(obs[1000:1100].contiguous())
    assert torch.equal(small, a[1000:1100])
    assert torch.isfinite(a).all() and a.abs().max() <= 1.0 and a.std() > 1e-3
    pol.close()


@pytest.mark.gpu
def test_cuda_policy_rejects_bad_input():
    import torch
    from mujoco_rl_manipulate_unknown_objects_b200.policy import GripperPolicy
    pol = GripperPolicy(max_envs=4, obs_shape=(5, 64, 64), action_dim=6)
    with pytest.raises(ValueError):
        pol(torch.zeros((2, 5, 32, 32), dtype=torch.uint8, device="cuda"))
    with pytest.raises(RuntimeError):
        pol(torch.zeros((8, 5, 64, 64), dtype=torch.uint8, device="cuda"))  # more than max_envs
    sd = pol.state_dict()
    sd["mu.weight"] = sd["mu.weight"][:3]
    with pytest.raises(ValueError):
        pol.load_state_dict(sd)
    pol.close()
