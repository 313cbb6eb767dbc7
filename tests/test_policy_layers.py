"""Policy forward, layer by layer, against the rounding-faithful fp64 restatement of the kernels (oracle/policy_ref.py).

tests/test_policy.py anchors the network to fp32 torch and to the reference's own feature extractor; its tolerances are about
the size of the signal at torch-default parameters, so a dropped k-block or a one-ulp slip passes it.  The checks here are
sharp:
  * arithmetic: every layer's output against y* computed in fp64 from the GPU's OWN input to that layer and the kernel's rounded
    weights, within  1/2 ulp_bf16(max(|y*|, |y|)) + s K 2^-23 sum|x||w| + 2^-24 |y*|  (fp32 outputs: K 2^-23 s sum|x||w| +
    2^-23 |y*|).  The bound is derived, not tuned: a CPU self-check shows a simulated kernel inside it and each plausible kernel
    bug (one K = 16 slice, one input channel, the direct features, a one-ulp shift) outside it;
  * routing: one-hot weights of value 1 and per-channel biases make every output RN_bf16(RN_fp32(x_tap * s + b)), compared bit for
    bit, over every K index of every layer, every observation shape the kernels distinguish and batch sizes around the SM count;
  * stale rows and the programmatic-dependent-launch chain of back-to-back forwards, bit for bit.
The hidden activations of the fused MLP never leave shared memory; they are made visible through the public API by setting
latent_pi.2 to the identity and the head to unit vectors (action_dim 8: mu rows), which copy them exactly.
"""
import numpy as np
import pytest
import torch

from oracle import policy_ref as R

# (C, H, W) -> conv maps o1, o2, o3 and nflat (the generic chain runs every shape but (5, 64, 64))
SHAPES = [(5, 64, 64), (4, 64, 64), (5, 48, 48), (5, 64, 40), (5, 36, 36)]
DEV = "cuda"
C1W, C2W, C3W, FCW = ("features_extractor.cnn.0.weight", "features_extractor.cnn.2.weight", "features_extractor.cnn.4.weight",
                      "features_extractor.linear.0.weight")


def maps(shape):
    _, h, w = shape
    o1 = ((h - 8) // 4 + 1, (w - 8) // 4 + 1)
    o2 = ((o1[0] - 4) // 2 + 1, (o1[1] - 4) // 2 + 1)
    o3 = (o2[0] - 2, o2[1] - 2)
    return o1, o2, o3, 64 * o3[0] * o3[1]


# ------------------------------------------------------------------------------------------------ parameters and inputs
def default_params(shape, adim=6, seed=0):
    from mujoco_rl_manipulate_unknown_objects_b200.policy import init_params
    return init_params(shape[0], adim, maps(shape)[3], seed)


def trained_params(shape, adim=6, seed=0):
    """Weights scaled so that activations reach O(1)..O(10), and biases of both signs of the activations' size, so ReLU zeroes
    a real fraction of every layer (what a trained policy looks like, rather than torch's shrinking default init)."""
    rng = np.random.default_rng(1000 + seed)
    p = default_params(shape, adim, seed)
    gain = {"features_extractor.cnn.0": (12.0, 1.0), "features_extractor.cnn.2": (4.0, 2.0), "features_extractor.cnn.4": (3.0, 2.0),
            "features_extractor.linear.0": (3.0, 2.0), "latent_pi.0": (3.0, 2.0), "latent_pi.2": (3.0, 2.0), "mu": (1.0, 0.5),
            "log_std": (1.0, 0.5)}
    for layer, (g, b) in gain.items():
        p[layer + ".weight"] = (p[layer + ".weight"] * g).astype(np.float32)
        p[layer + ".bias"] = rng.uniform(-b, b, p[layer + ".bias"].shape).astype(np.float32)
    return p


def subnormal_params(shape, adim=6, seed=0):
    """conv1 weights log-uniform over |w| in [2^-27, 2^2]: fp16 subnormals (< 2^-14), values that round to zero (< 2^-25) and
    normal ones, of both signs."""
    rng = np.random.default_rng(2000 + seed)
    p = default_params(shape, adim, seed)
    w = p[C1W]
    p[C1W] = (np.exp2(rng.uniform(-27, 2, w.shape)) * rng.choice([-1.0, 1.0], w.shape)).astype(np.float32)
    p["features_extractor.cnn.0.bias"] = rng.uniform(-0.05, 0.1, 32).astype(np.float32)
    return p


PARAMS = {"default": default_params, "trained": trained_params, "subnormal": subnormal_params}


def images(shape, n, seed):
    """Random images, with an all-0 and an all-255 image among them; the direct features obs[:, C-1, 0, :2] span 0..255."""
    g = torch.Generator().manual_seed(seed)
    c, h, w = shape
    obs = torch.randint(0, 256, (n, c, h, w), dtype=torch.uint8, generator=g)
    if n >= 3:
        obs[1], obs[2] = 0, 255
    obs[:, c - 1] = 0
    obs[:, c - 1, 0, :2] = torch.randint(0, 256, (n, 2), dtype=torch.uint8, generator=g)
    obs[0, c - 1, 0, :2] = torch.tensor([0, 255], dtype=torch.uint8)
    return obs


# ------------------------------------------------------------------------------------------------ layer-local checks
def conv_ratios(kw, obs, out, K1):
    """Max error / bound of conv1, conv2, conv3 and the linear layer, each from its own input in `out` (NCHW, [n, 576]); the direct
    features and the zero padding of the feature row are exact."""
    r = {}
    for name, fn, x, y, K in (("conv1", R.conv1, obs, out["act1"], K1), ("conv2", R.conv2, out["act1"], out["act2"], 512),
                              ("conv3", R.conv3, out["act2"], out["act3"], 576), ("linear", R.linear, out["act3"], out["feat"][:, :512], None)):
        ys, acc = fn(kw, x)
        r[name] = R.ratio_bf16(y, ys, acc, K if K is not None else x[0].numel()).max().item()
    assert torch.equal(out["feat"][:, 512:514].to(torch.float64), R.direct_features(obs)), "direct features"
    assert not out["feat"][:, 514:].any(), "feature padding"
    return r


def mlp_ratios(kw, feat, h1, h2, mu, ls):
    r = {}
    ys, acc = R.dense(kw, "latent_pi.0", feat[:, :514])
    r["latent_pi.0"] = R.ratio_bf16(h1, ys, acc, R.FEAT_LD).max().item()
    ys, acc = R.dense(kw, "latent_pi.2", h1)
    r["latent_pi.2"] = R.ratio_bf16(h2, ys, acc, 256).max().item()
    r.update(head_ratios(kw, h2, mu, ls))
    return r


def head_ratios(kw, h2, mu, ls):
    r = {}
    ys, acc = R.dense(kw, "mu", h2, relu=False)
    r["mu"] = R.ratio_fp32(mu, ys, acc, 256).max().item()
    ys, acc = R.log_std(kw, h2)
    r["log_std"] = R.ratio_fp32(ls, ys, acc, 256).max().item()
    return r


# ------------------------------------------------------------------------------------------------ CPU: the bounds themselves
def _bump_ulp(y):
    """+1 bf16 ulp (y >= 0: the ReLU outputs) / +1 bf16 ulp of |y| away from zero for signed fp32 outputs."""
    b = y.to(torch.float32).to(torch.bfloat16)
    up = (b.view(torch.int16) + 1).view(torch.bfloat16).to(torch.float64)
    if (y >= 0).all():
        return up
    return y.to(torch.float64) + torch.sign(y.to(torch.float64)) * R.ulp(y, 7)


def simulate(params, obs, mutate=None):
    """The kernels restated on the CPU: the same rounded operands, fp32 accumulation (in torch's order, not the tensor core's),
    the fp32 epilogues and the bf16 stores.  `mutate` applies one plausible kernel bug."""
    import torch.nn.functional as F
    kw = {k: v.to(torch.float32) for k, v in R.kernel_weights(params).items()}
    w1, w2, w3, wfc = kw[C1W], kw[C2W].clone(), kw[C3W].clone(), kw[FCW].clone()
    w0, wmu, wls = kw["latent_pi.0.weight"].clone(), kw["mu.weight"].clone(), kw["log_std.weight"].clone()
    if mutate == "conv3_k16":       # the kernel's K order is (ky, kx, c): slice 17 = tap (1, 1), channels 16..31
        w3[:, 16:32, 1, 1] = 0
    elif mutate == "conv2_channel":  # one input channel never read
        w2[:, 5] = 0
    elif mutate == "linear_k16":    # the last K = 16 slice of the (y, x, c) order: channels 48..63 of the last position
        hw = wfc.shape[1] // 64
        wfc.view(512, 64, hw)[:, 48:, hw - 1] = 0
    elif mutate == "head_k16":
        wmu[:, 240:], wls[:, 240:] = 0, 0
    elif mutate == "latent0_direct":
        w0[:, 512:514] = 0

    def store(acc_plus_b):  # ReLU, bf16
        return R.bf16(acc_plus_b.clamp_min(0.0))

    x = obs[:, :-1].to(torch.float32)
    acc = F.conv2d(x, w1, stride=4)
    a1 = store((acc.to(torch.float64) * R.S_CONV1 + kw["features_extractor.cnn.0.bias"].view(1, -1, 1, 1).double()).to(torch.float32))  # fmaf
    a2 = store(F.conv2d(a1.float(), w2, stride=2) + kw["features_extractor.cnn.2.bias"].view(1, -1, 1, 1))
    a3 = store(F.conv2d(a2.float(), w3, stride=1) + kw["features_extractor.cnn.4.bias"].view(1, -1, 1, 1))
    f = store(a3.float().flatten(1) @ wfc.T + kw["features_extractor.linear.0.bias"])
    feat = torch.cat((f, R.direct_features(obs), torch.zeros(obs.shape[0], R.FEAT_LD - 514, dtype=torch.float64)), 1)
    h1 = store(feat[:, :514].float() @ w0.T + kw["latent_pi.0.bias"])
    h2 = store(h1.float() @ kw["latent_pi.2.weight"].T + kw["latent_pi.2.bias"])
    mu = (h2.float() @ wmu.T + kw["mu.bias"]).double()
    ls = (h2.float() @ wls.T + kw["log_std.bias"]).clamp(R.LOG_STD_MIN, R.LOG_STD_MAX).double()
    out = dict(act1=a1, act2=a2, act3=a3, feat=feat, h1=h1, h2=h2, mu=mu, ls=ls)
    if mutate == "ulp":
        out = {k: (_bump_ulp(v) if k != "feat" else torch.cat((_bump_ulp(v[:, :512]), v[:, 512:]), 1)) for k, v in out.items()}
    return out


def all_ratios(params, obs, out):
    kw = R.kernel_weights(params)
    r = conv_ratios(kw, obs, out, (obs.shape[1] - 1) * 64)
    r.update(mlp_ratios(kw, out["feat"], out["h1"], out["h2"], out["mu"], out["ls"]))
    return r


@pytest.mark.parametrize("kind", ["default", "trained", "subnormal"])
def test_simulated_kernel_is_within_the_bounds(kind):
    shape = (5, 64, 64)
    params = PARAMS[kind](shape, seed=3)
    obs = images(shape, 37, 3)
    out = simulate(params, obs)
    r = all_ratios(params, obs, out)
    print("[%s] max error / bound: %s" % (kind, " ".join("%s %.3f" % kv for kv in r.items())))
    assert max(r.values()) <= 1.0, r
    if kind == "trained":  # the trained-scale set does what it is for: O(1)..O(10) activations, ReLU zeroing a real fraction
        for k in ("act1", "act2", "act3", "h1", "h2"):
            assert 1.0 < out[k].max() < 100.0 and 0.1 < (out[k] == 0).double().mean() < 0.9, k


# mutation -> the layer whose bound it must break
MUTATIONS = {"conv3_k16": ["conv3"], "conv2_channel": ["conv2"], "linear_k16": ["linear"], "head_k16": ["mu", "log_std"],
             "latent0_direct": ["latent_pi.0"], "ulp": ["conv1", "conv2", "conv3", "linear", "latent_pi.0", "latent_pi.2", "mu"]}


@pytest.mark.parametrize("mutation", sorted(MUTATIONS))
def test_each_plausible_kernel_bug_breaks_its_layer_bound(mutation):
    shape = (5, 64, 64)
    params = default_params(shape, seed=3)
    obs = images(shape, 37, 3)
    r = all_ratios(params, obs, simulate(params, obs, mutation))
    print("[%s] max error / bound: %s" % (mutation, " ".join("%s %.1f" % kv for kv in r.items())))
    for layer in MUTATIONS[mutation]:
        assert r[layer] > 1.5, (layer, r)
    if mutation != "ulp":  # layer-local: only the mutated layer fails, the others start from its (wrong) output and pass
        assert all(v <= 1.0 for k, v in r.items() if k not in MUTATIONS[mutation]), r


def test_action_bound_accepts_the_documented_errors_and_rejects_an_ulp_shift():
    """tanhf (2 ulp) and __expf (2 + floor(|1.173 x|) ulp) as documented: torch's fp32 tanh / exp pass, and three fp32 ulps
    added to the deterministic action fail."""
    g = torch.Generator().manual_seed(0)
    mu = (torch.randn(4096, generator=g) * 3).to(torch.float32)
    ls = (torch.rand(4096, generator=g) * 22 - 20).to(torch.float32)
    noise = torch.tensor([0.0, 1.0, -1.0, 5.0, -5.0]).repeat(820)[:4096]
    a = torch.tanh(mu)
    assert R.ratio_action(a, mu).max() <= 1.0
    sto = torch.tanh(mu + torch.exp(ls) * noise)
    assert R.ratio_action(sto, mu, ls, noise).max() <= 1.0
    bad = torch.nextafter(torch.nextafter(torch.nextafter(a, a + 1), a + 1), a + 1)
    inside = a.abs() < 0.9
    assert R.ratio_action(bad[inside], mu[inside]).max() > 1.0


# ------------------------------------------------------------------------------------------------ GPU helpers
def _policy(shape, n, adim=6, params=None):
    from mujoco_rl_manipulate_unknown_objects_b200.policy import GripperPolicy
    return GripperPolicy(max_envs=n, obs_shape=shape, action_dim=adim, params=params)


def gpu_outputs(pol, n):
    """The last forward's intermediates, NCHW / [n, 576] fp64 on the device."""
    o1, o2, o3, _ = maps(pol.obs_shape)
    b = lambda name, hw, c: pol.buffer(name, (pol.max_envs, hw[0], hw[1], c), torch.bfloat16)[:n].permute(0, 3, 1, 2).to(torch.float64)
    return dict(act1=b("act1", o1, 32), act2=b("act2", o2, 64), act3=b("act3", o3, 64), feat=pol.features[:n].to(torch.float64))


def selector_head(p, cols):
    """mu row k = h2[:, cols[k]] exactly (action_dim 8, zero biases); log_std rows unused (zero)."""
    p = dict(p)
    p["mu.weight"] = np.zeros((8, 256), np.float32)
    p["mu.weight"][np.arange(8), cols] = 1.0
    p["mu.bias"] = np.zeros(8, np.float32)
    p["log_std.weight"], p["log_std.bias"] = np.zeros((8, 256), np.float32), np.zeros(8, np.float32)
    return p


def hidden(pol8, params, obs_dev, layer):
    """h1 (layer 1: latent_pi.2 set to the identity) or h2 (layer 2) [n, 256] of `params`, read eight columns per forward through
    the mu rows of an action_dim-8 policy: every step of the copy (identity MMA, + 0, ReLU of a bf16 value >= 0, bf16 store,
    unit-vector head) is exact."""
    p = dict(params)
    if layer == 1:
        p["latent_pi.2.weight"], p["latent_pi.2.bias"] = np.eye(256, dtype=np.float32), np.zeros(256, np.float32)
    cols = []
    for u in range(32):
        pol8.load_state_dict(selector_head(p, np.arange(8 * u, 8 * u + 8)))
        pol8(obs_dev)
        cols.append(pol8.mu[:obs_dev.shape[0]].to(torch.float64))
    return torch.cat(cols, 1)


# ------------------------------------------------------------------------------------------------ GPU: arithmetic
@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["default", "trained", "subnormal"])
@pytest.mark.parametrize("shape", [(5, 64, 64), (4, 64, 64)], ids=["direct", "generic"])
def test_every_layer_is_within_its_rounding_bound(shape, kind):
    n = 150
    params = PARAMS[kind](shape, adim=8, seed=5)
    obs = images(shape, n, 11)
    obs_dev = obs.to(DEV)
    pol = _policy(shape, n, 8, params)
    noise = torch.tensor([0.0, 1.0, -1.0, 5.0, -5.0, 0.5, -2.0, 3.0], device=DEV).repeat(n, 1)
    act_det = pol(obs_dev).clone()
    act_sto = pol(obs_dev, deterministic=False, noise=noise).clone()
    out = gpu_outputs(pol, n)
    mu, ls = pol.mu[:n].clone(), pol.log_std[:n].clone()
    kw = R.kernel_weights(params, DEV)
    r = conv_ratios(kw, obs_dev, out, (shape[0] - 1) * 64)
    h1 = hidden(pol, params, obs_dev, 1)
    h2 = hidden(pol, params, obs_dev, 2)
    r.update(mlp_ratios(kw, out["feat"], h1, h2, mu, ls))
    r["action"] = R.ratio_action(act_det, mu).max().item()
    r["action_noise"] = R.ratio_action(act_sto, mu, ls, noise).max().item()
    print("[%s %s] max error / bound: %s" % (shape, kind, " ".join("%s %.3f" % kv for kv in r.items())))
    assert max(r.values()) <= 1.0, r
    pol.close()


@pytest.mark.gpu
def test_head_clamps_saturates_and_runs_every_action_dim():
    shape, n = (5, 64, 64), 64
    base = trained_params(shape, adim=8, seed=7)
    obs_dev = images(shape, n, 7).to(DEV)
    pol8 = _policy(shape, n, 8, base)
    h2 = hidden(pol8, base, obs_dev, 2)
    pol8.close()
    noise_vals = torch.tensor([0.0, 1.0, -1.0, 5.0, -5.0, 0.0, 1.0, -5.0], device=DEV)
    for adim in (1, 5, 6, 8):
        p = trained_params(shape, adim=adim, seed=7)
        pol = _policy(shape, n, adim, p)
        noise = noise_vals[:adim].repeat(n, 1)
        act = pol(obs_dev, deterministic=False, noise=noise).clone()
        kw = R.kernel_weights(p, DEV)
        r = head_ratios(kw, h2, pol.mu[:n], pol.log_std[:n])
        ra = R.ratio_action(act, pol.mu[:n], pol.log_std[:n], noise).max().item()
        print("[action_dim %d] mu %.3f log_std %.3f action %.3f" % (adim, r["mu"], r["log_std"], ra))
        assert r["mu"] <= 1.0 and r["log_std"] <= 1.0 and ra <= 1.0
        # biases past both clamps: log_std exactly 2 and -20; |mu| >= 20: actions exactly +-1, with any noise, and no NaN
        sgn = np.where(np.arange(adim) % 2 == 0, 1.0, -1.0).astype(np.float32)
        p["log_std.bias"] = (1000.0 * sgn).astype(np.float32)
        p["mu.bias"] = (100.0 * sgn).astype(np.float32)
        pol.load_state_dict(p)
        for det in (True, False):
            a = pol(obs_dev, deterministic=det, noise=None if det else noise)
            ls = pol.log_std[:n]
            assert (pol.mu[:n] * torch.as_tensor(sgn, device=DEV) >= 20).all()
            assert torch.equal(ls, torch.where(torch.as_tensor(sgn, device=DEV) > 0, 2.0, -20.0).expand(n, adim))
            assert torch.equal(a, torch.as_tensor(sgn, device=DEV).expand(n, adim)), a
        pol.close()


# ------------------------------------------------------------------------------------------------ GPU: routing probes (bit-exact)
def _tap_gather(x, c, ky, kx, stride, oh, ow):
    """out[n, o, y, x] = x[n, c[o], stride y + ky[o], stride x + kx[o]]."""
    dev = x.device
    rows = stride * torch.arange(oh, device=dev)[None, :, None] + ky[:, None, None]
    cols = stride * torch.arange(ow, device=dev)[None, None, :] + kx[:, None, None]
    return x[:, c[:, None, None], rows, cols]


def _rn(x):  # fp64 value (exact sum) -> fp32 -> bf16, as fmaf / fadd and the bf16 store round it
    return x.to(torch.float32).to(torch.bfloat16).to(torch.float64)


def probe_params(shape, adim, t, r=0, u=0, perm=False, conv1_values=None):
    """One-hot parameters of probe forward t: output o of each layer reads one input (a tap of value 1.0) and adds a small bias
    (o + 1) 2^-k distinct per output.  conv1 output o reads tap (32 t + o) mod cin*64, conv2 / conv3 tap (64 t + o) mod 512 / 576,
    the linear layer input (512 t + o) mod nflat (torch's orders).  latent_pi.0 row j reads feature column (256 r + j) mod 514;
    latent_pi.2 is the identity (perm=False) or the permutation j -> (37 j + 11) mod 256 with biases; the head's mu / log_std rows
    k read h2 columns 16 u + k / 16 u + 8 + k.  With weights of 1 every value stays below 2, where log_std is not clamped."""
    cin = shape[0] - 1
    nflat = maps(shape)[3]
    p = {}

    def onehot(o_count, k_count, off, kshape):
        w = np.zeros((o_count, k_count), np.float32)
        w[np.arange(o_count), (off + np.arange(o_count)) % k_count] = 1.0
        return w.reshape((o_count,) + kshape)

    p[C1W] = onehot(32, cin * 64, 32 * t, (cin, 8, 8))
    p["features_extractor.cnn.0.bias"] = ((np.arange(32) + 1) * 2.0 ** -10).astype(np.float32)
    if conv1_values is not None:
        p[C1W] = p[C1W] * np.asarray(conv1_values, np.float32).reshape(32, 1, 1, 1)
        p["features_extractor.cnn.0.bias"][:] = 0
    p[C2W] = onehot(64, 512, 64 * t, (32, 4, 4))
    p["features_extractor.cnn.2.bias"] = ((np.arange(64) + 1) * 2.0 ** -10).astype(np.float32)
    p[C3W] = onehot(64, 576, 64 * t, (64, 3, 3))
    p["features_extractor.cnn.4.bias"] = ((np.arange(64) + 1) * 2.0 ** -10).astype(np.float32)
    p[FCW] = onehot(512, nflat, 512 * t, (nflat,))
    p["features_extractor.linear.0.bias"] = ((np.arange(512) + 1) * 2.0 ** -12).astype(np.float32)
    p["latent_pi.0.weight"] = onehot(256, 514, 256 * r, (514,))
    p["latent_pi.0.bias"] = ((np.arange(256) + 1) * 2.0 ** -12).astype(np.float32)
    if perm:
        p["latent_pi.2.weight"] = np.eye(256, dtype=np.float32)[(37 * np.arange(256) + 11) % 256]
        p["latent_pi.2.bias"] = ((np.arange(256) + 1) * 2.0 ** -12).astype(np.float32)
    else:
        p["latent_pi.2.weight"], p["latent_pi.2.bias"] = np.eye(256, dtype=np.float32), np.zeros(256, np.float32)
    for name, off in (("mu", 0), ("log_std", 8)):
        w = np.zeros((adim, 256), np.float32)
        w[np.arange(adim), 16 * u + off + np.arange(adim)] = 1.0
        p[name + ".weight"], p[name + ".bias"] = w, np.zeros(adim, np.float32)
    return p


def check_probe(pol, params, obs_dev, n):
    """Every observable output of a probe forward, bit for bit, each from the kernel's own input to that layer."""
    shape, adim = pol.obs_shape, pol.action_dim
    (o1, o2, o3, nflat), cin = maps(shape), shape[0] - 1
    out = gpu_outputs(pol, n)
    dev = obs_dev.device

    def taps(w, kshape):  # the (c, ky, kx) each output reads, from the one-hot weights
        k = torch.as_tensor(np.abs(w).reshape(w.shape[0], -1).argmax(1), device=dev)
        return k // (kshape[1] * kshape[2]), k // kshape[2] % kshape[1], k % kshape[2]

    def bias(name):
        return torch.as_tensor(params[name], device=dev, dtype=torch.float64).view(1, -1, 1, 1)

    v1 = torch.as_tensor(np.abs(params[C1W]).reshape(32, -1).max(1), device=dev).to(torch.float16).to(torch.float64).view(1, -1, 1, 1)
    x = _tap_gather(obs_dev[:n, :cin].to(torch.float64), *taps(params[C1W], (cin, 8, 8)), 4, *o1)
    exp1 = _rn(x * v1 * R.S_CONV1 + bias("features_extractor.cnn.0.bias"))
    assert torch.equal(out["act1"], exp1), "act1: %d of %d differ" % ((out["act1"] != exp1).sum(), exp1.numel())
    exp2 = _rn(_tap_gather(out["act1"], *taps(params[C2W], (32, 4, 4)), 2, *o2) + bias("features_extractor.cnn.2.bias"))
    assert torch.equal(out["act2"], exp2), "act2: %d of %d differ" % ((out["act2"] != exp2).sum(), exp2.numel())
    exp3 = _rn(_tap_gather(out["act2"], *taps(params[C3W], (64, 3, 3)), 1, *o3) + bias("features_extractor.cnn.4.bias"))
    assert torch.equal(out["act3"], exp3), "act3: %d of %d differ" % ((out["act3"] != exp3).sum(), exp3.numel())
    kfc = torch.as_tensor(params[FCW].argmax(1), device=dev)
    fb = torch.as_tensor(params["features_extractor.linear.0.bias"], device=dev, dtype=torch.float64)
    expf = _rn(out["act3"].flatten(1)[:, kfc] + fb)
    assert torch.equal(out["feat"][:, :512], expf), "features: %d of %d differ" % ((out["feat"][:, :512] != expf).sum(), expf.numel())
    assert torch.equal(out["feat"][:, 512:514], R.direct_features(obs_dev[:n]))
    assert not out["feat"][:, 514:].any()
    k0 = torch.as_tensor(params["latent_pi.0.weight"].argmax(1), device=dev)
    h1 = _rn(out["feat"][:, k0] + torch.as_tensor(params["latent_pi.0.bias"], device=dev, dtype=torch.float64))
    k1 = torch.as_tensor(params["latent_pi.2.weight"].argmax(1), device=dev)
    h2 = _rn(h1[:, k1] + torch.as_tensor(params["latent_pi.2.bias"], device=dev, dtype=torch.float64))
    for name, buf in (("mu", pol.mu), ("log_std", pol.log_std)):
        exp = h2[:, torch.as_tensor(params[name + ".weight"].argmax(1), device=dev)].to(torch.float32)
        if name == "log_std":
            exp = exp.clamp_max(R.LOG_STD_MAX)
        assert torch.equal(buf[:n], exp), "%s: %d of %d differ" % (name, (buf[:n] != exp).sum(), exp.numel())


SM = None


def _sm_count():
    global SM
    if SM is None:
        SM = torch.cuda.get_device_properties(0).multi_processor_count
    return SM


@pytest.mark.gpu
@pytest.mark.parametrize("shape", SHAPES, ids=lambda s: "x".join(map(str, s)))
def test_probes_route_every_k_index_of_every_layer(shape):
    """Probe forwards 0..8 cover every K index of conv1 (cin 64), conv2 (512), conv3 (576) and the linear layer (nflat); probes
    (r, u) cover all 514 feature columns into h1 and every h1 / h2 column (identity latent_pi.2), then every h2 column through a
    permuted latent_pi.2 with biases."""
    n = 131
    obs_dev = images(shape, n, 1).to(DEV)
    pol = _policy(shape, n, 8, probe_params(shape, 8, 0))
    for t in range(9):
        p = probe_params(shape, 8, t, r=t % 3, u=t)
        pol.load_state_dict(p)
        pol(obs_dev)
        check_probe(pol, p, obs_dev, n)
    for r in range(3):
        for u in range(16):
            p = probe_params(shape, 8, 0, r=r, u=u)
            pol.load_state_dict(p)
            pol(obs_dev)
            check_probe(pol, p, obs_dev, n)
    for u in range(16):
        p = probe_params(shape, 8, 0, u=u, perm=True)
        pol.load_state_dict(p)
        pol(obs_dev)
        check_probe(pol, p, obs_dev, n)
    pol.close()


# fp32 weights across the fp16 range: subnormals (min 2^-24), the subnormal / normal boundary, ties of both parities in both
# ranges (2^-25 -> 0, 3 * 2^-25 -> 2^-23, 1 + 2^-11 -> 1, 1 + 3 * 2^-11 -> 1 + 2^-9), values below the smallest subnormal that
# round to it, the largest fp16 (65504) and 65519 (-> 65504), and ordinary values
FP16_PROBE = [2.0 ** -24, 3 * 2.0 ** -24, 2.0 ** -25, 3 * 2.0 ** -25, 0.7 * 2.0 ** -24, 2.0 ** -24 * 1.5000001, 1023 * 2.0 ** -24,
              2.0 ** -14 - 2.0 ** -25, 2.0 ** -14, 2.0 ** -14 + 2.0 ** -25, 1.0, 1 + 2.0 ** -11, 1 + 3 * 2.0 ** -11, 1 + 2.0 ** -12,
              0.1, 0.3333333, 3.14159, 255.0, 1000.1, 2049.0, 4097.0, 65504.0, 65519.0, 65519.99, 3e-8, 5.9604645e-08, 1e-5,
              6.1e-5, 0.5 + 2.0 ** -12, 2.0 ** -15 * 1.75, 32768.0 + 16.0, 12345.678]


@pytest.mark.gpu
@pytest.mark.parametrize("shape", [(5, 64, 64), (4, 64, 64)], ids=["direct", "generic"])
def test_conv1_weights_are_rounded_to_fp16_across_its_range(shape):
    n = 64
    assert len(FP16_PROBE) == 32
    obs_dev = images(shape, n, 2).to(DEV)
    pol = _policy(shape, n, 8, probe_params(shape, 8, 0))
    cin = shape[0] - 1
    for t in range(cin * 2):
        p = probe_params(shape, 8, t, conv1_values=np.roll(FP16_PROBE, t))
        pol.load_state_dict(p)
        pol(obs_dev)
        check_probe(pol, p, obs_dev, n)
    pol.close()


@pytest.mark.gpu
def test_conv1_weights_outside_fp16_are_refused():
    """A weight that would round to +-inf in fp16 (|w| >= 65520, or not finite) is refused with its name and index; the policy
    keeps its previous parameters.  65519.99 rounds to 65504 and is accepted."""
    shape, n = (5, 64, 64), 8
    pol = _policy(shape, n)
    before = pol.state_dict()
    for bad in (65520.0, -70000.0, float("inf"), float("nan")):
        sd = dict(before)
        sd[C1W] = sd[C1W].copy()
        sd[C1W][3, 1, 2, 5] = bad
        with pytest.raises(RuntimeError, match=r"features_extractor\.cnn\.0\.weight\[3, 1, 2, 5\]"):
            pol.load_state_dict(sd)
        after = pol.state_dict()
        assert all(np.array_equal(after[k], before[k]) for k in before)
    sd = dict(before)
    sd[C1W] = sd[C1W].copy()
    sd[C1W][3, 1, 2, 5] = 65519.99
    pol.load_state_dict(sd)
    assert torch.isfinite(pol(images(shape, n, 0).to(DEV))).all()
    pol.close()


# ------------------------------------------------------------------------------------------------ GPU: shapes and batch edges
def _batch_sizes():
    s = _sm_count()
    return [1, 2, 3, 5, 127, 128, 129, s - 1, s, s + 1, 2 * s - 1, 2 * s, 2 * s + 1, 3 * s + 4]


@pytest.mark.gpu
@pytest.mark.parametrize("shape", SHAPES, ids=lambda s: "x".join(map(str, s)))
def test_batch_sizes_around_the_sm_count(shape):
    """Persistent CTAs over images (conv1: min(n, #SM)) and image pairs (conv2 / conv3: min((n + 1) / 2, #SM)), 128-row tiles:
    a probe forward (bit-exact) and a default-init forward (bounds) at every batch size."""
    sizes = _batch_sizes()
    worst = {}
    for n in sizes:
        obs = images(shape, n, n)
        obs_dev = obs.to(DEV)
        p = probe_params(shape, 6, n % 9, r=n % 3, u=n % 16, perm=n % 2 == 1)
        pol = _policy(shape, n, 6, p)
        pol(obs_dev)
        check_probe(pol, p, obs_dev, n)
        params = default_params(shape, seed=n)
        pol.load_state_dict(params)
        act = pol(obs_dev)
        r = conv_ratios(R.kernel_weights(params, DEV), obs_dev, gpu_outputs(pol, n), (shape[0] - 1) * 64)
        r["action"] = R.ratio_action(act, pol.mu[:n]).max().item()
        for k, v in r.items():
            worst[k] = max(worst.get(k, 0.0), v)
        assert max(r.values()) <= 1.0, (n, r)
        pol.close()
    print("[%s] n %s: max error / bound %s" % (shape, sizes, " ".join("%s %.3f" % kv for kv in worst.items())))


@pytest.mark.gpu
def test_probe_at_16384_environments():
    shape, n = (5, 64, 64), 16384
    g = torch.Generator(device=DEV).manual_seed(16384)
    obs_dev = torch.randint(0, 256, (n,) + shape, dtype=torch.uint8, device=DEV, generator=g)
    p = probe_params(shape, 6, 4, r=1, u=3, perm=True)
    pol = _policy(shape, n, 6, p)
    pol(obs_dev)
    check_probe(pol, p, obs_dev, n)
    pol.close()


@pytest.mark.gpu
@pytest.mark.parametrize("shape", [(5, 64, 64), (5, 48, 48)], ids=["direct", "generic"])
def test_smaller_odd_batch_after_a_full_one_leaves_no_stale_rows(shape):
    """A full max_envs forward, then a smaller odd n on other images: every row below n is what a fresh policy computes, bit for
    bit (the last image pair of conv2 / conv3 is half stale), and the feature padding is zero."""
    N, n = 2 * _sm_count() + 1, _sm_count() + 1 + _sm_count() % 2
    params = trained_params(shape, seed=2)
    pol = _policy(shape, N, 6, params)
    pol(images(shape, N, 100).to(DEV))
    obs_dev = images(shape, n, 200).to(DEV)
    noise = torch.randn(n, 6, device=DEV)
    a = pol(obs_dev, deterministic=False, noise=noise).clone()
    fresh = _policy(shape, n, 6, params)
    b = fresh(obs_dev, deterministic=False, noise=noise)
    assert torch.equal(a, b)
    for k, v in gpu_outputs(pol, n).items():
        assert torch.equal(v, gpu_outputs(fresh, n)[k]), k
    assert torch.equal(pol.mu[:n], fresh.mu[:n]) and torch.equal(pol.log_std[:n], fresh.log_std[:n])
    assert not pol.features[:n, 514:].any()
    p = probe_params(shape, 6, 3, r=2, u=5, perm=True)
    pol.load_state_dict(p)
    pol(images(shape, N, 300).to(DEV))
    pol(obs_dev)
    check_probe(pol, p, obs_dev, n)
    pol.close()
    fresh.close()


@pytest.mark.gpu
@pytest.mark.parametrize("shape", [(5, 64, 64), (4, 64, 64)], ids=["direct", "generic"])
def test_back_to_back_forwards_equal_isolated_ones(shape):
    """Forwards issued on one stream without a sync (every kernel is a programmatic dependent launch, and k_mlp_fused lets the next
    forward's conv1 start early), with alternating batch sizes and inputs and separate outputs: each equals its isolated forward."""
    N = 2 * _sm_count() + 1
    pol = _policy(shape, N, 6, trained_params(shape, seed=4))
    sizes = [N, 17, N - 2, 1, _sm_count(), 129, N]
    obs = [images(shape, n, 50 + i).to(DEV) for i, n in enumerate(sizes)]
    noise = [torch.randn(n, 6, device=DEV) if i % 2 else None for i, n in enumerate(sizes)]
    isolated = []
    for o, z in zip(obs, noise):
        isolated.append(pol(o, deterministic=z is None, noise=z).clone())
        torch.cuda.synchronize()
    outs = [torch.full((n, 6), float("nan"), device=DEV) for n in sizes]
    torch.cuda.synchronize()
    for o, z, out in zip(obs, noise, outs):
        pol(o, deterministic=z is None, noise=z, out=out)
    torch.cuda.synchronize()
    for i, (a, b) in enumerate(zip(outs, isolated)):
        assert torch.equal(a, b), (i, sizes[i])
    pol.close()
