"""ORACLE (test infrastructure, never on the product path): fp32 torch restatement of the rollout policy forward.

Follows
  * SB3 `preprocess_obs` — uint8 image observations are divided by 255 (all C channels, so the two direct features arrive
    as v/255; SURVEY.md §3.4),
  * reference models/feature_extractor.py:19-49 `AugmentedNatureCNN`: NatureCNN on the first C-1 channels -> 512, concat
    observation[:, -1, 0, :2] -> 514,
  * SB3 sac/policies.py `Actor`: latent_pi = MLP(514 -> 256 -> 256, ReLU) (net_arch from reference train_agent.py:18-20),
    mu = Linear(256, A), log_std = Linear(256, A) clamped to [-20, 2], action = tanh(mu [+ exp(log_std) * noise]).
Pinned by tests/golden/policy_vectors.npz: the feature part against the reference's own AugmentedNatureCNN class executed in
the build container (tools/gen_policy_golden.py); the SB3 actor head is absent from /root/reference (third-party,
un-vendored) and is restated from its published definition.
"""
import numpy as np
import torch
import torch.nn.functional as F

LOG_STD_MIN, LOG_STD_MAX = -20.0, 2.0


def _t(params, name):
    v = params[name]
    return v if isinstance(v, torch.Tensor) else torch.as_tensor(np.asarray(v), dtype=torch.float32)


def features(params, obs_u8):
    """obs uint8 [n, C, H, W] (tensor or array) -> float32 [n, 514]."""
    obs = torch.as_tensor(np.asarray(obs_u8)) if not isinstance(obs_u8, torch.Tensor) else obs_u8
    x = obs.to(torch.float32) / 255.0
    img, pad = x[:, :-1], x[:, -1]
    p = "features_extractor."
    h = F.relu(F.conv2d(img, _t(params, p + "cnn.0.weight"), _t(params, p + "cnn.0.bias"), stride=4))
    h = F.relu(F.conv2d(h, _t(params, p + "cnn.2.weight"), _t(params, p + "cnn.2.bias"), stride=2))
    h = F.relu(F.conv2d(h, _t(params, p + "cnn.4.weight"), _t(params, p + "cnn.4.bias"), stride=1))
    h = h.flatten(1)
    h = F.relu(F.linear(h, _t(params, p + "linear.0.weight"), _t(params, p + "linear.0.bias")))
    return torch.cat((h, pad[:, 0, :2]), dim=1)


def actor(params, obs_u8, noise=None):
    """-> dict(features, mu, log_std, action) float32 tensors."""
    f = features(params, obs_u8)
    h = F.relu(F.linear(f, _t(params, "latent_pi.0.weight"), _t(params, "latent_pi.0.bias")))
    h = F.relu(F.linear(h, _t(params, "latent_pi.2.weight"), _t(params, "latent_pi.2.bias")))
    mu = F.linear(h, _t(params, "mu.weight"), _t(params, "mu.bias"))
    log_std = torch.clamp(F.linear(h, _t(params, "log_std.weight"), _t(params, "log_std.bias")), LOG_STD_MIN, LOG_STD_MAX)
    pre = mu if noise is None else mu + torch.exp(log_std) * torch.as_tensor(np.asarray(noise), dtype=torch.float32)
    return dict(features=f, mu=mu, log_std=log_std, action=torch.tanh(pre))


# ------------------------------------------------------------------------------------------------ rounding-faithful fp64 layers
# The tensor-core kernels (policy_kernels.cu) round at fixed points: conv1 multiplies raw uint8 pixels (exact in fp16) by fp16
# weights and applies fmaf(acc, 1.0f/255.0f, b); every other layer multiplies bf16 activations by bf16 weights and adds its fp32
# bias; every hidden activation is stored as bf16 (round to nearest even), mu / log_std as fp32.  The functions below restate
# each layer in fp64 from the layer's own input, with the kernel's rounded weights, and return y* (the exact value before the
# output rounding) together with s * sum |x| |w| (s the accumulator scale), from which `ratio_bf16` / `ratio_fp32` bound the
# kernel's error: fp32 accumulation of K exact products loses at most K * 2^-23 * sum |x w| (one ulp per addition, a bound that
# also holds for truncating adders), the fp32 epilogue one 2^-24 relative rounding, and the bf16 store half a bf16 ulp.
S_CONV1 = float(np.float32(1.0) / np.float32(255.0))  # the kernel's 1.0f / 255.0f, itself an fp32 rounding of 1/255
U23, U24 = 2.0 ** -23, 2.0 ** -24
FEAT_LD = 576  # the feature matrix's row: 512 CNN features, the two direct features, zero padding


def bf16(x):
    """fp32 -> bf16, round to nearest even, returned as fp64 (the stores of the kernels: the value is first an fp32)."""
    return x.to(torch.float32).to(torch.bfloat16).to(torch.float64)


def kernel_weights(params, device="cpu"):
    """The parameters as the kernels multiply them (fp64 tensors in the torch layouts): conv1 weights rounded to fp16, every
    other weight to bf16, biases fp32."""
    out = {}
    for k, v in params.items():
        t = _t(params, k).to(torch.float32).to(device)
        if k.endswith("bias"):
            out[k] = t.to(torch.float64)
        elif k == "features_extractor.cnn.0.weight":
            out[k] = t.to(torch.float16).to(torch.float64)
        else:
            out[k] = bf16(t)
    return out


def _conv(x, w, stride):
    # fp64 convolution as an explicit im2col product: no algorithm choice of a convolution library enters the reference
    n, (o, _, kh, kw) = x.shape[0], w.shape
    oh, ow = (x.shape[2] - kh) // stride + 1, (x.shape[3] - kw) // stride + 1
    cols = F.unfold(x, (kh, kw), stride=stride)
    return (w.reshape(o, -1) @ cols).reshape(n, o, oh, ow)


def _layer(z, za, bias, scale, relu=True):
    shape = (1, -1) + (1,) * (z.dim() - 2)
    y = scale * z + bias.reshape(shape)
    return (y.clamp_min(0.0) if relu else y), scale * za


def conv1(kw, obs_u8):
    """obs uint8 [n, C, H, W] -> (y*, s * sum|x||w|) [n, 32, o1h, o1w]; K = (C - 1) * 64."""
    x = obs_u8[:, :-1].to(torch.float64)
    w = kw["features_extractor.cnn.0.weight"]
    return _layer(_conv(x, w, 4), _conv(x, w.abs(), 4), kw["features_extractor.cnn.0.bias"], S_CONV1)


def conv2(kw, act1):
    """act1 [n, 32, o1h, o1w] (the kernel's bf16 values) -> [n, 64, o2h, o2w]; K = 512."""
    w, x = kw["features_extractor.cnn.2.weight"], act1.to(torch.float64)
    return _layer(_conv(x, w, 2), _conv(x.abs(), w.abs(), 2), kw["features_extractor.cnn.2.bias"], 1.0)


def conv3(kw, act2):
    """act2 [n, 64, o2h, o2w] -> [n, 64, o3h, o3w]; K = 576."""
    w, x = kw["features_extractor.cnn.4.weight"], act2.to(torch.float64)
    return _layer(_conv(x, w, 1), _conv(x.abs(), w.abs(), 1), kw["features_extractor.cnn.4.bias"], 1.0)


def linear(kw, act3):
    """act3 [n, 64, o3h, o3w] (torch's flatten order is (c, y, x)) -> [n, 512]; K = nflat."""
    x, w = act3.to(torch.float64).flatten(1), kw["features_extractor.linear.0.weight"]
    return _layer(x @ w.T, x.abs() @ w.abs().T, kw["features_extractor.linear.0.bias"], 1.0)


def direct_features(obs_u8):
    """The two direct features exactly as stored: bf16(float(p) * (1.0f / 255.0f)) with an fp32 product."""
    return bf16(obs_u8[:, -1, 0, :2].to(torch.float32) * torch.tensor(S_CONV1, dtype=torch.float32))


def dense(kw, name, x, relu=True):
    """latent_pi.0 (x = the 514 features, K = 576 with the zero padding), latent_pi.2 (K = 256) or a head half (mu / log_std,
    K = 256, relu=False)."""
    x, w = x.to(torch.float64), kw[name + ".weight"]
    return _layer(x @ w.T, x.abs() @ w.abs().T, kw[name + ".bias"], 1.0, relu)


def log_std(kw, h2):
    y, a = dense(kw, "log_std", h2, relu=False)
    return y.clamp(LOG_STD_MIN, LOG_STD_MAX), a  # clamping is 1-Lipschitz: the bound of the unclamped value still holds


def ulp(v, mant_bits):
    """ulp of |v| in a binary format with `mant_bits` stored mantissa bits and fp32's exponent range (bf16: 7, fp32: 23)."""
    e = torch.frexp(v.abs().to(torch.float64))[1].to(torch.float64) - 1  # floor(log2 |v|)
    e = torch.where(v == 0, torch.full_like(e, -126.0), e.clamp_min(-126.0))
    return torch.exp2(e - mant_bits)


def ratio_bf16(y_gpu, y_star, acc_abs, K):
    """|y_gpu - y*| / (1/2 ulp_bf16(max(|y*|, |y_gpu|)) + K 2^-23 s sum|x||w| + 2^-24 |y*|), elementwise."""
    y_gpu = y_gpu.to(torch.float64)
    bound = 0.5 * ulp(torch.maximum(y_star.abs(), y_gpu.abs()), 7) + K * U23 * acc_abs + U24 * y_star.abs()
    return (y_gpu - y_star).abs() / bound


def ratio_fp32(y_gpu, y_star, acc_abs, K):
    """The same for an fp32 output: no store rounding beyond the epilogue's, taken as 2^-23 |y*|."""
    y_gpu = y_gpu.to(torch.float64)
    bound = K * U23 * acc_abs + U23 * y_star.abs()
    return (y_gpu - y_star).abs() / torch.where(bound > 0, bound, torch.full_like(bound, 1e-300))


# CUDA's documented maximum errors (CUDA C++ Programming Guide, mathematical functions): tanhf 2 ulp; the __expf intrinsic
# 2 + floor(|1.173 x|) ulp.
def ratio_action(a_gpu, mu_gpu, ls_gpu=None, noise=None):
    """Action a = tanhf(mu [+ __expf(ls) * noise]) against tanh in fp64 from the kernel's own fp32 mu / log_std."""
    mu = mu_gpu.to(torch.float64)
    if noise is None:
        pre, dpre = mu, torch.zeros_like(mu)
    else:
        ls, nz = ls_gpu.to(torch.float64), noise.to(torch.float64).abs()
        e = torch.exp(ls)
        nulp = 2.0 + torch.floor((1.173 * ls).abs())
        e_err = nulp * ulp(e * (1.0 + nulp * U23), 23)  # the ulp of the larger of exp(ls) and the returned value
        pre = mu + e * noise.to(torch.float64)
        # __expf's error times |noise|; then the product and the sum each round once in fp32 (or fewer times, as an fma)
        dprod = e_err * nz + U24 * (e + e_err) * nz
        dpre = dprod + U24 * (pre.abs() + dprod)
    a_star = torch.tanh(pre)
    # tanh' = sech^2 is largest where |pre| is smallest: its value at max(|pre*| - dpre, 0) bounds the slope over the interval
    slope = 1.0 / torch.cosh((pre.abs() - dpre).clamp_min(0.0)) ** 2
    a = a_gpu.to(torch.float64)
    bound = slope * dpre + 2.0 * ulp(torch.maximum(a.abs(), a_star.abs() + slope * dpre), 23)
    return (a - a_star).abs() / bound
