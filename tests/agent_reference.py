"""Float64 reference of the agent's DiagGaussian head (agent_action_kernel, smenv_mlp.cuh) and the NumPy restatement of its
Philox normal noise, shared by test_agent_cpu.py and test_gpu_agent.py.

RLlib's DiagGaussian (rllib/models/tf/tf_action_dist.py) over the outputs of a Keras fcnet with a tanh last layer
(keras_fcnet_last_layer_activation.py:187-202): the first nj outputs are the means, the last nj the log-std
pre-activations t, remapped to log_std = lo + (t + 1) / 2 (hi - lo).  A sample is mean + exp(log_std) eps, the env
executes it clipped to [-1, 1] (RLlib's clip_actions) and its log-likelihood is that of the unclipped sample.
"""
import numpy as np

AGENT_TAG = 0xA6E7   # fourth Philox counter word of the agent's noise


def diag_gaussian(out, nj, lo, hi, eps):
    """(sample, clipped sample, logp, dist inputs) in float64 for network outputs out [N, 2 nj] and standard normal noise
    eps [N, nj]; eps None: the deterministic action (the mean, logp 0)."""
    out = np.asarray(out, np.float64)
    mean = out[:, :nj]
    log_std = lo + 0.5 * (out[:, nj:2 * nj] + 1.0) * (hi - lo)
    if eps is None:
        sample, logp = mean.copy(), np.zeros(out.shape[0])
    else:
        eps = np.asarray(eps, np.float64)
        sample = mean + np.exp(log_std) * eps
        logp = -0.5 * (eps ** 2).sum(1) - log_std.sum(1) - 0.5 * nj * np.log(2.0 * np.pi)
    return sample, np.clip(sample, -1.0, 1.0), logp, np.concatenate([mean, log_std], axis=1)


def philox(c0, c1, c2, c3, k0, k1):
    """Philox4x32-10 over arrays (philox of smenv_device.cuh)."""
    m = np.uint64(0xFFFFFFFF)
    c = [np.asarray(v, np.uint64) & m for v in (c0, c1, c2, c3)]
    k0, k1 = np.uint64(k0), np.uint64(k1)
    for _ in range(10):
        p0, p1 = np.uint64(0xD2511F53) * c[0], np.uint64(0xCD9E8D57) * c[2]
        c = [((p1 >> np.uint64(32)) ^ c[1] ^ k0) & m, p1 & m, ((p0 >> np.uint64(32)) ^ c[3] ^ k1) & m, p0 & m]
        k0, k1 = (k0 + np.uint64(0x9E3779B9)) & m, (k1 + np.uint64(0xBB67AE85)) & m
    return [v.astype(np.uint32) for v in c]


def agent_eps(n, nj, step, seed):
    """The agent's noise [n, nj] of the step with counter `step`: Philox stream (env, step, joint, 0xA6E7), key = seed,
    Box-Muller in float32 (diag_gaussian_sample of smenv_device.cuh)."""
    e, j = np.meshgrid(np.arange(n), np.arange(nj), indexing="ij")
    r = philox(e, step, j, AGENT_TAG, seed & 0xFFFFFFFF, seed >> 32)
    u01 = lambda v: (v >> np.uint32(8)).astype(np.float32) * np.float32(1.0 / 16777216.0)   # noqa: E731
    u1, u2 = np.maximum(u01(r[0]), np.float32(5.9604645e-8)), u01(r[1])
    return np.sqrt(np.float32(-2) * np.log(u1)) * np.cos(np.float32(np.pi) * (np.float32(2) * u2))
