"""The float64 reference of the agent's DiagGaussian head (tests/agent_reference.py) against scipy, on the CPU."""
import numpy as np
import pytest

from agent_reference import agent_eps, diag_gaussian, philox

stats = pytest.importorskip("scipy.stats")

LO, HI = -1.375, 0.0


def test_logp_is_the_diag_gaussian_density_of_the_unclipped_sample():
    rng = np.random.default_rng(0)
    nj, n = 7, 4096
    out = rng.uniform(-1, 1, (n, 2 * nj))
    eps = rng.standard_normal((n, nj)) * 2.0
    sample, clipped, logp, dist = diag_gaussian(out, nj, LO, HI, eps)
    mean, log_std = dist[:, :nj], dist[:, nj:]
    want = stats.norm.logpdf(sample, loc=mean, scale=np.exp(log_std)).sum(1)
    assert np.abs(logp - want).max() < 1e-10
    assert (np.abs(sample) > 1).any()                        # some samples leave the action box ...
    assert np.array_equal(clipped, np.clip(sample, -1, 1))   # ... the env gets them clipped, the log-likelihood does not
    assert np.abs(clipped).max() == 1.0


def test_remap_and_clip_at_the_edges():
    nj = 3
    out = np.array([[1.0, -1.0, 0.0, -1.0, 1.0, 0.0]])
    _, _, _, dist = diag_gaussian(out, nj, LO, HI, np.zeros((1, nj)))
    assert dist[0, nj:].tolist() == [LO, HI, 0.5 * (LO + HI)]      # t = -1 -> lo, t = 1 -> hi
    eps = np.array([[10.0, -10.0, 0.0]])
    sample, clipped, _, _ = diag_gaussian(out, nj, LO, HI, eps)
    assert clipped.tolist() == [[1.0, -1.0, 0.0]]
    assert sample[0, 0] > 1 and sample[0, 1] < -1


def test_deterministic_head_is_the_mean_with_zero_logp():
    rng = np.random.default_rng(1)
    out = rng.uniform(-1, 1, (64, 14))
    sample, clipped, logp, dist = diag_gaussian(out, 7, LO, HI, None)
    assert np.array_equal(sample, out[:, :7]) and np.array_equal(clipped, out[:, :7])
    assert not logp.any()
    assert np.array_equal(dist[:, :7], out[:, :7])


def test_agent_noise_is_standard_normal_and_depends_on_every_stream_word():
    eps = agent_eps(65536, 7, 3, 3)
    assert stats.kstest(eps.ravel(), "norm").pvalue > 1e-3
    assert not np.array_equal(eps, agent_eps(65536, 7, 4, 3))       # step counter
    assert not np.array_equal(eps, agent_eps(65536, 7, 3, 4))       # seed
    assert not np.array_equal(eps[:, 0], eps[:, 1])                 # joint
    human = philox(np.arange(16), 3, 0, 0x4057, 3, 0)[0]              # the human's stream of the same env and step
    assert not np.array_equal(human, philox(np.arange(16), 3, 0, 0xA6E7, 3, 0)[0])
