"""Packaged network weights (tools/export_networks.py) and the NumPy reference forward pass (oracle/mlp.py)."""
import os

import numpy as np
import pytest

from oracle import mlp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ASSETS = os.path.join(ROOT, "safemotionsrisk_b200", "assets")


@pytest.mark.parametrize("scene,obs", [("space", 23), ("ball", 27)])
def test_packaged_weights_have_the_checkpoint_shapes(scene, obs):
    """Observation widths 23 / 27 are those of risk_config.json and of the checkpoints' fc_1 kernels (SURVEY 8a a11)."""
    w = np.load(os.path.join(ASSETS, "networks_{}.npz".format(scene)))
    assert int(w["risk/observation_size"]) == obs and int(w["risk/action_size"]) == 7
    assert [w["risk/dense_{}/kernel".format(i)].shape for i in range(4)] == [(obs + 7, 512), (512, 256), (256, 128),
                                                                              (128, 1)]
    assert [w["backup/{}/kernel".format(n)].shape for n in ("fc_1", "fc_2", "fc_out")] == [(obs, 256), (256, 128),
                                                                                            (128, 14)]
    for k in w.files:
        assert np.all(np.isfinite(w[k]))


def test_reference_forward_is_well_behaved():
    w = np.load(os.path.join(ASSETS, "networks_space.npz"))
    rng = np.random.default_rng(0)
    obs = rng.uniform(-1, 1, (512, 23)).astype(np.float32)
    act = rng.uniform(-1, 1, (512, 7)).astype(np.float32)
    risk = mlp.risk_forward(w, obs, act)
    pol = mlp.backup_forward(w, obs)
    assert risk.shape == (512,) and np.all((risk >= 0) & (risk <= 1))
    assert pol.shape == (512, 7) and np.all(np.abs(pol) <= 1)
    assert risk.std() > 1e-3 and pol.std() > 1e-2           # trained weights, not constants
    gated, r, risky = mlp.gate(w, obs, act, 0.065)
    assert np.array_equal(gated[~risky], act[~risky]) and np.allclose(gated[risky], pol[risky])


@pytest.mark.parametrize("scene", ["space", "ball", "human"])
def test_float64_forward_agrees_with_the_float32_functions(scene):
    """forward64 restates the shipped networks: risk and backup policy of every scene and the human's policy (whose
    float32 forward pass is written out here, swish / tanh, 16 outputs)."""
    w = np.load(os.path.join(ASSETS, "networks_{}.npz".format(scene)))
    rng = np.random.default_rng(1)
    n_obs = w["backup/fc_1/kernel"].shape[0]
    obs = rng.uniform(-1, 1, (2000, n_obs)).astype(np.float32)
    act = rng.uniform(-1, 1, (2000, 7)).astype(np.float32)
    risk = mlp.forward64(mlp.shipped_layers(w, "risk"), np.concatenate([obs, act], 1), "selu", "sigmoid")[:, 0]
    assert np.abs(risk - mlp.risk_forward(w, obs, act)).max() < 1e-5
    pol = mlp.forward64(mlp.shipped_layers(w, "backup"), obs, "swish", "tanh")
    assert pol.shape == (2000, 14) and np.abs(pol[:, :7] - mlp.backup_forward(w, obs)).max() < 1e-5
    if scene == "human":
        hl = mlp.shipped_layers(w, "human")
        hobs = rng.uniform(-1, 1, (2000, hl[0][0].shape[0])).astype(np.float32)
        x = hobs
        for k, b in hl[:-1]:
            x = mlp.swish(x @ k + b)
        want = np.tanh(x @ hl[-1][0] + hl[-1][1]).astype(np.float32)
        got = mlp.forward64(hl, hobs, "swish", "tanh")
        assert got.shape == (2000, 16) and np.abs(got - want).max() < 1e-5


def _tiny(kernels, biases):
    return [(np.array(k, np.float32).reshape(len(k), -1), np.array(b, np.float32)) for k, b in zip(kernels, biases)]


def test_tensor_core_reference_rounds_exactly_where_the_kernel_does():
    """One-unit nets whose outputs tell each rounding point of forward_tc apart.  x = 1 and a bias of 2^-12 give a
    pre-activation 1 + 2^-12 that fp16 (spacing 2^-10 at 1) cannot hold: it must survive (sums and biases are not
    rounded), the activation that feeds a second tensor-core layer must be rounded, the last hidden activation must not;
    inputs and hidden kernels of 1 + 2^-13 round to 1, the output kernel keeps them."""
    f16 = lambda v: float(np.float16(v))   # noqa: E731
    s = mlp._act64
    one = np.ones((1, 1), np.float32)
    e12, e13 = 2.0 ** -12, 1 + 2.0 ** -13
    for hidden, out in (("selu", "sigmoid"), ("swish", "tanh"), ("selu", "tanh"), ("swish", "sigmoid")):
        # one tensor-core layer: the sum, the bias and the (last) hidden activation stay unrounded
        net1 = _tiny([[1.0], [1.0]], [[e12], [0.0]])
        h = s(np.float64(1 + e12), hidden)
        assert f16(h) != h
        assert mlp.forward_tc(net1, one, hidden, out)[0, 0] == s(h, out)
        assert mlp.forward_tc(net1, one, hidden, out)[0, 0] != s(f16(h), out)
        assert mlp.forward_tc(net1, one, hidden, out)[0, 0] == mlp.forward64(net1, one, hidden, out)[0, 0]
        # two tensor-core layers: the first activation is rounded to fp16 before it meets the second kernel, the second
        # (last) one is not
        net2 = _tiny([[1.0], [1.0], [1.0]], [[e12], [e12], [0.0]])
        h2 = s(f16(h) + e12, hidden)
        assert f16(h2) != h2
        assert mlp.forward_tc(net2, one, hidden, out)[0, 0] == s(h2, out)
        assert mlp.forward_tc(net2, one, hidden, out)[0, 0] != s(f16(h2), out)
        assert mlp.forward_tc(net2, one, hidden, out)[0, 0] != mlp.forward64(net2, one, hidden, out)[0, 0]
        # the input and the hidden kernel go to fp16, the output kernel stays float32
        x13 = np.full((1, 1), e13, np.float32)
        assert mlp.forward_tc(net1, x13, hidden, out)[0, 0] == mlp.forward_tc(net1, one, hidden, out)[0, 0]
        assert mlp.forward_tc(_tiny([[e13], [1.0]], [[e12], [0.0]]), one, hidden, out)[0, 0] == s(h, out)
        assert mlp.forward_tc(_tiny([[1.0], [e13]], [[e12], [0.0]]), one, hidden, out)[0, 0] == s(h * np.float64(
            np.float32(e13)), out)
        assert mlp.forward64(net1, x13, hidden, out)[0, 0] != mlp.forward64(net1, one, hidden, out)[0, 0]


def test_activation_closed_forms():
    x = np.array([-2.0, -0.5, 0.0, 0.5, 2.0], dtype=np.float32)
    assert np.allclose(mlp.selu(x)[2:], 1.0507009873554805 * x[2:])
    assert np.allclose(mlp.selu(x)[:2], 1.0507009873554805 * 1.6732632423543772 * (np.exp(x[:2]) - 1), rtol=1e-6)
    assert np.allclose(mlp.swish(x), x / (1 + np.exp(-x)))
