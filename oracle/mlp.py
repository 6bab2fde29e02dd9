"""NumPy float32 restatement of the networks the reference evaluates inside the step (TEST INFRASTRUCTURE ONLY).

  * risk network  (train_risk_network.py; Keras SavedModel, layer list in keras_metadata.pb):
        Dense 512 selu -> Dense 256 selu -> Dense 128 selu -> Dense 1 sigmoid on [observation, action]
        (dropout 0.05 between the layers is inactive at inference), used by _is_action_risky
        (safe_motions_base.py:1498-1603).
  * backup policy (keras_fcnet_last_layer_activation.py:86-136, :187-202): Dense 256 swish -> Dense 128 swish ->
        Dense 2 n_joints tanh; the deterministic action (explore=False, safe_motions_base.py:632) is the first n_joints
        outputs (the rest parameterise log_std).
Weights: safemotionsrisk_b200/assets/networks_<scene>.npz (tools/export_networks.py).
"""
import numpy as np

SELU_SCALE, SELU_ALPHA = np.float32(1.0507009873554805), np.float32(1.6732632423543772)


def selu(x):
    return SELU_SCALE * np.where(x > 0, x, SELU_ALPHA * (np.exp(np.minimum(x, 0)) - 1)).astype(np.float32)


def swish(x):
    return (x / (1 + np.exp(-x))).astype(np.float32)


def risk_forward(w, obs, action):
    x = np.concatenate([obs, action], axis=1).astype(np.float32)
    for i in range(3):
        x = selu(x @ w["risk/dense_{}/kernel".format(i)] + w["risk/dense_{}/bias".format(i)])
    z = x @ w["risk/dense_3/kernel"] + w["risk/dense_3/bias"]
    return (1 / (1 + np.exp(-z)))[:, 0].astype(np.float32)


def backup_forward(w, obs, n_joints=7):
    x = obs.astype(np.float32)
    for name in ("fc_1", "fc_2"):
        x = swish(x @ w["backup/{}/kernel".format(name)] + w["backup/{}/bias".format(name)])
    out = np.tanh(x @ w["backup/fc_out/kernel"] + w["backup/fc_out/bias"]).astype(np.float32)
    return out[:, :n_joints]


def gate(w, obs, action, threshold, n_joints=7):
    """(gated actions, risk, risky) of actions.py:303-340 with the state-action risk network."""
    risk = risk_forward(w, obs, action)
    risky = risk >= np.float32(threshold)
    out = action.copy()
    out[risky] = backup_forward(w, obs[risky], n_joints)
    return out, risk, risky


# ---------------------------------------------------------------------------------------------- float64 references
# Generic networks: `layers` is a list of (kernel [in][out], bias [out]) pairs, the hidden layers followed by the output
# layer; hidden is "selu" or "swish", out is "sigmoid" or "tanh".

def shipped_layers(w, net):
    """Layer list of a shipped network: net = "risk", "backup" or "human"."""
    names = ["dense_{}".format(i) for i in range(4)] if net == "risk" else ["fc_1", "fc_2", "fc_out"]
    return [(w["{}/{}/kernel".format(net, n)], w["{}/{}/bias".format(net, n)]) for n in names]


def _act64(x, kind):
    if kind == "selu":
        return 1.0507009873554805 * np.where(x > 0, x, 1.6732632423543772 * np.expm1(np.minimum(x, 0)))
    if kind == "swish":
        return x / (1 + np.exp(-x))
    if kind == "sigmoid":
        return 1 / (1 + np.exp(-x))
    if kind == "tanh":
        return np.tanh(x)
    raise ValueError(kind)


def _f16(x):
    return np.asarray(x, dtype=np.float64).astype(np.float16).astype(np.float64)


def forward64(layers, x, hidden="selu", out="sigmoid"):
    """Plain float64 forward pass (the float32 parameters widened exactly)."""
    h = np.asarray(x, dtype=np.float64)
    for k, b in layers[:-1]:
        h = _act64(h @ np.asarray(k, np.float64) + np.asarray(b, np.float64), hidden)
    k, b = layers[-1]
    return _act64(h @ np.asarray(k, np.float64) + np.asarray(b, np.float64), out)


def forward_tc(layers, x, hidden="selu", out="sigmoid"):
    """float64 forward pass that rounds where mlp_kernel (smenv_mlp.cuh) rounds, and nowhere else: the inputs and the
    kernels of the hidden (tensor-core) layers to fp16 (round to nearest even); products summed in float64, the float32
    bias added and the activation applied in float64; a hidden activation that feeds another tensor-core layer to fp16.
    The last hidden activation stays unrounded: the kernel keeps it in fp32 registers and contracts it with the float32
    output kernel on the CUDA cores."""
    h = _f16(x)
    for i, (k, b) in enumerate(layers[:-1]):
        h = _act64(h @ _f16(k) + np.asarray(b, np.float64), hidden)
        if i < len(layers) - 2:
            h = _f16(h)
    k, b = layers[-1]
    return _act64(h @ np.asarray(k, np.float64) + np.asarray(b, np.float64), out)
