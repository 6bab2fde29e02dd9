"""The network kernels of smenv_mlp.cuh value by value against float64 references (oracle/mlp.py).

mlp_kernel (tcgen05, fp16 operands, fp32 accumulators) is compared with forward_tc, a float64 forward pass that rounds
exactly where the kernel rounds (inputs, hidden kernels and every hidden activation but the last to fp16).  What is left
is the kernel's fp32 summation and its fast exp: now and then they flip the fp16 rounding of an activation by one ulp.
The mean error per output column stays near 1e-6 (measured on a B200: at most 2.5e-6 over all tests here), while a
dropped K block, a dropped block of the output contraction, a bias shifted by one column or fp16 rounding toward zero
each cost 2e-5 to 1e-1: the mean bound of 1e-5 (over at least 128 rows) is what tells a wrong kernel.  The maximum is
the tail of the flips: a CPU emulation of the kernel's arithmetic (fp16 operands, float32 sums and activations) reaches
2.2e-3 against forward_tc on 65 536 uniform rows of the human's policy and 1.6e-3 on the Ball backup policy, and the
B200 2.5e-3 on a log-std column of the Ball backup policy, so the max bound is 4e-3 per column.

mlp_exact_kernel (float32 on the CUDA cores) is compared with forward64 to 2e-5, the precision of any float32
evaluation of the shipped backup policies: their last hidden activations reach 27 and their pre-tanh sums 76, where a
float32 ulp is 2e-6 to 8e-6, and a NumPy float32 forward pass of the Space and Ball backup policies differs from
float64 by up to 1.3e-5 and 1.5e-5 on 65 536 uniform rows.

Row counts cross the tile and grid boundaries of mlp_kernel: one CTA per SM, 128 rows per tile, so above 128 x SMs
rows a CTA loops over tiles, and the weight prefetch ring and the partial-sum buffer carry over from tile to tile.
"""
import os
import zlib

import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

from oracle import mlp, oracle  # noqa: E402
from safemotionsrisk_b200 import (ball_backup_config, cabi, human_backup_config, space_backup_config,  # noqa: E402
                                  space_task_config)

ASSETS = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "safemotionsrisk_b200", "assets")
MAX_TOL, MEAN_TOL, EXACT_TOL = 4e-3, 1e-5, 2e-5
HIDDEN, OUT = {"selu": 0, "swish": 1}, {"sigmoid": 0, "tanh": 1}
WIDTHS = (16, 32, 48, 64, 128, 192, 256, 512)
FULL = 65536
SM_ERR_ARG, SM_ERR_STATE = -1, -4   # SmStatus (include/smenv.h)


def sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


def tile_rows():
    """Row counts around one tile, one tile per CTA (128 x SMs) and several uneven tiles per CTA."""
    g = 128 * sms()
    return [1, 127, 128, 129, g - 1, g, g + 1, 3 * g + 77, 65536, 100003]


def make_env(cfg, n, **kw):
    from safemotionsrisk_b200.vec_env import SafeMotionsVecEnv
    opts = dict(seed=3, auto_reset=False)
    opts.update(kw)
    return SafeMotionsVecEnv(num_envs=n, config=cfg, **opts)


@pytest.fixture(scope="module")
def env():
    """Slots 0 and 1 take the networks under test; the row count of smenv_mlp_forward does not depend on num_envs."""
    e = make_env(space_backup_config(ball_machine_mode=True), 128, fill_pools=False)
    yield e
    e.close()


def load(env, slot, layers, hidden, out):
    """smenv_mlp_load of a (kernel, bias) list; returns the status code."""
    dims = np.array([layers[0][0].shape[0]] + [k.shape[1] for k, _ in layers], dtype=np.int32)
    flat = np.concatenate([np.concatenate([np.asarray(k, np.float32).ravel(), np.asarray(b, np.float32).ravel()])
                           for k, b in layers])
    return env._lib.smenv_mlp_load(env._handle, slot, len(layers) - 1, dims.ctypes.data, HIDDEN[hidden], OUT[out],
                                   flat.ctypes.data)


def load_ok(env, slot, layers, hidden, out):
    cabi.check(load(env, slot, layers, hidden, out), "smenv_mlp_load")


def random_net(rng, n_in, hidden, n_out):
    dims = [n_in] + list(hidden) + [n_out]
    return [(rng.normal(0, 1.0 / np.sqrt(dims[i]), (dims[i], dims[i + 1])).astype(np.float32),
             rng.normal(0, 0.1, dims[i + 1]).astype(np.float32)) for i in range(len(dims) - 1)]


def tc(env, slot, x, n_out):
    return env.mlp_forward(slot, x, None, n_out=n_out).cpu().numpy()


def exact(env, slot, x, n_out):
    return env.mlp_forward_exact(slot, x, None, n_out=n_out).cpu().numpy()


def check_tc(got, want, what):
    """max <= MAX_TOL per output column, and mean <= MEAN_TOL per column over at least 128 rows; returns (max, mean)."""
    d = np.abs(got.astype(np.float64) - want)
    mx, mn = d.max(0), d.mean(0)
    print("tc {}: rows {} max {:.2e} mean {:.2e}".format(what, d.shape[0], mx.max(), mn.max()))
    assert (mx <= MAX_TOL).all(), "{}: max error per column {}".format(what, mx)
    if d.shape[0] >= 128:
        assert (mn <= MEAN_TOL).all(), "{}: mean error per column {}".format(what, mn)
    return mx.max(), mn.max()


def check_exact(got, want, what):
    d = np.abs(got.astype(np.float64) - want)
    print("exact {}: rows {} max {:.2e}".format(what, d.shape[0], d.max()))
    assert d.max() <= EXACT_TOL, "{}: max error per column {}".format(what, d.max(0))


# ---------------------------------------------------------------------------------------------- shapes
def _edge_shapes():
    """(n_in, hidden widths, n_out, hidden activation, output activation) at the edges of what smenv_mlp_load accepts."""
    acts = [("selu", "sigmoid"), ("swish", "tanh"), ("selu", "tanh"), ("swish", "sigmoid")]
    shapes = []
    for i, n_in in enumerate((1, 16, 17, 32, 33, 64)):                  # k_in padding to 16 / 32 / 64
        shapes.append((n_in, (64,), 1 + i % 3, *acts[i % 4]))
    for i, hidden in enumerate([(16,), (32,), (48,), (64,), (128,), (192,), (256,), (48, 48), (16, 16, 16),
                                (512, 512, 256), (512, 128), (192, 48, 16), (256, 256, 256), (64, 512, 64)]):
        shapes.append((30, hidden, 7, *acts[i % 4]))                       # 512 -> 512: 32-column chunks; 48: one chunk
    for i, n_out in enumerate((1, 2, 7, 8, 9, 15, 16)):
        shapes.append((23, (256, 128), n_out, *acts[i % 4]))
    shapes.append((38, (256, 128), 16, "swish", "tanh"))                  # 128 x 16 = the 2048-float w_out limit
    shapes.append((38, (512, 256), 8, "selu", "sigmoid"))                 # 256 x 8
    for hidden_act, out_act in acts:
        shapes.append((33, (48, 128), 9, hidden_act, out_act))          # a 48-column K chunk, 16 outputs
    return shapes


def _sampled_shapes(count=40):
    rng = np.random.default_rng(2024)
    shapes = []
    while len(shapes) < count:
        hidden = tuple(int(w) for w in rng.choice(WIDTHS, size=int(rng.integers(1, 4))))
        n_out = int(rng.integers(1, 17))
        if hidden[-1] > 256 or hidden[-1] * (8 if n_out <= 8 else 16) > 2048:
            continue
        shapes.append((int(rng.integers(1, 65)), hidden, n_out, ("selu", "swish")[rng.integers(2)],
                       ("sigmoid", "tanh")[rng.integers(2)]))
    return shapes


SHAPES = _edge_shapes() + _sampled_shapes()


@pytest.mark.parametrize("shape", SHAPES, ids=["{}-{}-{}-{}-{}".format(s[0], "x".join(map(str, s[1])), *s[2:])
                                                for s in SHAPES])
def test_every_accepted_shape_matches_the_rounding_reference(env, shape):
    """Both kernels on 333 rows of every edge shape and of a seeded sample of accepted shapes: input widths at the
    16 / 32 / 64 padding edges, every hidden width, 1 to 3 layers, 1 to 16 outputs, both hidden and both output
    activations.  Measured on a B200 (1000 W power limit), worst shape: tensor cores max 3.0e-4, mean 2.5e-6; exact max 1.1e-6."""
    n_in, hidden, n_out, hidden_act, out_act = shape
    rng = np.random.default_rng(zlib.crc32(repr(shape).encode()))
    net = random_net(rng, n_in, hidden, n_out)
    load_ok(env, 0, net, hidden_act, out_act)
    assert env.mlp_shape(0) == (n_in, n_out)
    x = rng.uniform(-1, 1, (333, n_in)).astype(np.float32)
    check_tc(tc(env, 0, x, n_out), mlp.forward_tc(net, x, hidden_act, out_act), str(shape))
    check_exact(exact(env, 0, x, n_out), mlp.forward64(net, x, hidden_act, out_act), str(shape))


REFUSED = {
    "no hidden layer": (0, [30, 1]),
    "four hidden layers": (4, [30, 64, 64, 64, 64, 1]),
    "no input": (1, [0, 64, 1]),
    "65 inputs": (1, [65, 64, 1]),
    "width 80": (2, [30, 80, 64, 1]),
    "width 96": (2, [30, 96, 64, 1]),
    "width 320": (2, [30, 320, 64, 1]),
    "last hidden 512": (2, [30, 256, 512, 1]),
    "256 x 16 outputs": (2, [30, 512, 256, 16]),
    "256 x 9 outputs": (1, [30, 256, 9]),
    "no output": (1, [30, 64, 0]),
    "17 outputs": (1, [30, 64, 17]),
}


@pytest.mark.parametrize("name", sorted(REFUSED))
def test_unsupported_shapes_are_refused(env, name):
    """smenv_mlp_load refuses what mlp_kernel cannot run, and the slot keeps the network it had."""
    n_tc, dims = REFUSED[name]
    load_ok(env, 1, random_net(np.random.default_rng(0), 23, (64,), 5), "swish", "tanh")
    weights = np.zeros(sum(max(dims[i], 1) * (max(dims[i + 1], 1) + 1) for i in range(len(dims) - 1)), np.float32)
    d = np.array(dims, dtype=np.int32)
    assert env._lib.smenv_mlp_load(env._handle, 1, n_tc, d.ctypes.data, 0, 0, weights.ctypes.data) == SM_ERR_ARG
    assert env.mlp_shape(1) == (23, 5)


# ---------------------------------------------------------------------------------------------- rows
def _row_nets():
    w_space, w_human = np.load(os.path.join(ASSETS, "networks_space.npz")), np.load(os.path.join(ASSETS, "networks_human.npz"))
    rng = np.random.default_rng(77)
    return {
        "space_risk": (mlp.shipped_layers(w_space, "risk"), "selu", "sigmoid"),
        "human_policy": (mlp.shipped_layers(w_human, "human"), "swish", "tanh"),
        "512x512x256_8": (random_net(rng, 17, (512, 512, 256), 8), "swish", "tanh"),
        "48_9": (random_net(rng, 33, (48,), 9), "selu", "sigmoid"),
    }


ROW_NETS = _row_nets()
_ROW_CACHE = {}


def _row_case(name):
    """Inputs of the largest row count and their references; smaller row counts take a prefix."""
    if name not in _ROW_CACHE:
        layers, hidden, out = ROW_NETS[name]
        x = np.random.default_rng(5).uniform(-1, 1, (max(tile_rows()), layers[0][0].shape[0])).astype(np.float32)
        _ROW_CACHE[name] = (x, mlp.forward_tc(layers, x, hidden, out))
    return _ROW_CACHE[name]


@pytest.mark.parametrize("name", sorted(ROW_NETS))
def test_row_counts_across_tiles_and_ctas(env, name):
    """mlp_kernel at every row count of tile_rows(): a partial first tile, one tile per CTA, and 2 to 6 tiles per CTA
    spread unevenly over the CTAs (128 x SMs x 3 + 77, 65 536, 100 003).  Every count agrees with the reference, and a
    row gives the same bits at every count.  Measured on a B200 (1000 W power limit), worst row count: Space risk max 4.8e-4, mean 1.2e-6;
    human's policy max 1.0e-3, mean 8.4e-7; 17 -> 512 -> 512 -> 256 -> 8 max 8.3e-5, mean 1.5e-6; 33 -> 48 -> 9 max
    1.3e-7, mean 4.3e-8."""
    layers, hidden, out = ROW_NETS[name]
    x, want = _row_case(name)
    n_out = want.shape[1]
    load_ok(env, 0, layers, hidden, out)
    xd = torch.from_numpy(x).cuda()
    first = None
    for n in tile_rows():
        got = tc(env, 0, xd[:n], n_out)
        check_tc(got, want[:n], "{} at {} rows".format(name, n))
        if first is not None:
            k = min(n, first.shape[0])
            assert np.array_equal(got[:k], first[:k]), "{}: rows change bits with the row count {}".format(name, n)
        if first is None or n > first.shape[0]:
            first = got


def test_shipped_networks_at_full_size(env, rollouts):
    """All seven shipped networks at 65 536 rows, on uniform [-1, 1] inputs and on observations of a short rollout:
    risk network and backup policy (all 14 outputs) of the Space, Ball and Human scenes, and the human's policy (16
    outputs), on the tensor cores against forward_tc and in float32 against forward64.  Measured on a B200 (1000 W power limit), uniform /
    rollout rows, tensor cores max (mean): Space risk 9.4e-4 (1.2e-6) / 4.8e-4 (8.9e-7), backup 9.7e-4 (7.6e-7) /
    8.8e-4 (7.6e-7); Ball risk 1.0e-3 (7.0e-7) / 7.0e-4 (8.1e-7), backup 2.5e-3 (8.1e-7) / 1.0e-3 (7.1e-7); Human risk
    5.8e-4 (8.6e-7) / 6.4e-4 (8.2e-7), backup 2.5e-4 (3.8e-7) / 4.0e-4 (4.0e-7), human's policy 1.0e-3 (4.4e-7) /
    6.8e-4 (7.3e-7).  Exact max: 1.4e-5 (Ball backup, uniform), 1.1e-5 (Space backup, rollout), the others 1.4e-6 to
    9.6e-6."""
    rng = np.random.default_rng(12)
    for scene in ("space", "ball", "human"):
        w = np.load(os.path.join(ASSETS, "networks_{}.npz".format(scene)))
        ro = rollouts[{"space": "space_bm", "ball": "ball_bm", "human": "human"}[scene]]
        obs = ro.risk_observation().cpu().numpy()
        nets = [("risk", "selu", "sigmoid"), ("backup", "swish", "tanh")] + ([("human", "swish", "tanh")] if scene == "human" else [])
        for net, hidden, out in nets:
            layers = mlp.shipped_layers(w, net)
            n_in, n_out = layers[0][0].shape[0], layers[-1][0].shape[1]
            if net == "risk":
                observed = np.concatenate([obs, rng.uniform(-1, 1, (FULL, 7)).astype(np.float32)], 1)
            elif net == "human":
                observed = ro.hobs.cpu().numpy()[:, :n_in]
            else:
                observed = obs
            load_ok(env, 1, layers, hidden, out)
            for kind, x in (("uniform", rng.uniform(-1, 1, (FULL, n_in)).astype(np.float32)), ("rollout", observed)):
                what = "{} {} {}".format(scene, net, kind)
                check_tc(tc(env, 1, x, n_out), mlp.forward_tc(layers, x, hidden, out), what)
                check_exact(exact(env, 1, x, n_out), mlp.forward64(layers, x, hidden, out), what)


def test_exact_kernel_past_its_block_cap(env):
    """mlp_exact_kernel launches at most 4 x SMs blocks of 16 rows and strides over the rest: twice that many rows and
    an odd remainder, 16 outputs.  Measured on a B200 (1000 W power limit): max 5.5e-6."""
    layers, hidden, out = ROW_NETS["human_policy"]
    load_ok(env, 1, layers, hidden, out)
    n = 2 * 4 * sms() * 16 + 37
    x = np.random.default_rng(8).uniform(-1, 1, (n, layers[0][0].shape[0])).astype(np.float32)
    check_exact(exact(env, 1, x, 16), mlp.forward64(layers, x, hidden, out), "human policy at {} rows".format(n))


@pytest.mark.parametrize("name", ["space_risk", "human_policy"])
def test_a_row_gives_the_same_bits_wherever_it_sits(env, name):
    """Row 70 001 of 100 003 alone, in place, inside a permuted batch and over two launches: the same bits from both
    kernels (every row is computed by one thread's fixed sequence of operations, whatever the tile and CTA)."""
    layers, hidden, out = ROW_NETS[name]
    x, _ = _row_case(name)
    n_out = layers[-1][0].shape[1]
    load_ok(env, 0, layers, hidden, out)
    r = 70001
    perm = np.random.default_rng(3).permutation(x.shape[0])
    at = int(np.nonzero(perm == r)[0][0])
    for f in (tc, exact):
        alone = f(env, 0, x[r:r + 1], n_out)[0]
        batch = f(env, 0, x, n_out)
        again = f(env, 0, x, n_out)
        permuted = f(env, 0, x[perm], n_out)
        assert np.array_equal(batch[r], alone), f.__name__
        assert np.array_equal(permuted[at], alone), f.__name__
        assert np.array_equal(batch, again), f.__name__
        assert np.array_equal(permuted, batch[perm]), f.__name__


# ---------------------------------------------------------------------------------------------- ABI refusals
def test_forward_calls_refuse_buffers_and_counts_that_do_not_fit(env):
    """Refusals of smenv_mlp_forward / smenv_mlp_forward_exact and of their wrappers; the buffers are large enough that
    an unchecked launch would stay in bounds, and the output must stay untouched."""
    load_ok(env, 1, random_net(np.random.default_rng(1), 23, (64,), 7), "swish", "tanh")
    n = 256
    x = torch.rand((n, 23), device="cuda")
    out = torch.full((n, 16), 7.0, device="cuda")
    lib, h = env._lib, env._handle

    def forward(stride):
        return lib.smenv_mlp_forward(h, 1, x.data_ptr(), 23, None, 0, out.data_ptr(), stride, n, None)

    def forward_exact(which, stride, n_out, e=env):
        return e._lib.smenv_mlp_forward_exact(e._handle, which, x.data_ptr(), 23, None, 0, out.data_ptr(), stride, n_out, n,
                                              None)

    assert forward(6) == SM_ERR_ARG                      # the kernel writes 7 outputs per row
    assert forward_exact(1, 16, 8) == SM_ERR_ARG         # more outputs than the network has
    assert forward_exact(1, 6, 7) == SM_ERR_ARG          # row stride below the outputs written
    fresh = make_env(space_backup_config(ball_machine_mode=True), 32, fill_pools=False)
    try:
        assert forward_exact(2, 16, 1, fresh) == SM_ERR_STATE   # nothing loaded in the slot
        assert "not loaded" in fresh._lib.smenv_last_error().decode()
        with pytest.raises(cabi.SmEnvError, match="not loaded"):
            fresh.mlp_shape(2)
    finally:
        fresh.close()
    torch.cuda.synchronize()
    assert bool((out == 7.0).all())
    for wrapper in (env.mlp_forward, env.mlp_forward_exact):
        for n_out in (1, 6, 8, 16):
            with pytest.raises(ValueError, match="7 outputs"):
                wrapper(1, x, None, n_out=n_out)
    assert forward(7) == 0 and forward_exact(1, 7, 3) == 0     # what fits still runs
    torch.cuda.synchronize()
    assert bool((out.view(-1)[n * 7:] == 7.0).all())            # rows of 7 floats, nothing past them


# ---------------------------------------------------------------------------------------------- inside the step
GATE_SCENES = {"space_bm": (lambda: space_backup_config(ball_machine_mode=True), "space"),
               "ball_bm": (lambda: ball_backup_config(ball_machine_mode=True), "ball"),
               "human": (lambda: human_backup_config(), "human"),
               "space_task_bm": (lambda: space_task_config(ball_machine_mode=True), "space")}


@pytest.fixture(scope="module")
def rollouts():
    """65 536 envs of every gate scene with both networks loaded, a few random steps in."""
    envs = {}
    for name, (cfg, _) in GATE_SCENES.items():
        e = make_env(cfg(), FULL, auto_reset=True)
        e.load_networks()
        e.reset()
        for _ in range(3):
            e.step_random()
        envs[name] = e
    torch.cuda.synchronize()
    yield envs
    for e in envs.values():
        e.close()


@pytest.mark.parametrize("name", sorted(GATE_SCENES))
def test_risk_gate_at_full_size(rollouts, name):
    """risk_gate over 65 536 envs (space_task_bm: the risk observation skips the target-point entries, a strided
    three-segment input).  Tensor-core mode: risk and the backup actions of the risky envs against forward_tc.  Exact
    mode: the rows within the band of the threshold carry the float32 risk of a dense smenv_mlp_forward_exact and the
    others the tensor-core risk, bit for bit; the risky rows carry the backup action of a dense exact launch, bit for
    bit (the gate computes it through a row list); all of it against the float64 reference as in
    test_risk_gate_replaces_exactly_the_risky_actions.  Measured on a B200 (1000 W power limit), tensor-core mode, risk / backup actions max
    (mean): space_bm 8.8e-4 (9.8e-7) / 5.8e-4 (7.6e-7); ball_bm 3.7e-4 (7.9e-7) / 5.6e-4 (6.4e-7); human 1.0e-3
    (8.5e-7) / 1.7e-4 (3.7e-7); space_task_bm 4.5e-4 (8.9e-7) / 3.9e-4 (7.4e-7)."""
    env = rollouts[name]
    w = np.load(os.path.join(ASSETS, "networks_{}.npz".format(GATE_SCENES[name][1])))
    risk_l, backup_l = mlp.shipped_layers(w, "risk"), mlp.shipped_layers(w, "backup")
    robs_d = env.risk_observation()
    robs = robs_d.cpu().numpy()
    act = np.random.default_rng(9).uniform(-1, 1, (FULL, 7)).astype(np.float32)
    x = np.concatenate([robs, act], 1)
    r_tc, r64 = mlp.forward_tc(risk_l, x, "selu", "sigmoid")[:, 0], mlp.forward64(risk_l, x, "selu", "sigmoid")[:, 0]
    thr = float(np.float32(np.median(r64)))
    b_tc, b64 = mlp.forward_tc(backup_l, robs, "swish", "tanh")[:, :7], mlp.forward64(backup_l, robs, "swish", "tanh")[:, :7]

    env.set_gate_exact(False)
    env.actions.copy_(torch.from_numpy(act))
    risk, risky = env.risk_gate(thr)
    torch.cuda.synchronize()
    risk_t, risky_t, gated = risk.cpu().numpy().copy(), risky.cpu().numpy().astype(bool), env.actions.cpu().numpy()
    check_tc(risk_t[:, None], r_tc[:, None], name + " gate risk")
    assert np.array_equal(risky_t, risk_t >= np.float32(thr)) and 0 < risky_t.sum() < FULL
    check_tc(gated[risky_t], b_tc[risky_t], name + " gate backup actions")
    assert np.array_equal(gated[~risky_t], act[~risky_t])

    env.set_gate_exact(True)
    env.actions.copy_(torch.from_numpy(act))
    risk, risky = env.risk_gate(thr)
    torch.cuda.synchronize()
    risk_e, risky_e, gated = risk.cpu().numpy(), risky.cpu().numpy().astype(bool), env.actions.cpu().numpy()
    band = np.abs(risk_t - np.float32(thr)) < np.float32(0.01)
    dense = env.mlp_forward_exact(0, robs_d, torch.from_numpy(act).cuda(), n_out=1).cpu().numpy()[:, 0]
    assert band.sum() > 100
    assert np.array_equal(risk_e, np.where(band, dense, risk_t))
    assert np.array_equal(gated[risky_e], env.mlp_forward_exact(1, robs_d, n_out=7).cpu().numpy()[risky_e])
    assert np.array_equal(gated[~risky_e], act[~risky_e])
    near = np.abs(r64 - thr) < 5e-3
    assert np.abs(risk_e - r64)[near].max() < EXACT_TOL
    clear = np.abs(r64 - thr) > 1e-5
    assert np.array_equal(risky_e[clear], (r64 >= thr)[clear])
    assert np.abs(gated[risky_e] - b64[risky_e]).max() < EXACT_TOL


def philox(c0, c1, c2, c3, k0, k1):
    """Philox4x32-10 over arrays (smo_philox of the oracle)."""
    m = np.uint64(0xFFFFFFFF)
    c = [np.asarray(v, np.uint64) & m for v in (c0, c1, c2, c3)]
    k0, k1 = np.uint64(k0), np.uint64(k1)
    for _ in range(10):
        p0, p1 = np.uint64(0xD2511F53) * c[0], np.uint64(0xCD9E8D57) * c[2]
        c = [((p1 >> np.uint64(32)) ^ c[1] ^ k0) & m, p1 & m, ((p0 >> np.uint64(32)) ^ c[3] ^ k1) & m, p0 & m]
        k0, k1 = (k0 + np.uint64(0x9E3779B9)) & m, (k1 + np.uint64(0xBB67AE85)) & m
    return [v.astype(np.uint32) for v in c]


def test_human_policy_actions_at_full_size():
    """The human's actions of one step at 65 536 envs rebuilt from the observation before the step: mean and log-std
    from forward_tc, the Philox normal noise of human_action_kernel (stream (env, step, joint, 0x4057), key = seed),
    Box-Muller in float32, clipped to [-1, 1].  Measured on a B200 (1000 W power limit): max |difference| 6.8e-4, max |difference| / (1 + |eps|)
    4.2e-4 against the bound 2e-3."""
    env = make_env(human_backup_config(), FULL, auto_reset=True)
    try:
        env.reset()
        steps = 3
        for _ in range(steps):                # the first step of the env uses step counter 0
            env.step_random()
        hobs = env.hobs.cpu().numpy().copy()
        env.step_random()
        torch.cuda.synchronize()
        ha = env.hactions.cpu().numpy()
        w = np.load(os.path.join(ASSETS, "networks_human.npz"))
        layers = mlp.shipped_layers(w, "human")
        o = mlp.forward_tc(layers, hobs[:, :layers[0][0].shape[0]], "swish", "tanh")
        h = env.scene.struct.human
        mean, log_std = o[:, :8], h.log_std_lo + 0.5 * (o[:, 8:] + 1) * (h.log_std_hi - h.log_std_lo)
        e, j = np.meshgrid(np.arange(FULL), np.arange(8), indexing="ij")
        seed = env._seed
        r = philox(e, steps, j, 0x4057, seed & 0xFFFFFFFF, seed >> 32)
        for k in (0, 1, 5, 7, FULL - 1):
            assert [int(v[k, 3]) for v in r] == oracle.philox(k, steps, 3, 0x4057, seed & 0xFFFFFFFF, seed >> 32)
        u01 = lambda v: (v >> np.uint32(8)).astype(np.float32) * np.float32(1.0 / 16777216.0)   # noqa: E731
        u1, u2 = np.maximum(u01(r[0]), np.float32(5.9604645e-8)), u01(r[1])
        eps = np.sqrt(np.float32(-2) * np.log(u1)) * np.cos(np.float32(np.pi) * (np.float32(2) * u2))
        want = np.clip(mean + np.exp(log_std) * eps, -1, 1)
        d = np.abs(ha - want)
        print("human policy actions: max {:.2e}, max / (1 + |eps|) {:.2e}".format(d.max(), (d / (1 + np.abs(eps))).max()))
        assert (d <= 2e-3 * (1 + np.abs(eps))).all()
        assert (np.abs(ha) < 1).mean() > 0.5          # most actions are not clipped
    finally:
        env.close()
