"""Batched, GPU-resident mirror of the reference env API.

``SafeMotionsVecEnv(num_envs, device, **env_config)`` keeps the surface RLlib and the reference's scripts use on
``SafeMotionsEnvCollisionAvoidance`` (safe_motions_env.py:38-45; SURVEY.md section 8b):

    reset() -> obs                         observations.py:144-187, safe_motions_base.py:913-1022
    step(action) -> obs, reward, done, info   safe_motions_base.py:1043-1227
    observation_space / action_space       Box(-1, 1, (n,), float32)  actions.py:50-51, observations.py:116-117
    set_seed, close, TERMINATION_* constants, termination_reason, episode_counter, trajectory_time_step, pid

for N independent environments at once.  With ``num_envs == 1`` and ``squeeze=True`` the scalar gym API is reproduced
(NumPy in / NumPy out, python float reward, bool done, info dict).  Otherwise observations, rewards and dones are
torch tensors that view the pre-allocated device buffers of the env (valid until the next ``step``).

All numerics run in libsmenv.so (hand-written sm_100a CUDA, include/smenv.h).  PyTorch only provides device memory
and streams.  There is no CPU path: constructing the env without a CUDA device raises.
"""
import ctypes as C
import os

import numpy as np
import torch

from . import abi, cabi
from .config import EnvConfig
from .scene import Scene


class Box:
    """Minimal stand-in for gym.spaces.Box (gym is not a dependency of this package)."""

    def __init__(self, low, high, shape, dtype=np.float32):
        self.low = np.full(shape, low, dtype=dtype)
        self.high = np.full(shape, high, dtype=dtype)
        self.shape = tuple(shape)
        self.dtype = np.dtype(dtype)

    def sample(self):
        return np.random.uniform(self.low, self.high).astype(self.dtype)

    def contains(self, x):
        x = np.asarray(x)
        return x.shape == self.shape and bool(np.all(x >= self.low) and np.all(x <= self.high))

    def __repr__(self):
        return "Box({}, {}, {}, {})".format(self.low.min(), self.high.max(), self.shape, self.dtype)


class SafeMotionsVecEnv:
    # safe_motions_base.py:64-70
    TERMINATION_UNSET = abi.TERMINATION_UNSET
    TERMINATION_SUCCESS = abi.TERMINATION_SUCCESS
    TERMINATION_JOINT_LIMITS = abi.TERMINATION_JOINT_LIMITS
    TERMINATION_TRAJECTORY_LENGTH = abi.TERMINATION_TRAJECTORY_LENGTH
    TERMINATION_SELF_COLLISION = abi.TERMINATION_SELF_COLLISION
    TERMINATION_COLLISION_WITH_STATIC_OBSTACLE = abi.TERMINATION_COLLISION_WITH_STATIC_OBSTACLE
    TERMINATION_COLLISION_WITH_MOVING_OBSTACLE = abi.TERMINATION_COLLISION_WITH_MOVING_OBSTACLE

    def __init__(self, num_envs=1, device=None, seed=None, auto_reset=True, squeeze=False, fill_pools=True,
                 config=None, **env_config):
        if not torch.cuda.is_available():
            raise cabi.SmEnvError("SafeMotionsVecEnv needs a CUDA device (sm_100a); there is no CPU fallback")
        self._lib = cabi.load()
        self.config = config if isinstance(config, EnvConfig) else EnvConfig(seed=seed, **env_config)
        if device is None:
            device = "cuda:{}".format(int(os.environ.get("LOCAL_RANK", 0)))
        self.device = torch.device(device)
        self.num_envs = int(num_envs)
        self.auto_reset = bool(auto_reset)
        self._squeeze = bool(squeeze) and self.num_envs == 1
        self.scene = Scene(self.config)
        self._seed = int(seed if seed is not None else (self.config.seed if self.config.seed is not None else 0))
        self._handle = C.c_void_p()
        dev_index = self.device.index if self.device.index is not None else torch.cuda.current_device()
        torch.cuda.set_device(dev_index)
        cabi.check(self._lib.smenv_create(self.scene.pointer(), self.num_envs, dev_index, self._seed,
                                          C.byref(self._handle)), "smenv_create")
        n, nj, d = self.num_envs, self.scene.n_joints, self.scene.obs_size
        dev = self.device
        # device-resident env state (SoA of per-env records, see include/smenv.h)
        self.kin = torch.zeros((n, abi.SM_KIN_STRIDE), dtype=torch.float64, device=dev)
        self.obst = torch.zeros((n, abi.SM_OBST_STRIDE), dtype=torch.float64, device=dev)
        self.episode = torch.zeros((n, 4), dtype=torch.int32, device=dev)
        self.ep_return = torch.zeros(n, dtype=torch.float64, device=dev)
        self.actions = torch.zeros((n, nj), dtype=torch.float32, device=dev)
        self.obs = torch.zeros((n, d), dtype=torch.float32, device=dev)
        self.reward = torch.zeros(n, dtype=torch.float32, device=dev)
        self.done = torch.zeros(n, dtype=torch.uint8, device=dev)
        self.term_reason = torch.full((n,), -1, dtype=torch.int32, device=dev)
        self.info = torch.zeros((n, abi.SM_INFO_STRIDE), dtype=torch.float32, device=dev)
        self.stats = torch.zeros(32, dtype=torch.float64, device=dev)
        # target-point records of the reaching task (use_target_points), else absent
        self.target = torch.zeros((n, abi.SM_TP_STRIDE), dtype=torch.float64, device=dev) \
            if self.scene.struct.use_target_points else None
        # Human scene: state of the nested env that moves the human's arms (ctlp.py:4647-4959)
        self.has_human = bool(self.scene.struct.human.enabled)
        self.hkin = self.hstate = self.hbrake = self.hobs = self.hactions = None
        if self.has_human:
            self.hkin = torch.zeros((n, abi.SM_KIN_STRIDE), dtype=torch.float64, device=dev)
            self.hstate = torch.zeros((n, abi.SM_HSTATE_STRIDE), dtype=torch.float64, device=dev)
            self.hbrake = torch.zeros((n, abi.SM_HBRAKE_STEPS * abi.SM_HUMAN_JOINTS), dtype=torch.float64, device=dev)
            self.hobs = torch.zeros((n, abi.SM_HOBS_STRIDE), dtype=torch.float32, device=dev)
            self.hactions = torch.zeros((n, abi.SM_HUMAN_JOINTS), dtype=torch.float32, device=dev)
        # per-episode aggregates of the step info (include/smenv.h SM_EP_*): running record and last finished episode
        self.epacc = torch.zeros((n, abi.SM_EP_STRIDE), dtype=torch.float32, device=dev)
        self.epinfo = torch.zeros((n, abi.SM_EP_STRIDE), dtype=torch.float32, device=dev)
        opt = lambda t: t.data_ptr() if t is not None else None
        self._buf = abi.SmBuffers(
            kin=self.kin.data_ptr(), obst=self.obst.data_ptr(), episode=self.episode.data_ptr(),
            ep_return=self.ep_return.data_ptr(), actions=self.actions.data_ptr(), obs=self.obs.data_ptr(),
            reward=self.reward.data_ptr(), done=self.done.data_ptr(), term_reason=self.term_reason.data_ptr(),
            info=self.info.data_ptr(), stats=self.stats.data_ptr(), target=opt(self.target),
            hkin=opt(self.hkin), hstate=opt(self.hstate), hbrake=opt(self.hbrake), hobs=opt(self.hobs),
            epacc=self.epacc.data_ptr(), epinfo=self.epinfo.data_ptr(), hactions=opt(self.hactions))
        # pinned host staging for the host-buffer API (step_host)
        self._h_actions = torch.zeros((n, nj), dtype=torch.float32).pin_memory()
        self.host_actions = self._h_actions.numpy()   # pinned input buffer of step_host
        self._h_obs = torch.zeros((n, d), dtype=torch.float32).pin_memory()
        self._h_reward = torch.zeros(n, dtype=torch.float32).pin_memory()
        self._h_done = torch.zeros(n, dtype=torch.uint8).pin_memory()
        self.observation_space = Box(-1.0, 1.0, (d,), np.float32)
        self.action_space = Box(-1.0, 1.0, (nj,), np.float32)
        self.episode_counter = 0
        self.pid = os.getpid()
        self._pools_filled = False
        self._networks = False
        self._gate_threshold = None
        self._auto_reset_done = None   # envs the last step re-initialised on the device (see reset_at)
        if self.has_human:
            self.load_human_policy()
        if fill_pools:
            self.fill_pools(self._seed)
        # risk gate as the reference wires it (safe_motions_base.py:527-579, actions.py:303-340): risk_config_dir names
        # the risk network (its backup policy comes with it), risk_threshold switches the gate on inside step()
        if self.config.risk_config_dir is not None:
            self.load_networks(self._resolve_risk_config_dir(self.config.risk_config_dir))
            if self.config.risk_state_config == 3:
                self.set_risk_next_state(True)
            elif self.config.risk_state_config == 4:
                self.set_risk_lookahead(self.config.risk_state_backup_trajectory_steps or 20)
            self.set_risk_gate(self.config.risk_threshold)
            if self.config.risk_check_initial_backup_trajectory and not fill_pools:
                raise ValueError("risk_check_initial_backup_trajectory needs the start pools (fill_pools=True)")

    # ------------------------------------------------------------------ reference helper surface
    @property
    def trajectory_time_step(self):
        return self.config.trajectory_time_step

    @property
    def use_real_robot(self):
        return False

    @property
    def max_resampling_attempts(self):
        return 0

    @property
    def termination_reason(self):
        r = self.term_reason
        return int(r[0].item()) if self._squeeze else r

    @property
    def observation_size(self):
        return self.scene.obs_size

    def set_seed(self, seed=None):
        """safe_motions_base.py:1704-1710: re-seeds every sampling stream: the library's Philox key (pool picks of
        resets / balls / target points, random actions), the per-env draw counters and the pools, so that the env
        continues exactly like one constructed with this seed."""
        if seed is not None:
            self._seed = int(seed)
            cabi.check(self._lib.smenv_set_seed(self._handle, self._seed), "smenv_set_seed")
            self.episode.zero_()
            if self.target is not None:
                self.target[:, abi.TP_DRAWS] = 0.0
            self.fill_pools(self._seed)
        return [seed]

    def _resolve_risk_config_dir(self, path):
        """risk_config_dir of the reference (a Keras SavedModel directory under trained_networks/risk_networks/
        state_action/<scene>, README.md:223-235) -> the packaged export of that scene's networks, or an .npz path."""
        if str(path).endswith(".npz") and os.path.isfile(path):
            return path
        trained = os.path.join(str(path), "risk_network.npz")   # a directory written by safemotionsrisk_b200.risk_train
        if os.path.isfile(trained):
            return trained
        name = os.path.basename(os.path.normpath(str(path)))
        packaged = os.path.join(os.path.dirname(os.path.abspath(__file__)), "assets", "networks_{}.npz".format(name))
        if name in ("space", "ball", "human") and os.path.isfile(packaged):
            return packaged
        raise ValueError("risk_config_dir {!r}: expected .../state_action/<space|ball|human> (the networks exported by "
                         "tools/export_networks.py) or the path of an exported .npz".format(path))

    def set_risk_gate(self, threshold):
        """Switches the risk gate inside step() / step_random() / step_host() on (threshold in [0, 1]) or off (None);
        smenv_set_risk_gate.  The networks must be loaded (load_networks, or risk_config_dir in the env_config)."""
        thr = -1.0 if threshold is None else float(threshold)
        cabi.check(self._lib.smenv_set_risk_gate(self._handle, thr), "smenv_set_risk_gate")
        self._gate_threshold = None if threshold is None else float(threshold)

    def set_risk_lookahead(self, backup_steps):
        """risk_state_config 4 (RISK_CHECK_NEXT_STATE_SIMULATE_NEXT_STEP_AND_BACKUP_TRAJECTORY, safe_motions_base.py:
        1520-1592) inside the step: while the risk gate is on, an env's action is risky exactly when a copy of the env
        that executes it and then follows the backup policy for `backup_steps` steps (no auto reset, the episode clock
        from 0) ends its episode for a reason other than the trajectory length -- the labelling rule of
        risk_ground_truth.  The risk network is not consulted, so the threshold does not change the decision.  0 or None
        switches back to the network gate (smenv_set_risk_lookahead).  Needs the backup policy (load_networks)."""
        cabi.check(self._lib.smenv_set_risk_lookahead(self._handle, int(backup_steps or 0)), "smenv_set_risk_lookahead")

    def set_risk_next_state(self, enable):
        """risk_state_config 3 (RISK_CHECK_NEXT_STATE_SIMULATE_NEXT_STEP) inside the step: while the risk gate is on, a
        copy of every env executes the proposed action for one step (no auto reset, the episode clock as it is, the real
        step's random stream), and the action is risky when the state risk network rates the state it leads to >= the
        threshold, or when that step ends the episode for a reason other than the trajectory length
        (smenv_set_risk_next_state).  Needs a state risk network (input: the risk observation alone; risk_train on
        state_risk data) and the backup policy (load_networks).  False switches back; with the gate on and a state network
        loaded, switch the gate off first."""
        cabi.check(self._lib.smenv_set_risk_next_state(self._handle, int(bool(enable))), "smenv_set_risk_next_state")

    def _initial_backup_steps(self):
        return int(self.config.risk_state_initial_backup_trajectory_steps or
                   self.config.risk_state_backup_trajectory_steps or 20)

    def set_initial_backup_check(self, steps):
        """risk_check_initial_backup_trajectory (observations.py:155-185) as a property of the start pool: every pool
        entry is checked once, when the pool is filled -- the backup policy acts for `steps` steps from the entry (episode
        clock at 0, no auto reset, gate off), and the entry fails if its episode ends in that window for a reason other
        than the trajectory length (initial_backup_trajectory_unsafe's rule) -- and every reset, reset() and the device
        auto reset of step() / step_random() / step_host() alike, draws from the passing entries only.  The current
        pools are checked at once, and every later fill (set_seed) again.  0 or None switches the check off: resets draw
        from the whole pool again (smenv_set_initial_backup_check).  Needs the backup policy (load_networks); raises if no
        entry passes."""
        cabi.check(self._lib.smenv_set_initial_backup_check(self._handle, int(steps or 0), self._stream()),
                   "smenv_set_initial_backup_check")

    def initial_backup_check_counts(self):
        """(checked, passed): the start-pool entries the initial-backup-trajectory check rated for the current pools (0
        while it is off), and the entries resets draw from (the passing ones; the whole pool while the check is off)."""
        checked, passed = C.c_int(), C.c_int()
        cabi.check(self._lib.smenv_initial_backup_check_counts(self._handle, C.byref(checked), C.byref(passed)),
                   "smenv_initial_backup_check_counts")
        return checked.value, passed.value

    def close(self):
        if self._handle:
            self._lib.smenv_destroy(self._handle)
            self._handle = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ------------------------------------------------------------------ plumbing
    def _stream(self):
        return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    def fill_pools(self, seed=0):
        cabi.check(self._lib.smenv_fill_pools(self._handle, int(seed), self._stream()), "smenv_fill_pools")
        self._pools_filled = True

    def human_pools(self):
        """(start states of the nested env [P, 32] = q, v, a, spare; target points [2, T, 4] per arm), host copies."""
        ps, pt = C.c_int(), C.c_int()
        cabi.check(self._lib.smenv_human_pool_sizes(self._handle, C.byref(ps), C.byref(pt)), "smenv_human_pool_sizes")
        start, target = np.zeros((ps.value, 32)), np.zeros((2, pt.value, 4))
        cabi.check(self._lib.smenv_copy_human_pools(self._handle, start.ctypes.data, target.ctypes.data),
                   "smenv_copy_human_pools")
        return start, target

    def set_human_state(self, hq, hv, ha, first_target, active_arm, mask=None):
        """Injects the start state of the nested env (parity protocol): joint state [N, 8], the first target point
        [N, 3] and the arm [N] it belongs to; call after set_state."""
        def prep(x, cols, dtype=torch.float64):
            t = torch.as_tensor(np.asarray(x) if not torch.is_tensor(x) else x, dtype=dtype)
            return t.reshape(self.num_envs, cols).to(self.device).contiguous() if cols else \
                t.reshape(self.num_envs).to(self.device).contiguous()
        tq, tv, ta, tt = prep(hq, 8), prep(hv, 8), prep(ha, 8), prep(first_target, 3)
        tarm = prep(active_arm, 0, torch.int32)
        tm = None if mask is None else torch.as_tensor(mask, dtype=torch.uint8, device=self.device).contiguous()
        cabi.check(self._lib.smenv_set_human_state(self._handle, C.byref(self._buf), tq.data_ptr(), tv.data_ptr(),
                                                   ta.data_ptr(), tt.data_ptr(), tarm.data_ptr(),
                                                   C.c_void_p(tm.data_ptr()) if tm is not None else None,
                                                   self._stream()), "smenv_set_human_state")
        return self.obs

    def set_human_actions_external(self, external=True):
        """With external=True the step reads the human's actions from ``self.hactions`` instead of evaluating the
        human's policy (parity tests: the reference samples them from a stochastic policy, ctlp.py:4701, :4827)."""
        cabi.check(self._lib.smenv_set_human_actions_external(self._handle, int(bool(external))),
                   "smenv_set_human_actions_external")

    def load_human_policy(self, source=None):
        """The policy that moves the human's arms (trained_networks/human_network, exported by
        tools/export_networks.py): 38 -> 256 -> 128 -> 16 (means and log-std outputs), swish / tanh."""
        if source is None:
            source = os.path.join(os.path.dirname(os.path.abspath(__file__)), "assets", "networks_human.npz")
        w = np.load(source)
        layers = [(w["human/{}/kernel".format(k)], w["human/{}/bias".format(k)]) for k in ("fc_1", "fc_2", "fc_out")]
        if layers[0][0].shape[0] != self.scene.struct.human.obs_size or layers[-1][0].shape[1] != 16:
            raise ValueError("unexpected shape of the human policy")
        dims = np.array([layers[0][0].shape[0]] + [k.shape[1] for k, _ in layers], dtype=np.int32)
        flat = np.concatenate([np.concatenate([k.astype(np.float32).ravel(), b.astype(np.float32).ravel()])
                               for k, b in layers])
        cabi.check(self._lib.smenv_mlp_load(self._handle, abi.SM_NET_HUMAN, len(layers) - 1, dims.ctypes.data, 1, 1,
                                            flat.ctypes.data), "smenv_mlp_load")

    def pools(self):
        """(start_pool [P, 48], ball_pool [B, 12] or None) copied to the host, for inspection and tests."""
        ps, pb = C.c_int(), C.c_int()
        cabi.check(self._lib.smenv_pool_sizes(self._handle, C.byref(ps), C.byref(pb)), "smenv_pool_sizes")
        start = np.zeros((ps.value, 48))
        ball = np.zeros((pb.value, 12)) if pb.value else None
        cabi.check(self._lib.smenv_copy_pools(self._handle, start.ctypes.data,
                                              ball.ctypes.data if ball is not None else None), "smenv_copy_pools")
        return start, ball

    # ------------------------------------------------------------------ reset / step
    def reset(self, mask=None):
        """Resets all (or the masked) envs from the device-resident start pool; returns the first observations."""
        m = None
        if mask is not None:
            m = torch.as_tensor(mask, dtype=torch.uint8, device=self.device).contiguous()
        cabi.check(self._lib.smenv_reset(self._handle, C.byref(self._buf), C.c_void_p(m.data_ptr()) if m is not None
                                         else None, self._stream()), "smenv_reset")
        self.episode_counter += self.num_envs if m is None else int(m.sum().item())
        if self._squeeze:
            return self.obs[0].cpu().numpy()
        return self.obs

    def initial_backup_trajectory_unsafe(self, steps=None):
        """risk_check_initial_backup_trajectory (observations.py:155-185): from a copy of the current state the backup
        policy acts for `steps` steps (default: the episode length of the backup policy's training env, 20); an env is
        unsafe if its episode ends in that window for a reason other than the trajectory length.  The state is
        restored.  Returns a bool tensor [N]."""
        steps = int(steps or self._initial_backup_steps())
        snap = self.snapshot()
        auto, gate = self.auto_reset, self._gate_threshold
        self.auto_reset = False
        self.set_risk_gate(None)
        try:
            self.episode[:, 0] = 0        # switch_to_backup_client: _episode_length = 0 (safe_motions_base.py:1818-1822)
            unsafe = torch.zeros(self.num_envs, dtype=torch.bool, device=self.device)
            for _ in range(steps):
                self._step_device(self.backup_policy_actions())
                unsafe |= self.done.bool() & (self.term_reason != self.TERMINATION_TRAJECTORY_LENGTH)
        finally:
            self.restore(snap)
            self.auto_reset = auto
            self.set_risk_gate(gate)
        return unsafe

    def set_state(self, q, v, a, obst=None, mask=None, first_target=None):
        """Injects start states (parity protocol, SURVEY 8c): q, v, a [N, n_joints] float64, obst [N, 16] or None;
        first_target [N, 3]: the first target point of every env (reaching task), else drawn from the pool."""
        def prep(x, cols):
            if x is None:
                return None
            t = torch.as_tensor(np.asarray(x) if not torch.is_tensor(x) else x, dtype=torch.float64)
            return t.reshape(self.num_envs, cols).to(self.device).contiguous()
        nj = self.scene.n_joints
        tq, tv, ta, tob = prep(q, nj), prep(v, nj), prep(a, nj), prep(obst, abi.SM_OBST_STRIDE)
        tm = None if mask is None else torch.as_tensor(mask, dtype=torch.uint8, device=self.device).contiguous()
        ptr = lambda t: C.c_void_p(t.data_ptr()) if t is not None else None
        cabi.check(self._lib.smenv_set_state(self._handle, C.byref(self._buf), ptr(tq), ptr(tv), ptr(ta), ptr(tob),
                                             ptr(tm), self._stream()), "smenv_set_state")
        if first_target is not None:
            ft = prep(first_target, 3)
            cabi.check(self._lib.smenv_set_targets(self._handle, C.byref(self._buf), ptr(ft), ptr(tm), self._stream()),
                       "smenv_set_targets")
        self.done.zero_()
        return self.obs

    def _step_device(self, actions):
        if torch.is_tensor(actions) and actions.device == self.device:
            self.actions.copy_(actions.reshape(self.num_envs, -1), non_blocking=True)
        else:
            arr = np.asarray(actions, dtype=np.float32).reshape(self.num_envs, -1)
            self.actions.copy_(torch.from_numpy(arr), non_blocking=False)
        cabi.check(self._lib.smenv_step(self._handle, C.byref(self._buf), int(self.auto_reset), self._stream()),
                   "smenv_step")

    def _after_step(self):
        # finished envs were re-initialised inside the step (with risk_check_initial_backup_trajectory from the checked
        # start pool, set_initial_backup_check)
        self._auto_reset_done = self.done if self.auto_reset else None

    def step(self, actions):
        """One env step for all envs.  actions: [N, n_joints] in [-1, 1] (torch on the env's device, or array-like).
        With ``random_agent`` in the env_config the actions are ignored and drawn on the device
        (safe_motions_base.py:1047-1048); with the risk gate on, risky actions are replaced (actions.py:303-340)."""
        if self.config.random_agent:
            return self.step_random()
        self._step_device(actions)
        self._after_step()
        return self._outputs()

    def step_random(self):
        """Step with device-generated U(-1, 1) actions (``random_agent``, safe_motions_base.py:1047-1048)."""
        cabi.check(self._lib.smenv_step_random(self._handle, C.byref(self._buf), int(self.auto_reset), self._stream()),
                   "smenv_step_random")
        self._after_step()
        return self._outputs()

    def set_step_ranges(self, ranges):
        """Env ranges the device step runs side by side (smenv_set_step_ranges); results do not depend on it."""
        cabi.check(self._lib.smenv_set_step_ranges(self._handle, int(ranges)), "smenv_set_step_ranges")

    def step_host(self, actions_np, gate_threshold=None, chunks=2):
        """Host-buffer API: NumPy actions in, NumPy (obs, reward, done) out through pinned staging buffers.
        `host_actions` is the pinned input buffer itself: a sampler that writes its actions there (and passes it, or
        None) saves the host-side copy.  chunks: env ranges whose copies and kernels overlap (smenv_step_host); the
        results do not depend on it.  gate_threshold: run this step with the risk gate at that threshold (default: the
        env's own gate setting)."""
        if actions_np is not None and actions_np is not self.host_actions:
            self.host_actions[...] = np.asarray(actions_np, dtype=np.float32).reshape(self.num_envs, -1)
        prev = self._gate_threshold
        if gate_threshold is not None and gate_threshold != prev:
            self.set_risk_gate(gate_threshold)
        try:   # the gate runs inside the env ranges of the host step (same CUDA graph as the ungated step)
            cabi.check(self._lib.smenv_step_host(self._handle, C.byref(self._buf), self._h_actions.data_ptr(),
                                                 self._h_obs.data_ptr(), self._h_reward.data_ptr(),
                                                 self._h_done.data_ptr(), int(self.auto_reset), int(chunks),
                                                 self._stream()), "smenv_step_host")
        finally:
            if gate_threshold is not None and gate_threshold != prev:
                self.set_risk_gate(prev)
        self._auto_reset_done = self.done if self.auto_reset else None
        return self._h_obs.numpy(), self._h_reward.numpy(), self._h_done.numpy()

    def _outputs(self):
        if self._squeeze:
            done = bool(self.done[0].item())
            return self.obs[0].cpu().numpy(), float(self.reward[0].item()), done, self.infos()[0]
        return self.obs, self.reward, self.done, self.info

    # ------------------------------------------------------------------ info dicts (materialised on demand)
    def _step_info(self, row):
        """The step's info of one env as the reference nests it ('average' / 'max' / 'min' hold the step's values,
        safe_motions_base.py:1350-1365, rewards.py:490-498, actions.py:339-340)."""
        step = dict(collision_rate_self=float(row[abi.INFO["coll_self"]]),
                    collision_rate_static_obstacles=float(row[abi.INFO["coll_static"]]),
                    collision_rate_moving_obstacles=float(row[abi.INFO["coll_moving"]]),
                    action_punishment=float(row[abi.INFO["action_punishment"]]),
                    self_collision_reward=float(row[abi.INFO["r_self"]]),
                    static_obstacles_collision_reward=float(row[abi.INFO["r_static"]]),
                    moving_obstacles_collision_reward=float(row[abi.INFO["r_moving"]]))
        if self.scene.struct.use_target_points:
            step["target_point_reward"] = float(row[abi.INFO["tp_reward"]])
        if self._gate_threshold is not None:
            step["risky_action_rate"] = float(row[abi.INFO["risky_action"]])
        mx = dict(step, joint_jerk_violation=float(row[abi.INFO["max_jerk_rel"]] > 1.002))
        return {"average": step, "max": mx, "min": dict(step)}

    def _episode_info(self, rec, row, reason):
        """End-of-episode keys (safe_motions_base.py:1367-1396, ctlp.py:1141-1309) plus, under 'episode', what
        train.py:59-117 derives from the per-step info dicts of the reference: <key>_average / _max / _min over the
        episode, aggregated on the device (SmBuffers.epinfo)."""
        n = max(1.0, float(rec[abi.EPC["length"]]))
        agg = {}
        for k, name in enumerate(abi.EP_SCALARS):
            if name == "target_point_reward" and not self.scene.struct.use_target_points:
                continue
            if name == "risky_action_rate" and self._gate_threshold is None:
                continue
            if name.endswith("_violation"):
                agg[name + "_max"] = float(rec[16 + k])
                continue
            agg[name + "_average"] = float(rec[k]) / n
            if not name.startswith("joint_vel_norm") and name != "observation_clipping_rate":
                agg[name + "_max"] = float(rec[16 + k])
                agg[name + "_min"] = float(rec[32 + k])
        d = {"episode": agg,
             "episode_length": int(rec[abi.EPC["length"]]),
             "trajectory_length": self.scene.struct.episode_steps + 1,
             "termination_reason": int(reason),
             "trajectory_successful": 0.0 if int(reason) == self.TERMINATION_JOINT_LIMITS else 1.0,
             "episode_return": float(rec[abi.EPC["ret"]]),
             # the braking-trajectory method is off for the robot: the reference logs 1.0 per step for both lists
             # (SURVEY Appendix A, Q4)
             "obstacles_time_influenced_by_braking_trajectory": 2.0,
             "obstacles_time_influenced_by_braking_trajectory_collision": 1.0,
             "obstacles_time_influenced_by_braking_trajectory_torque": 1.0,
             "obstacles_num_target_points_reached": float(rec[abi.EPC["targets_reached"]])}
        if self._gate_threshold is not None:
            first = float(rec[abi.EPC["first_risky_step"]])
            d["risk_network_first_risky_action_step"] = first if first >= 0 else float("nan")
        if self.config.use_moving_objects:
            hit, missed = float(rec[abi.EPC["balls_hit_robot"]]), float(rec[abi.EPC["balls_missed"]])
            d["moving_object_hit_robot_total"] = hit
            d["moving_object_missed_robot_total"] = missed     # includes balls that ended on the table or the floor
            if hit + missed > 0:
                d["moving_object_hit_robot_fraction"] = hit / (hit + missed)
                d["moving_object_missed_robot_fraction"] = missed / (hit + missed)
        if self.has_human:
            d["human_braking_trajectory_steps"] = float(rec[abi.EPC["human_braked"]])
        return d

    def infos(self, only_done=False):
        """Per-env info dicts with the reference's key names.  only_done: dicts only for the envs whose episode ended in
        the last step (what RLlib's callbacks need), the others get {}: host work proportional to the number of finished
        episodes, not to the number of envs."""
        done = self.done.cpu().numpy()
        idx = np.nonzero(done)[0]
        out = [{} for _ in range(self.num_envs)]
        if only_done and idx.size == 0:
            return out
        if only_done:
            sel = torch.as_tensor(idx, device=self.device)
            info = self.info.index_select(0, sel).cpu().numpy()
            rec = self.epinfo.index_select(0, sel).cpu().numpy()
            reason = self.term_reason.index_select(0, sel).cpu().numpy()
            for i, e in enumerate(idx):
                d = self._step_info(info[i])
                d.update(self._episode_info(rec[i], info[i], reason[i]))
                out[e] = d
            return out
        info = self.info.cpu().numpy()
        rec = self.epinfo.cpu().numpy()
        reason = self.term_reason.cpu().numpy()
        for e in range(self.num_envs):
            d = self._step_info(info[e])
            if done[e]:
                d.update(self._episode_info(rec[e], info[e], reason[e]))
            out[e] = d
        return out

    def episode_statistics(self, reset=False):
        """Accumulated episode statistics of this shard (the quantities train.py:59-117 turns into custom_metrics):
        [episodes, sum return, sum length, count by termination reason ...]; all-reduced over ranks by the caller."""
        s = self.stats.clone()
        if reset:
            self.stats.zero_()
        return s

    # ------------------------------------------------------------------ RLlib VectorEnv duck-typing
    def vector_reset(self):
        return list(self.reset().cpu().numpy())

    def reset_at(self, index):
        """RLlib calls this for every env that reported done.  An env that the last step already re-initialised on the
        device (auto_reset) is not reset a second time: its first observation is returned as it is."""
        if self._auto_reset_done is not None and bool(self._auto_reset_done[index].item()):
            return self.obs[index].cpu().numpy()
        mask = np.zeros(self.num_envs, dtype=np.uint8)
        mask[index] = 1
        self.reset(mask)
        return self.obs[index].cpu().numpy()

    def vector_step(self, actions):
        obs, rew, done, _ = self.step(np.asarray(actions, dtype=np.float32))
        if self._squeeze:
            return [obs], [rew], [done], [self.infos()[0]]
        return list(obs.cpu().numpy()), list(rew.cpu().numpy()), [bool(x) for x in done.cpu().numpy()], \
            self.infos(only_done=True)

    def get_unwrapped(self):
        return [self]

    # ------------------------------------------------------------------ parity / measurement hooks
    def safe_range(self, kin=None):
        kin = self.kin if kin is None else torch.as_tensor(kin, dtype=torch.float64, device=self.device).contiguous()
        n = kin.shape[0]
        lo = torch.zeros((n, abi.SM_MAX_JOINTS), dtype=torch.float64, device=self.device)
        hi = torch.zeros_like(lo)
        code = torch.zeros((n, abi.SM_MAX_JOINTS), dtype=torch.int32, device=self.device)
        cabi.check(self._lib.smenv_safe_range(self._handle, kin.data_ptr(), lo.data_ptr(), hi.data_ptr(),
                                              code.data_ptr(), n, self._stream()), "smenv_safe_range")
        nj = self.scene.n_joints
        return lo[:, :nj], hi[:, :nj], code[:, :nj]

    def distances(self, kin=None, obst=None, hkin=None):
        kin = self.kin if kin is None else torch.as_tensor(kin, dtype=torch.float64, device=self.device).contiguous()
        obst = self.obst if obst is None else torch.as_tensor(obst, dtype=torch.float64,
                                                              device=self.device).contiguous()
        n = kin.shape[0]
        out = [torch.zeros(n, dtype=torch.float32, device=self.device) for _ in range(3)]
        hp = None
        if self.scene.struct.human.enabled:
            hkin = self.hkin if hkin is None else torch.as_tensor(hkin, dtype=torch.float64,
                                                                   device=self.device).contiguous()
            hp = C.c_void_p(hkin.data_ptr())
        cabi.check(self._lib.smenv_distances(self._handle, kin.data_ptr(), obst.data_ptr(), hp, out[0].data_ptr(),
                                             out[1].data_ptr(), out[2].data_ptr(), n, self._stream()),
                   "smenv_distances")
        return out

    def enable_counters(self, enable=True):
        cabi.check(self._lib.smenv_enable_counters(self._handle, int(enable)), "smenv_enable_counters")

    def counters(self, reset=False):
        c = abi.SmCounters()
        torch.cuda.synchronize(self.device)
        cabi.check(self._lib.smenv_counters(self._handle, C.byref(c), int(reset)), "smenv_counters")
        out = {k: int(getattr(c, k)) for k, _ in abi.SmCounters._fields_ if k != "aux"}
        out["gjk_iteration_histogram"] = [int(x) for x in c.aux]   # pairs with <= 4, 8, 12, 16, 24, more iterations
        return out

    # ------------------------------------------------------------------ networks in the step loop (risk gate)
    def load_networks(self, source=None):
        """Loads the risk network and the backup policy (weights exported from the reference's checkpoints by
        tools/export_networks.py).  source: path of an .npz, or None for the packaged weights of the env's scene."""
        if source is None:
            scene = "human" if self.has_human else "ball" if self.config.use_moving_objects else "space"
            source = os.path.join(os.path.dirname(os.path.abspath(__file__)), "assets",
                                  "networks_{}.npz".format(scene))
        w = np.load(source)
        nj = self.scene.n_joints
        n_risk = len([k for k in w.files if k.startswith("risk/") and k.endswith("/kernel")])
        if not 2 <= n_risk <= 4:
            raise ValueError("{}: the risk network needs 1 to 3 hidden layers and an output layer".format(source))
        risk = [(w["risk/dense_{}/kernel".format(i)], w["risk/dense_{}/bias".format(i)]) for i in range(n_risk)]
        if "backup/fc_1/kernel" not in w.files:   # a risk network trained here (risk_train.py): the backup policy is the
            packaged = os.path.join(os.path.dirname(os.path.abspath(__file__)), "assets", "networks_{}.npz".format(   # scene's
                "human" if self.has_human else "ball" if self.config.use_moving_objects else "space"))
            wp = np.load(packaged)
        else:
            wp = w
        pol = [(wp["backup/{}/kernel".format(n)], wp["backup/{}/bias".format(n)]) for n in ("fc_1", "fc_2", "fc_out")]
        pol[-1] = (pol[-1][0][:, :nj], pol[-1][1][:nj])  # deterministic action = the mean head
        risk_obs = self.scene.obs_size - self.scene.obs_target_size   # without the target-point entries
        if risk[0][0].shape[0] not in (risk_obs, risk_obs + nj) or pol[0][0].shape[0] != risk_obs:
            raise ValueError("networks expect a risk observation of size {}, the env produces {}".format(
                pol[0][0].shape[0], risk_obs))
        # the risk network's kind by its input width: the risk observation alone (a state network, risk_train on
        # state_risk data) or followed by the action (a state-action network, the shipped ones)
        kind = "state" if risk[0][0].shape[0] == risk_obs else "state_action"
        if kind == "state" and self.config.risk_state_config not in (3, 4):
            raise ValueError("{}: a state risk network (input: the risk observation, {} values) rates states, not "
                             "actions; the network gate of risk_state_config={} needs a state-action network (input {}); "
                             "risk_state_config=3 rates the simulated next state with it".format(
                                 source, risk_obs, self.config.risk_state_config, risk_obs + nj))
        if kind == "state_action" and self.config.risk_state_config == 3:
            raise NotImplementedError("{}: risk_state_config=3 rates the simulated next state with a state risk network; "
                                      "rating it with a state-action network is not implemented".format(source))
        risk_hidden = 0
        if "risk/hidden_layer_activation" in w.files:   # written by risk_train.export_weights
            act, last = str(w["risk/hidden_layer_activation"]), str(w["risk/last_layer_activation"])
            if act not in ("selu", "swish") or last != "sigmoid":
                raise ValueError("{}: the step loop runs selu or swish hidden layers and a sigmoid output, not {} / {}".format(
                    source, act, last))
            risk_hidden = 0 if act == "selu" else 1
        for which, layers, hidden, out_act in ((0, risk, risk_hidden, 0), (1, pol, 1, 1)):
            dims = np.array([layers[0][0].shape[0]] + [k.shape[1] for k, _ in layers], dtype=np.int32)
            flat = np.concatenate([np.concatenate([k.astype(np.float32).ravel(), b.astype(np.float32).ravel()])
                                   for k, b in layers])
            cabi.check(self._lib.smenv_mlp_load(self._handle, which, len(layers) - 1, dims.ctypes.data, hidden, out_act,
                                                flat.ctypes.data), "smenv_mlp_load")
        self.risk = torch.zeros(self.num_envs, dtype=torch.float32, device=self.device)
        self.risky = torch.zeros(self.num_envs, dtype=torch.uint8, device=self.device)
        self._networks = True
        self._network_source = source
        self.risk_network_kind = kind
        if self.config.risk_check_initial_backup_trajectory:
            self.set_initial_backup_check(self._initial_backup_steps())

    def mlp_shape(self, which):
        """(input width, output count) of the loaded network `which` (smenv_mlp_shape)."""
        n_in, n_out = C.c_int(), C.c_int()
        cabi.check(self._lib.smenv_mlp_shape(self._handle, which, C.byref(n_in), C.byref(n_out)), "smenv_mlp_shape")
        return n_in.value, n_out.value

    def _check_n_out(self, which, n_out):
        have = self.mlp_shape(which)[1]
        if n_out != have:
            raise ValueError("network {} has {} outputs, n_out={} was asked for".format(which, have, n_out))

    def mlp_forward(self, which, in0, in1=None, n_out=1):
        """Parity hook: the loaded network `which` (0 risk, 1 backup policy) on caller-supplied rows; n_out must be the
        network's output count."""
        self._check_n_out(which, n_out)
        in0 = torch.as_tensor(in0, dtype=torch.float32, device=self.device).contiguous()
        n = in0.shape[0]
        out = torch.zeros((n, n_out), dtype=torch.float32, device=self.device)
        p1, w1 = None, 0
        if in1 is not None:
            in1 = torch.as_tensor(in1, dtype=torch.float32, device=self.device).contiguous()
            p1, w1 = C.c_void_p(in1.data_ptr()), in1.shape[1]
        cabi.check(self._lib.smenv_mlp_forward(self._handle, which, in0.data_ptr(), in0.shape[1], p1, w1,
                                               out.data_ptr(), n_out, n, self._stream()), "smenv_mlp_forward")
        return out

    # ------------------------------------------------------------------ the agent: the policy that acts in the env
    def load_agent(self, source=None, log_std_range=(-1.375, 0.0), hidden_activation="swish"):
        """Loads the policy that acts in the env (smenv_mlp_load into SM_NET_AGENT), a Keras fcnet with a DiagGaussian
        head (keras_fcnet_last_layer_activation.py:86-136, :187-202): hidden Dense layers (swish, or selu), then a tanh
        Dense layer of 2 n_joints outputs, the means followed by the log-std pre-activations t, remapped to
        log_std = lo + (t + 1) / 2 (hi - lo) with log_std_range = (lo, hi) (smenv_set_agent_head).  source: an .npz with
        agent/fc_1/kernel, agent/fc_1/bias, ... agent/fc_out/bias, or None for the scene's packaged backup policy with all
        its outputs.  The agent sees the full observation (target-point entries included).  Raises ValueError if the
        input width is not the observation size or the output count is not 2 n_joints."""
        if hidden_activation not in ("swish", "selu"):
            raise ValueError("hidden_activation must be 'swish' or 'selu', not {!r}".format(hidden_activation))
        lo, hi = (float(x) for x in log_std_range)
        if lo > hi:
            raise ValueError("log_std_range ({}, {}): the lower end exceeds the upper".format(lo, hi))
        if source is None:
            scene = "human" if self.has_human else "ball" if self.config.use_moving_objects else "space"
            source = os.path.join(os.path.dirname(os.path.abspath(__file__)), "assets", "networks_{}.npz".format(scene))
            prefix = "backup"
        else:
            prefix = "agent"
        w = np.load(source)
        names, i = [], 1
        while "{}/fc_{}/kernel".format(prefix, i) in w.files:
            names.append("fc_{}".format(i))
            i += 1
        names.append("fc_out")
        if "{}/fc_out/kernel".format(prefix) not in w.files or len(names) < 2:
            raise ValueError("{}: expected {}/fc_1 ... {}/fc_out kernels and biases".format(source, prefix, prefix))
        layers = [(w["{}/{}/kernel".format(prefix, k)], w["{}/{}/bias".format(prefix, k)]) for k in names]
        nj, d = self.scene.n_joints, self.scene.obs_size
        if layers[0][0].shape[0] != d:
            raise ValueError("{}: the agent takes {} inputs, the env's observation has {}".format(
                source, layers[0][0].shape[0], d))
        if layers[-1][0].shape[1] != 2 * nj:
            raise ValueError("{}: the agent has {} outputs, its head needs 2 x {} (means, then log-std)".format(
                source, layers[-1][0].shape[1], nj))
        dims = np.array([layers[0][0].shape[0]] + [k.shape[1] for k, _ in layers], dtype=np.int32)
        flat = np.concatenate([np.concatenate([k.astype(np.float32).ravel(), b.astype(np.float32).ravel()])
                               for k, b in layers])
        cabi.check(self._lib.smenv_mlp_load(self._handle, abi.SM_NET_AGENT, len(layers) - 1, dims.ctypes.data,
                                            0 if hidden_activation == "selu" else 1, 1, flat.ctypes.data),
                   "smenv_mlp_load")
        cabi.check(self._lib.smenv_set_agent_head(self._handle, lo, hi), "smenv_set_agent_head")
        n, dev = self.num_envs, self.device
        self.agent_actions = torch.zeros((n, nj), dtype=torch.float32, device=dev)
        self.agent_logp = torch.zeros(n, dtype=torch.float32, device=dev)
        self.agent_dist_inputs = torch.zeros((n, 2 * nj), dtype=torch.float32, device=dev)

    def step_agent(self, explore=True):
        """One env step whose actions come from the agent (load_agent) on the current observation, on the device
        (smenv_step_agent).  explore=True samples mean + exp(log_std) eps (Philox normal noise), explore=False takes the
        mean; the env executes the sample clipped to [-1, 1] (through the risk gate when it is on), and self.actions holds
        that clipped proposal.  self.agent_actions (the unclipped samples), self.agent_logp (their DiagGaussian
        log-likelihood; 0 with explore=False) and self.agent_dist_inputs (mean, log_std) describe the step's actions and
        stay valid until the next step.  Returns what step() returns."""
        cabi.check(self._lib.smenv_step_agent(self._handle, C.byref(self._buf), int(self.auto_reset), int(bool(explore)),
                                              self.agent_actions.data_ptr(), self.agent_logp.data_ptr(),
                                              self.agent_dist_inputs.data_ptr(), self._stream()), "smenv_step_agent")
        self._after_step()
        return self._outputs()

    def rollout(self, steps, explore=True):
        """`steps` calls of step_agent, recorded on the device without a host synchronise, under RLlib's SampleBatch
        names: obs [T, N, D] (the observation each action was computed from), actions [T, N, n_joints] (unclipped),
        action_logp [T, N], action_dist_inputs [T, N, 2 n_joints], rewards [T, N], dones [T, N] (bool), risky [T, N]
        (bool; only while the risk gate is on), and last_obs [N, D], the observation after the last step.  With auto_reset
        an env that is done starts its next episode in the next row."""
        T, n, nj, d = int(steps), self.num_envs, self.scene.n_joints, self.scene.obs_size
        dev = self.device
        out = dict(obs=torch.empty((T, n, d), dtype=torch.float32, device=dev),
                   actions=torch.empty((T, n, nj), dtype=torch.float32, device=dev),
                   action_logp=torch.empty((T, n), dtype=torch.float32, device=dev),
                   action_dist_inputs=torch.empty((T, n, 2 * nj), dtype=torch.float32, device=dev),
                   rewards=torch.empty((T, n), dtype=torch.float32, device=dev),
                   dones=torch.empty((T, n), dtype=torch.bool, device=dev))
        gate = self._gate_threshold is not None
        if gate:
            out["risky"] = torch.empty((T, n), dtype=torch.bool, device=dev)
        for t in range(T):
            out["obs"][t].copy_(self.obs)
            self.step_agent(explore)
            out["actions"][t].copy_(self.agent_actions)
            out["action_logp"][t].copy_(self.agent_logp)
            out["action_dist_inputs"][t].copy_(self.agent_dist_inputs)
            out["rewards"][t].copy_(self.reward)
            out["dones"][t].copy_(self.done)
            if gate:
                out["risky"][t].copy_(self.info[:, abi.INFO["risky_action"]])
        out["last_obs"] = self.obs.clone()
        return out

    def set_gate_exact(self, exact=True, band=0.0):
        """Exact gate (default on): rows whose tensor-core risk lies within `band` (default 0.01) of the threshold are
        re-rated in float32 and the backup action of the risky rows is computed in float32 (smenv_set_gate_exact)."""
        cabi.check(self._lib.smenv_set_gate_exact(self._handle, int(bool(exact)), float(band)), "smenv_set_gate_exact")

    def mlp_forward_exact(self, which, in0, in1=None, n_out=1):
        """Parity hook: the loaded network `which` in float32 on the CUDA cores (the exact path of the gate); n_out must
        be the network's output count."""
        self._check_n_out(which, n_out)
        in0 = torch.as_tensor(in0, dtype=torch.float32, device=self.device).contiguous()
        n = in0.shape[0]
        out = torch.zeros((n, n_out), dtype=torch.float32, device=self.device)
        p1, w1 = None, 0
        if in1 is not None:
            in1 = torch.as_tensor(in1, dtype=torch.float32, device=self.device).contiguous()
            p1, w1 = C.c_void_p(in1.data_ptr()), in1.shape[1]
        cabi.check(self._lib.smenv_mlp_forward_exact(self._handle, which, in0.data_ptr(), in0.shape[1], p1, w1,
                                                     out.data_ptr(), n_out, n_out, n, self._stream()),
                   "smenv_mlp_forward_exact")
        return out

    def risk_gate(self, threshold=None):
        """Replaces, in self.actions, every action the risk network rates >= threshold by the backup policy's action
        for the current observation (actions.py:303-340).  Returns (risk [N], risky [N])."""
        thr = float(self.config.risk_threshold if threshold is None else threshold)
        cabi.check(self._lib.smenv_risk_gate(self._handle, C.byref(self._buf), thr, self.risk.data_ptr(),
                                             self.risky.data_ptr(), self._stream()), "smenv_risk_gate")
        return self.risk, self.risky

    def step_gated(self, actions=None, threshold=None):
        """One env step with the risk gate at `threshold` (the env's own gate setting is restored afterwards): the
        proposed actions (device-generated random actions if None) stay in self.actions, the executed ones differ where
        info[:, risky_action] is 1."""
        thr = float(self.config.risk_threshold if threshold is None else threshold)
        prev = self._gate_threshold
        self.set_risk_gate(thr)
        try:
            return self.step_random() if actions is None else self.step(actions)
        finally:
            self.set_risk_gate(prev)

    # ------------------------------------------------------------------ backup-client look-ahead (risk ground truth)
    _STATE = ("kin", "obst", "episode", "ep_return", "target", "stats", "obs", "reward", "done", "term_reason", "info",
              "hkin", "hstate", "hbrake", "hobs", "hactions", "epacc", "epinfo")

    def snapshot(self):
        """Copy of the whole env state (the reference clones its Bullet state into a "backup client" with
        saveBullet / restoreState plus attribute copies, safe_motions_base.py:1801-1891; here it is a tensor copy)."""
        return {k: getattr(self, k).clone() for k in self._STATE if getattr(self, k, None) is not None}

    def restore(self, snap):
        for k, v in snap.items():
            getattr(self, k).copy_(v)

    def risk_observation(self):
        """The observation without the target-point entries (observations.py:419-431): what the networks see."""
        nt = self.scene.obs_target_size
        if nt == 0:
            return self.obs
        k = 3 * self.scene.n_joints
        return torch.cat([self.obs[:, :k], self.obs[:, k + nt:]], dim=1).contiguous()

    def backup_policy_actions(self):
        """Deterministic actions of the backup policy for the current observations (explore=False)."""
        return self.mlp_forward(1, self.risk_observation(), None, n_out=self.scene.n_joints)

    def risk_ground_truth(self, actions, backup_steps=20):
        """Ground truth of the state-action risk (RISK_CHECK_NEXT_STATE_SIMULATE_NEXT_STEP_AND_BACKUP_TRAJECTORY,
        safe_motions_base.py:1520-1592): from a copy of the current state, apply `actions`, then let the backup policy
        act for `backup_steps` steps; an env is risky (1.0) if its episode ends in that window for any reason other
        than the trajectory length.  The env state is restored afterwards.  Returns (risk_observation, actions, risk)
        as device tensors -- one row of the reference's risk data set per env (safe_motions_base.py:1413-1461)."""
        state = self.risk_observation().clone()
        act = torch.as_tensor(actions, dtype=torch.float32, device=self.device).reshape(self.num_envs, -1).clone()
        snap = self.snapshot()
        auto = self.auto_reset
        self.auto_reset = False
        gate = self._gate_threshold
        self.set_risk_gate(None)
        try:
            # the look-ahead runs on its own episode clock (switch_to_backup_client: _episode_length = 0 and
            # trajectory_length = backup_steps + 2, safe_motions_base.py:1818-1822): the end of the real episode never
            # cuts the window short, and only a collision ends an env's look-ahead
            self.episode[:, 0] = 0
            risky = torch.zeros(self.num_envs, dtype=torch.bool, device=self.device)
            alive = torch.ones(self.num_envs, dtype=torch.bool, device=self.device)
            a = act
            for i in range(1 + int(backup_steps)):
                self._step_device(a)
                collided = self.done.bool() & (self.term_reason != self.TERMINATION_TRAJECTORY_LENGTH)
                risky |= alive & collided
                alive &= ~collided
                if i < backup_steps:
                    a = self.backup_policy_actions()
        finally:
            self.restore(snap)
            self.auto_reset = auto
            self.set_risk_gate(gate)
        return state, act, risky.float()

    def state_risk_ground_truth(self, backup_steps=20):
        """Ground truth of the state risk (the labels a state risk network learns, risk_state_config 3): from a copy of
        the current state the backup policy acts for `backup_steps` steps with the episode clock at 0 and no auto reset;
        a state is risky (1.0) if its episode ends in that window for any reason other than the trajectory length --
        initial_backup_trajectory_unsafe's rule.  The env state is restored afterwards.  Returns (risk_observation [N, D],
        risk [N]) as device tensors: rows for risk_data.write_risk_csv(directory, state, risk) (state_risk files)."""
        state = self.risk_observation().clone()
        risk = self.initial_backup_trajectory_unsafe(int(backup_steps)).float()
        return state, risk

    KERNELS = ("human_policy", "human_joint_kernels", "human_brake_traj_kernel", "human_brake_plan_kernel",
               "human_brake_gjk", "human_advance_outcome", "joint_kernel", "joint_heavy_kernel", "contact_plan_kernel",
               "distance_plan_kernel", "gjk_kernel", "finish_kernel")

    def kernel_timing(self, enable=True):
        """Measurement mode: every step brackets each of its kernels with CUDA events and synchronises."""
        cabi.check(self._lib.smenv_kernel_timing(self._handle, int(enable)), "smenv_kernel_timing")

    def kernel_times(self, reset=False):
        """{kernel name: mean milliseconds per step} accumulated in measurement mode, and the number of steps."""
        ms = (C.c_double * len(self.KERNELS))()
        steps = C.c_int()
        cabi.check(self._lib.smenv_kernel_times(self._handle, ms, C.byref(steps), int(reset)), "smenv_kernel_times")
        n = max(1, steps.value)
        return {k: ms[i] / n for i, k in enumerate(self.KERNELS)}, steps.value

    def launch_config(self):
        """Launch geometry the library chose for this scene (GJK CTAs / threads / shared memory, planning grid ...)."""
        out = (C.c_int32 * 8)()
        cabi.check(self._lib.smenv_launch_config(self._handle, out), "smenv_launch_config")
        keys = ("gjk_grid", "gjk_threads", "gjk_smem_bytes", "lut_words", "plan_grid", "plan_smem_bytes", "sms", "step_ranges")
        return dict(zip(keys, [int(x) for x in out]))

    def launch_count(self):
        n = C.c_ulonglong()
        cabi.check(self._lib.smenv_launch_count(self._handle, C.byref(n)), "smenv_launch_count")
        return int(n.value)


def make_env(env_config, num_envs=1, **kwargs):
    """``tune.register_env(name, lambda cfg: make_env(cfg))`` style factory (train.py:620, evaluate.py:748)."""
    return SafeMotionsVecEnv(num_envs=num_envs, **kwargs, **dict(env_config))
