"""CemMpc — the reference's CEM-MPC planner interface (simba/policies/cem_mpc.py) on one B200.

`generate_action(state)` (cem_mpc.py:31-33) is one call into libsimba_b200.so: the host state is
copied to the device, the whole CEM loop (cem_mpc.py:35-68) replays as one CUDA graph of the
sample / fused-rollout / score-reduce / select / refit kernels, and the action comes back. No
TensorFlow, no per-op dispatch, no host sync inside the loop (the early `break` of :66-67 is a
device flag).

Extra keyword-only arguments (not in the reference; all default to the reference behaviour):
  precision   'bf16' (tcgen05 tensor-core rollout, fp32 accumulate) or 'fp32' (SIMT parity kernel)
  seed        Philox base seed; call k uses seed + k (the reference uses TF's global stream)
  n_states    plan this many independent states per call (state is then [n_states, O])
  member_map  'split' = tf.split row->member map (reference); 'particle' = floor(p*E/P)
  rank, world_size   population shard of a multi-GPU plan (see simba_b200.distributed)
"""
import ctypes as C

import numpy as np
import torch

from .. import _device, _lib
from .mpc_policy import MpcPolicy


def _broadcast_act(value, a_dim):
    return np.broadcast_to(np.asarray(value, dtype=np.float32), (a_dim,)).copy()


class CemMpc(MpcPolicy):
    _objective = _lib.OBJ_REWARD

    def __init__(self, model, environment, horizon, iterations, smoothing, n_samples, n_elite,
                 particles, stddev_threshold, noise_stddev, *, precision='bf16', seed=0, n_states=1,
                 member_map='split', rank=0, world_size=1, objective=None,
                 posterior_mean_threashold=0.0):
        super().__init__(model, environment, horizon, n_samples, particles)
        self.iterations = iterations
        self.smoothing = smoothing
        self.elite = n_elite
        self.stddev_threshold = stddev_threshold
        self.noise_stddev = noise_stddev
        self.environment = environment
        self.precision = precision
        self.seed = int(seed)
        self.n_states = int(n_states)
        self.member_map = member_map
        self.rank, self.world_size = int(rank), int(world_size)
        if objective is not None:
            self._objective = objective
        self._posterior = float(posterior_mean_threashold)
        self._calls = 0
        self._planner = None
        self._external = None
        self._lib = _lib.load()
        self.iterations_run = None

    # -- planner handle ---------------------------------------------------------------------------
    def _scorer_struct(self):
        scorer = getattr(self.environment, '_scorer', None)
        if scorer is None or not hasattr(scorer, 'scorer_struct'):
            raise _lib.SimbaError(
                -6, "the fused planner needs environment._scorer to be a SafetyGymStateScorer "
                    "parameter set (simba_b200.environment_utils); arbitrary Python reward "
                    "callables cannot run inside the rollout kernel and there is no CPU fallback")
        return scorer.scorer_struct()

    def _config(self):
        lb, ub, mu, sigma = self.sampling_params
        a_dim = self.action_space.shape[0]
        if a_dim > _lib.SIMBA_MAX_ACT:
            raise _lib.SimbaError(-1, "act_dim %d > %d" % (a_dim, _lib.SIMBA_MAX_ACT))
        cfg = _lib.PlannerConfig()
        cfg.horizon, cfg.iterations = int(self.horizon), int(self.iterations)
        cfg.n_samples, cfg.n_elite = int(self.n_samples), int(self.elite)
        cfg.particles, cfg.n_states = int(self.particles), self.n_states
        cfg.smoothing = float(self.smoothing)
        cfg.stddev_threshold = float(self.stddev_threshold)
        cfg.noise_stddev = float(self.noise_stddev)
        cfg.posterior_mean_threshold = self._posterior
        cfg.prior_mu, cfg.prior_sigma = 0.5, 0.27                      # safe_cem_mpc.py:81
        cfg.objective = int(self._objective)
        cfg.sampling_propagation = int(bool(self.model.sampling_propagation))
        cfg.precision = _lib.PRECISIONS[self.precision]
        cfg.member_map = _lib.MEMBER_MAPS[self.member_map]
        cfg.rank, cfg.world_size = self.rank, self.world_size
        for name, value in (('act_low', lb), ('act_high', ub), ('init_mean', mu),
                            ('init_stddev', sigma)):
            arr = _broadcast_act(value, a_dim)
            field = getattr(cfg, name)
            for i in range(a_dim):
                field[i] = float(arr[i])
        cfg.scorer = self._scorer_struct()
        return cfg

    def _ensure_planner(self):
        if self._planner is None:
            _device.require_cuda()
            model_handle = self.model.model._ensure_handle()
            cfg = self._config()
            h = C.c_void_p()
            _lib.check(self._lib.simba_planner_create(model_handle, C.byref(cfg), C.byref(h)))
            try:
                self._configure_planner(h)
            except BaseException:
                self._lib.simba_planner_destroy(h)
                raise
            self._planner = h
            self._cfg = cfg
            if self._external is not None:
                self._apply_external()
        else:
            self.model.model._ensure_handle()        # re-commit if weights / scaler changed
        return self._planner

    def _configure_planner(self, handle):
        """Settings made right after simba_planner_create, before the first plan (none for CEM)."""

    def __del__(self):
        try:
            if self._planner is not None:
                self._lib.simba_planner_destroy(self._planner)
        except Exception:
            pass

    def build(self):
        self._ensure_planner()

    # -- parity hooks -----------------------------------------------------------------------------
    def set_external_draws(self, z_actions=None, eps=None, z_final=None):
        """Feed the planner the normal draws instead of Philox (parity mode): z_actions
        [I, S, N, H, A], eps [I, S, H, P*N, O], z_final [S, A] (S may be omitted when n_states == 1)."""
        def prep(x):
            return None if x is None else _device.to_device(x)[0]
        self._external = (prep(z_actions), prep(eps), prep(z_final))
        if self._planner is not None:
            self._apply_external()

    def _apply_external(self):
        z, e, f = self._external
        _lib.check(self._lib.simba_planner_set_external_draws(
            self._planner, _device.ptr(z), _device.ptr(e), _device.ptr(f)))

    def init_distributed(self, unique_id_bytes):
        """Join the NCCL communicator used for the per-iteration (return, cost) all-gather."""
        buf = (C.c_char * 128).from_buffer_copy(bytes(unique_id_bytes))
        _lib.check(self._lib.simba_planner_init_nccl(self._ensure_planner(), buf))

    def buffer(self, which, dtype=torch.float32):
        """Copy of an internal device buffer as a torch tensor (diagnostics / tests)."""
        p, n = C.c_void_p(), C.c_uint64()
        _lib.check(self._lib.simba_planner_buffer(self._ensure_planner(), which, C.byref(p), C.byref(n)))
        itemsize = torch.empty((), dtype=dtype).element_size()
        out = torch.empty((n.value // itemsize,), dtype=dtype, device='cuda')
        _lib.check(self._lib.simba_planner_copy_buffer(self._planner, which, _device.ptr(out),
                                                       _device.stream_ptr()))
        return out

    # -- the planning call ------------------------------------------------------------------------
    def _next_seed(self, seed):
        if seed is not None:
            return int(seed) & 0xFFFFFFFFFFFFFFFF
        s = (self.seed + self._calls) & 0xFFFFFFFFFFFFFFFF
        self._calls += 1
        return s

    def generate_action(self, state):
        """cem_mpc.py:31-33: numpy state [O] (or [n_states, O]) -> numpy action [A] (or [n_states, A])."""
        action, _ = self.do_generate_action(state)
        return action

    def do_generate_action(self, state, seed=None):
        """cem_mpc.py:35-68 -> (action, best_score). Host buffers in, host buffers out."""
        planner = self._ensure_planner()
        a_dim = self.action_space.shape[0]
        st = np.ascontiguousarray(np.asarray(state, dtype=np.float32))
        batched = st.ndim == 2
        if st.size != self.n_states * self.model.observation_space_dim:
            raise ValueError("state has %d values, expected %d x %d"
                             % (st.size, self.n_states, self.model.observation_space_dim))
        action = np.empty((self.n_states, a_dim), dtype=np.float32)
        score = np.empty((self.n_states,), dtype=np.float32)
        iters = np.empty((self.n_states,), dtype=np.int32)
        _lib.check(self._lib.simba_plan_host(planner, _device.ptr(st), self._next_seed(seed),
                                             _device.ptr(action), _device.ptr(score),
                                             _device.ptr(iters)))
        self.iterations_run = iters
        if batched:
            return action, score
        return action[0], score[0]

    def plan_device(self, states, seed=None, out_action=None, out_score=None, out_iterations=None):
        """Asynchronous planning call on device tensors (no host copies, no sync): states [S, O]."""
        planner = self._ensure_planner()
        a_dim = self.action_space.shape[0]
        dev = states.device
        if out_action is None:
            out_action = torch.empty((self.n_states, a_dim), dtype=torch.float32, device=dev)
        if out_score is None:
            out_score = torch.empty((self.n_states,), dtype=torch.float32, device=dev)
        if out_iterations is None:
            out_iterations = torch.empty((self.n_states,), dtype=torch.int32, device=dev)
        _lib.check(self._lib.simba_plan(planner, _device.ptr(states), self._next_seed(seed),
                                        _device.ptr(out_action), _device.ptr(out_score),
                                        _device.ptr(out_iterations), _device.stream_ptr()))
        return out_action, out_score, out_iterations

    @property
    def launches_per_plan(self):
        n = C.c_int32()
        _lib.check(self._lib.simba_planner_launches_per_plan(self._ensure_planner(), C.byref(n)))
        return n.value

    def compute_objective(self, trajectories, action_sequences=None):
        """mpc_policy.py:26-39 (SafeCemMpc: safe_cem_mpc.py:76-96) on materialised trajectories
        [P*N, H+1, O] -> scores [N]. (The planning call never materialises them; this is the
        reference's public method kept for drop-in use.)"""
        planner = self._ensure_planner()
        traj, kind = _device.to_device(trajectories)
        expected = (self.particles * self.n_samples, self.horizon + 1, self.model.observation_space_dim)
        if tuple(traj.shape) != expected:
            raise ValueError("trajectories must be %s, got %s" % (expected, tuple(traj.shape)))
        scores = torch.empty((self.n_samples,), dtype=torch.float32, device=traj.device)
        _lib.check(self._lib.simba_score_trajectories(planner, _device.ptr(traj), _device.ptr(scores),
                                                      None, _device.stream_ptr()))
        return _device.like_input(scores, kind)
