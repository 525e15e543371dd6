"""TransitionModel — mirrors simba/models/transition_model.py for the inference methods.

`unfold_sequences` (transition_model.py:64-77), `scale` (:79-87), `predict` (:52-56) and
`simulate_trajectories` (:58-62) run on the GPU through libsimba_b200.so. The rollout methods take
`precision='fp32'` (fp32 SIMT kernel, simba_unfold) or `precision='bf16'`: the bf16 tensor-core kernels
a bf16 CemMpc plans with (simba_unfold_tc), so the trajectories are the ones that planner scores. `fit` (:34-40) fits the
scaler statistics (`_fit_statistics`, :42-50) and trains the ensemble on scaled inputs and
observation deltas with the device trainer (MlpEnsemble.fit).
"""
import numpy as np
import torch

from .. import _device, _lib
from ..spaces import is_box_like
from .mlp_ensemble import MlpEnsemble
from .model import BaseModel

_MODELS = {'mlp_ensemble': MlpEnsemble, 'MlpEnsemble': MlpEnsemble}


class TransitionModel(BaseModel):
    def __init__(self, model, observation_space, action_space, scale_features,
                 sampling_propagation, **kwargs):
        assert is_box_like(observation_space) and is_box_like(action_space)
        super().__init__(observation_space.shape[0] + action_space.shape[0],
                         observation_space.shape[0])
        self.model_scope = model
        if isinstance(model, str):
            if model not in _MODELS:
                raise ValueError("unknown model %r" % (model,))
            self.model = _MODELS[model](inputs_dim=self.inputs_dim, outputs_dim=self.outputs_dim,
                                        **kwargs)
        else:
            self.model = model           # an existing MlpEnsemble (weights shared)
        self.observation_space = observation_space
        self.action_space = action_space
        self.scale_features = scale_features
        self.sampling_propagation = sampling_propagation
        self.observation_space_dim = observation_space.shape[0]
        self.action_space_dim = action_space.shape[0]
        self.inputs_min = np.concatenate([observation_space.low, action_space.low]).astype(np.float32)
        self.inputs_max = np.concatenate([observation_space.high, action_space.high]).astype(np.float32)
        self._lib = _lib.load()
        self._push_scaler()

    def _push_scaler(self):
        finite = np.all(np.isfinite(self.inputs_min)) and np.all(np.isfinite(self.inputs_max))
        if self.scale_features and not finite:
            # deferred: the handle reports SIMBA_ERR_NONFINITE when it is first used (the reference
            # would silently produce NaN, transition_model.py:85-87)
            self.model._set_scaler(self.inputs_min, self.inputs_max, True)
        else:
            self.model._set_scaler(self.inputs_min, self.inputs_max, self.scale_features)

    def set_statistics(self, inputs_min, inputs_max):
        self.inputs_min = np.asarray(inputs_min, dtype=np.float32)
        self.inputs_max = np.asarray(inputs_max, dtype=np.float32)
        self._push_scaler()

    def build(self):
        self.model.build()

    def _fit_statistics(self, inputs):
        """transition_model.py:42-50."""
        if not self.scale_features:
            return
        high = np.concatenate([self.observation_space.high, self.action_space.high])
        low = np.concatenate([self.observation_space.low, self.action_space.low])
        self.set_statistics(np.where(np.isfinite(low), low, inputs.min(axis=0)),
                            np.where(np.isfinite(high), high, inputs.max(axis=0)))

    def fit(self, inputs, targets):
        """transition_model.py:34-40."""
        inputs = np.asarray(inputs, dtype=np.float32)
        self._fit_statistics(inputs)
        observations = inputs[:, :self.observation_space_dim]
        next_observations = np.asarray(targets, dtype=np.float32)
        return self.model.fit(self.scale(inputs), (next_observations - observations).astype(np.float32))

    def predict(self, inputs, *, precision='fp32'):
        """transition_model.py:52-56 -> np[B, 2, O]. `precision` as in unfold_sequences."""
        inputs = np.asarray(inputs, dtype=np.float32)
        return self.simulate_trajectories(
            current_state=inputs[..., :self.observation_space_dim],
            action_sequences=np.expand_dims(inputs[..., -self.action_space_dim:], axis=1),
            precision=precision)

    def simulate_trajectories(self, current_state, action_sequences, eps=None, seed=0, *, precision='fp32'):
        """transition_model.py:58-62 -> np[B, H+1, O]. `precision` as in unfold_sequences."""
        out = self.unfold_sequences(np.asarray(current_state, dtype=np.float32),
                                    np.asarray(action_sequences, dtype=np.float32), eps=eps, seed=seed,
                                    precision=precision)
        return out if isinstance(out, np.ndarray) else out.cpu().numpy()

    def unfold_sequences(self, s_0, action_sequences, eps=None, seed=0, *, precision='fp32'):
        """transition_model.py:64-77. s_0 [B, O], action_sequences [B, H, A] -> [B, H+1, O].
        eps [H, B, O]: the N(0,1) draws of the per-step Normal.sample(); if None they come from
        the Philox NOISE stream with `seed` (row = batch index).

        precision='fp32' runs the fp32 SIMT kernel. precision='bf16' runs the bf16 tcgen05 kernel that a
        bf16 CemMpc plans with (weights, activations and draws rounded to bf16, states in fp32; s_0 is
        returned bit for bit): the same draws and actions give the trajectories that planner scores.
        Shapes no tcgen05 kernel covers raise SimbaError (code -6); there is no fp32 fall-back."""
        if precision not in ('fp32', 'bf16'):
            raise ValueError("precision must be 'fp32' or 'bf16', not %r" % (precision,))
        entry = self._lib.simba_unfold if precision == 'fp32' else self._lib.simba_unfold_tc
        s0, kind = _device.to_device(s_0)
        acts, _ = _device.to_device(action_sequences)
        b, horizon = acts.shape[0], acts.shape[1]
        e = None
        if eps is not None:
            e, _ = _device.to_device(eps)
            assert tuple(e.shape) == (horizon, b, self.observation_space_dim)
        traj = torch.empty((b, horizon + 1, self.observation_space_dim), dtype=torch.float32,
                           device=s0.device)
        h = self.model._ensure_handle()
        _lib.check(entry(h, _device.ptr(s0), _device.ptr(acts), _device.ptr(e),
                         int(seed), b, horizon, int(bool(self.sampling_propagation)),
                         _device.ptr(traj), _device.stream_ptr()))
        return _device.like_input(traj, kind)

    def scale(self, inputs):
        """transition_model.py:79-87."""
        x, kind = _device.to_device(inputs)
        out = torch.empty_like(x)
        h = self.model._ensure_handle()
        _lib.check(self._lib.simba_scale(h, _device.ptr(x), x.shape[0], _device.ptr(out),
                                         _device.stream_ptr()))
        return _device.like_input(out, kind)

    def save(self, path=None):
        """The reference's save() is a stub (transition_model.py:89-93). With a path: one .npz with
        the ensemble's Keras-ordered variables and the scaler statistics (SURVEY.md section 8 f2)."""
        if path is None:
            return
        np.savez(path, inputs_min=self.inputs_min, inputs_max=self.inputs_max,
                 scale_features=int(bool(self.scale_features)),
                 ensemble_size=self.model.ensemble_size, n_layers=self.model.n_layers,
                 units=self.model.units, inputs_dim=self.model.inputs_dim,
                 outputs_dim=self.model.outputs_dim, **self.model.state_arrays())

    def load(self, path=None):
        if path is None:
            return
        self.model.load_weights(path)
        with np.load(path) as f:
            self.set_statistics(f['inputs_min'], f['inputs_max'])
