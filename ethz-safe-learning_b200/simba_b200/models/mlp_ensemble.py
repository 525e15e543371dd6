"""MlpEnsemble — simba/models/mlp_ensemble.py behind the same interface.

The E Gaussian MLPs (mlp_ensemble.py:37-61, :111-112) live as packed fp32 + bf16 images inside a
`simba_model` handle of libsimba_b200.so; `forward` / `__call__` (mlp_ensemble.py:122-132,
:189-193) run the fp32 CUDA kernel, or with precision='bf16' the bf16 tcgen05 kernels a bf16 planner
rolls out on. Training (`training_step`, `validation_step`, `fit`,
mlp_ensemble.py:134-187; SURVEY.md section 8 f1) runs on fp32 master weights inside a
`simba_trainer` handle; the trained weights are handed back to the model handle (and to
`ensemble[e].get_weights()`) the next time either is used.
"""
import ctypes as C

import numpy as np
import torch

from .. import _device, _lib


class MemberWeights(object):
    """One GaussianDistMlp's variables in Keras order (mlp_ensemble.py:46-50, :28-30):
    L x (kernel[in, U], bias[U]), mu head (kernel[U, O], bias[O]), var head (kernel[U, O], bias[O])."""

    def __init__(self, owner, index, arrays):
        self._owner = owner
        self._index = index
        self._arrays = arrays

    def get_weights(self):
        self._owner._pull_trained()
        return [a.copy() for a in self._arrays]

    def set_weights(self, arrays):
        if len(arrays) != len(self._arrays):
            raise ValueError("expected %d arrays, got %d" % (len(self._arrays), len(arrays)))
        new = []
        for old, a in zip(self._arrays, arrays):
            a = np.ascontiguousarray(np.asarray(a, dtype=np.float32))
            if a.shape != old.shape:
                raise ValueError("shape %s does not match %s" % (a.shape, old.shape))
            new.append(a)
        self._owner._pull_trained()
        self._arrays = new
        self._owner._dirty = True
        self._owner._drop_trainer()      # Adam slots restart with the new variables

    @property
    def trainable_variables(self):
        return self.get_weights()


# mlp_params['activation'] spellings -> simba_activation
ACTIVATIONS = {'tf.nn.relu': _lib.ACT_RELU, 'relu': _lib.ACT_RELU,
               'tf.nn.swish': _lib.ACT_SWISH, 'tf.nn.silu': _lib.ACT_SWISH, 'swish': _lib.ACT_SWISH,
               'silu': _lib.ACT_SWISH}


def glorot_uniform(rng, fan_in, fan_out):
    """Keras Dense default initialiser (mlp_ensemble.py:13, :28-30)."""
    limit = np.sqrt(6.0 / (fan_in + fan_out))
    return rng.uniform(-limit, limit, size=(fan_in, fan_out)).astype(np.float32)


class MlpEnsemble(object):
    def __init__(self, inputs_dim, outputs_dim, ensemble_size, batch_size=64, validation_split=0.2,
                 learning_rate=0.00025, learning_rate_schedule=True, training_steps=5000,
                 mlp_params=None, train_epochs=1, seed=0, train_precision='fp32'):
        if train_precision not in _lib.PRECISIONS:
            raise ValueError("train_precision must be one of %s, got %r"
                             % (sorted(_lib.PRECISIONS), train_precision))
        mlp_params = dict(mlp_params or {})
        # 'fp32': the fp32 SIMT trainer; 'bf16': GEMMs on bf16 tcgen05 tensor cores with fp32 accumulation,
        # NLL and Adam (DESIGN.md section 5, "bf16 training"). Shapes the bf16 trainer does not cover raise
        # SimbaError SIMBA_ERR_UNSUPPORTED when the trainer is created.
        self.train_precision = train_precision
        self.inputs_dim = inputs_dim
        self.outputs_dim = outputs_dim
        self.ensemble_size = ensemble_size
        self.batch_size = batch_size
        self.validation_split = validation_split
        self.training_steps = training_steps
        self.learning_rate = learning_rate
        self.learning_rate_schedule = bool(learning_rate_schedule)
        self.train_epochs = train_epochs
        self.mlp_params = mlp_params
        self.n_layers = int(mlp_params.get('n_layers', 4))
        self.units = int(mlp_params.get('units', 128))
        activation = mlp_params.get('activation', 'tf.nn.relu')
        if activation not in ACTIVATIONS:
            raise _lib.SimbaError(-6, "only ReLU and swish hidden activations are fused (got %r)" % (activation,))
        # the reference eval()s the string (mlp_ensemble.py:14): tf.nn.silu is tf.nn.swish
        self.activation = ACTIVATIONS[activation]
        # inference runs with training=False, so dropout is the identity there; training_step applies
        # it after every hidden activation (mlp_ensemble.py:17-22) with Philox masks keyed by dropout_seed
        self.dropout_rate = float(mlp_params.get('dropout_rate', 0.0))
        self.dropout_seed = int(seed)
        rng = np.random.default_rng(seed)
        self.ensemble = []
        for e in range(ensemble_size):
            arrays = []
            fan_in = inputs_dim
            for _ in range(self.n_layers):
                arrays += [glorot_uniform(rng, fan_in, self.units), np.zeros(self.units, np.float32)]
                fan_in = self.units
            for _ in range(2):
                arrays += [glorot_uniform(rng, self.units, outputs_dim),
                           np.zeros(outputs_dim, np.float32)]
            self.ensemble.append(MemberWeights(self, e, arrays))
        self._handle = None
        self._dirty = True
        self._scaler = None          # (min, max, scale_features) set by TransitionModel
        self._trainer = None
        self._trained_ahead = False  # the trainer's master weights are newer than the model handle
        self._lib = _lib.load()

    # -- device image ------------------------------------------------------------------------
    def _ensure_handle(self):
        self._pull_trained()
        if self._handle is None:
            _device.require_cuda()
            cfg = _lib.ModelConfig(self.outputs_dim, self.inputs_dim - self.outputs_dim,
                                   self.ensemble_size, self.n_layers, self.units)
            h = C.c_void_p()
            _lib.check(self._lib.simba_model_create(C.byref(cfg), C.byref(h)))
            self._handle = h
            _lib.check(self._lib.simba_model_set_activation(h, self.activation))
            self._dirty = True
        if self._dirty:
            for e, member in enumerate(self.ensemble):
                arrays = member._arrays
                for l in range(self.n_layers + 2):
                    _lib.check(self._lib.simba_model_set_layer(
                        self._handle, e, l, _device.ptr(arrays[2 * l]), _device.ptr(arrays[2 * l + 1])))
            if self._scaler is None:
                _lib.check(self._lib.simba_model_set_scaler(self._handle, None, None, 0))
            else:
                mn, mx, on = self._scaler
                _lib.check(self._lib.simba_model_set_scaler(
                    self._handle, _device.ptr(mn), _device.ptr(mx), int(on)))
            _lib.check(self._lib.simba_model_commit(self._handle))
            self._dirty = False
        return self._handle

    def _set_scaler(self, inputs_min, inputs_max, scale_features):
        self._scaler = (np.ascontiguousarray(inputs_min, dtype=np.float32),
                        np.ascontiguousarray(inputs_max, dtype=np.float32), bool(scale_features))
        self._dirty = True

    def __del__(self):
        try:
            self._drop_trainer()
            if self._handle is not None:
                self._lib.simba_model_destroy(self._handle)
        except Exception:
            pass

    # -- reference interface --------------------------------------------------------------------
    def build(self):
        self._ensure_handle()

    def _run(self, inputs, eps, precision):
        if precision not in _lib.PRECISIONS:
            raise ValueError("precision must be one of %s, got %r" % (sorted(_lib.PRECISIONS), precision))
        x, kind = _device.to_device(inputs)
        if x.dim() != 2 or x.shape[1] != self.inputs_dim:
            raise ValueError("inputs must be [B, %d]" % self.inputs_dim)
        b = x.shape[0]
        h = self._ensure_handle()
        mu = torch.empty((b, self.outputs_dim), dtype=torch.float32, device=x.device)
        var = torch.empty_like(mu)
        smp, e = None, None
        if eps is not None:
            e, _ = _device.to_device(eps)
            smp = torch.empty_like(mu)
        fn = self._lib.simba_ensemble_forward if precision == 'fp32' else self._lib.simba_ensemble_forward_tc
        _lib.check(fn(h, _device.ptr(x), _device.ptr(e), b, _device.ptr(mu), _device.ptr(var),
                      _device.ptr(smp), _device.stream_ptr()))
        return mu, var, smp, kind

    def forward(self, inputs, *, precision='fp32'):
        """mlp_ensemble.py:122-132: rows split into E contiguous chunks -> (cat_mus, cat_vars).
        precision='bf16' runs the bf16 tcgen05 kernels of a bf16 planner (inputs, weights and
        activations rounded to bf16, fp32 accumulation); shapes they do not cover raise SimbaError
        SIMBA_ERR_UNSUPPORTED."""
        mu, var, _, kind = self._run(inputs, None, precision)
        return _device.like_input(mu, kind), _device.like_input(var, kind)

    def __call__(self, inputs, eps=None, *args, precision='fp32', **kwargs):
        """mlp_ensemble.py:189-193 -> (mean, stddev, sample). `eps` are the N(0,1) draws of
        Normal.sample(); if omitted they are drawn with torch on the device. precision as in
        `forward`; with 'bf16' the sample takes eps rounded to bf16, as a bf16 plan does."""
        if precision not in _lib.PRECISIONS:
            raise ValueError("precision must be one of %s, got %r" % (sorted(_lib.PRECISIONS), precision))
        x, _ = _device.to_device(inputs)
        if eps is None:
            eps = torch.randn((x.shape[0], self.outputs_dim), dtype=torch.float32, device=x.device)
        mu, var, smp, kind = self._run(inputs, eps, precision)
        return (_device.like_input(mu, kind), _device.like_input(torch.sqrt(var), kind),
                _device.like_input(smp, kind))

    # -- weight hand-off on disk (SURVEY.md section 8 f2) ------------------------------------------
    def state_arrays(self):
        """{'member{e}/var{i}': array} in Keras variable order (mlp_ensemble.py:46-50, :28-30):
        the stable exchange format between a TF/torch-trained ensemble and the planner images."""
        out = {}
        for e, member in enumerate(self.ensemble):
            for i, a in enumerate(member.get_weights()):
                out['member%d/var%d' % (e, i)] = a
        return out

    def load_state_arrays(self, arrays):
        for e, member in enumerate(self.ensemble):
            n = len(member._arrays)
            missing = [i for i in range(n) if 'member%d/var%d' % (e, i) not in arrays]
            if missing:
                raise KeyError("member %d: variables %s are missing" % (e, missing))
            member.set_weights([arrays['member%d/var%d' % (e, i)] for i in range(n)])

    def save_weights(self, path):
        np.savez(path, ensemble_size=self.ensemble_size, n_layers=self.n_layers, units=self.units,
                 inputs_dim=self.inputs_dim, outputs_dim=self.outputs_dim, **self.state_arrays())

    def load_weights(self, path):
        with np.load(path) as f:
            for key, want in (('ensemble_size', self.ensemble_size), ('n_layers', self.n_layers),
                              ('units', self.units), ('inputs_dim', self.inputs_dim),
                              ('outputs_dim', self.outputs_dim)):
                if int(f[key]) != want:
                    raise ValueError("%s: file has %d, model has %d" % (key, int(f[key]), want))
            self.load_state_arrays({k: f[k] for k in f.files if k.startswith('member')})

    # -- training (mlp_ensemble.py:134-187) --------------------------------------------------------
    EVAL_ROWS = 4096

    def _drop_trainer(self):
        if self._trainer is not None:
            self._lib.simba_trainer_destroy(self._trainer)
            self._trainer = None
        self._trained_ahead = False

    def _ensure_trainer(self):
        h = self._ensure_handle()
        if self._trainer is None:
            cfg = _lib.TrainerConfig(int(self.batch_size), self.EVAL_ROWS, float(self.learning_rate),
                                     int(self.learning_rate_schedule), int(self.training_steps),
                                     int(self.train_epochs), 0.9, 0.999, 1e-5, 1.0,
                                     float(self.dropout_rate), int(self.dropout_seed),
                                     _lib.PRECISIONS[self.train_precision])
            t = C.c_void_p()
            _lib.check(self._lib.simba_trainer_create(h, C.byref(cfg), C.byref(t)))
            self._trainer = t
        return self._trainer

    def _pull_trained(self):
        """Hand the trainer's master weights to the model handle and to the host arrays."""
        if not self._trained_ahead:
            return
        self._trained_ahead = False
        _lib.check(self._lib.simba_trainer_sync_model(self._trainer, _device.stream_ptr()))
        for e, member in enumerate(self.ensemble):
            for l in range(self.n_layers + 2):
                _lib.check(self._lib.simba_model_get_layer(
                    self._handle, e, l, _device.ptr(member._arrays[2 * l]),
                    _device.ptr(member._arrays[2 * l + 1])))

    @property
    def iterations(self):
        """optimizer.iterations (mlp_ensemble.py:113)."""
        return 0 if self._trainer is None else int(self._lib.simba_trainer_iterations(self._trainer))

    def trainer_arrays(self, which, member):
        """Debug/test view of the trainer: which in {'weights', 'grads', 'm', 'v'} -> Keras-ordered
        list of arrays of `member`."""
        t = self._ensure_trainer()
        code = {'weights': 0, 'grads': 1, 'm': 2, 'v': 3}[which]
        out = []
        for l in range(self.n_layers + 2):
            k = np.empty_like(self.ensemble[member]._arrays[2 * l])
            b = np.empty_like(self.ensemble[member]._arrays[2 * l + 1])
            _lib.check(self._lib.simba_trainer_get(t, code, member, l, _device.ptr(k), _device.ptr(b)))
            out += [k, b]
        return out

    def training_step(self, inputs, targets):
        """mlp_ensemble.py:134-146. inputs [E, B, in], targets [E, B, out] -> loss (0-dim CUDA
        tensor; float(loss) synchronises). B may be anything up to the `batch_size` the ensemble was
        constructed with (the trainer's workspace is sized once for it; the reference accepts any B —
        construct the ensemble with the largest batch you will pass, a larger one raises SimbaError
        SIMBA_ERR_SHAPE)."""
        t = self._ensure_trainer()
        x, _ = _device.to_device(inputs)
        y, _ = _device.to_device(targets)
        if x.dim() != 3 or x.shape[0] != self.ensemble_size or x.shape[2] != self.inputs_dim or \
                tuple(y.shape) != (x.shape[0], x.shape[1], self.outputs_dim):
            raise ValueError("inputs must be [E, B, %d] and targets [E, B, %d]"
                             % (self.inputs_dim, self.outputs_dim))
        loss = torch.empty((), dtype=torch.float32, device=x.device)
        _lib.check(self._lib.simba_trainer_step(t, _device.ptr(x), _device.ptr(y), x.shape[1],
                                                _device.ptr(loss), _device.stream_ptr()))
        self._trained_ahead = True
        return loss

    def validation_step(self, inputs, targets):
        """mlp_ensemble.py:148-156: every member on the same rows."""
        t = self._ensure_trainer()
        x, _ = _device.to_device(inputs)
        y, _ = _device.to_device(targets)
        loss = torch.empty((), dtype=torch.float32, device=x.device)
        _lib.check(self._lib.simba_trainer_validation(t, _device.ptr(x), _device.ptr(y), x.shape[0],
                                                      _device.ptr(loss), _device.stream_ptr()))
        return loss

    def split_train_validate(self, inputs, targets):
        """mlp_ensemble.py:158-162."""
        train_idx, val_idx = self._split_indices(inputs.shape[0])
        return inputs[train_idx, ...], targets[train_idx, ...], inputs[val_idx, ...], targets[val_idx, ...]

    def _split_indices(self, n):
        indices = np.random.permutation(n)
        num_val = int(n * self.validation_split)
        return indices[num_val:], indices[:num_val]

    def batch_schedule(self, n_train, steps):
        """The batches fit() draws (mlp_ensemble.py:172-186) as index arrays into the training
        rows: (index int32 [steps, E, batch_size], rows int32 [steps]). One permutation per member
        per pass, np.array_split into ceil(n / batch_size) batches (sizes may differ by one)."""
        n_batches = int(np.ceil(n_train / self.batch_size))
        index = np.zeros((steps, self.ensemble_size, self.batch_size), dtype=np.int32)
        rows = np.zeros((steps,), dtype=np.int32)
        step = 0
        while step < steps:
            shuffles = np.array([np.random.permutation(n_train) for _ in range(self.ensemble_size)])
            for b in np.array_split(shuffles, n_batches, axis=1):
                index[step, :, :b.shape[1]] = b
                rows[step] = b.shape[1]
                step += 1
                if step == steps:
                    break
        return index, rows

    def fit(self, inputs, targets):
        """mlp_ensemble.py:164-187 -> np[training_steps] losses. The whole loop runs on the device:
        the data and the batch schedule are uploaded once, each step is one CUDA-graph launch."""
        inputs = np.asarray(inputs, dtype=np.float32)
        targets = np.asarray(targets, dtype=np.float32)
        assert inputs.shape[0] == targets.shape[0], \
            "Inputs batch size ({}) doesn't match targets batch size ({})".format(
                inputs.shape[0], targets.shape[0])
        assert np.isfinite(inputs).all() and np.isfinite(targets).all(), "Training data is not finite."
        t = self._ensure_trainer()
        train_idx, val_idx = self._split_indices(inputs.shape[0])
        index, rows = self.batch_schedule(train_idx.shape[0], self.training_steps)
        index = train_idx.astype(np.int32)[index]          # rows of `inputs`, not of the train subset
        x, _ = _device.to_device(inputs)
        y, _ = _device.to_device(targets)
        d_index, _ = _device.to_device(index, dtype=torch.int32)
        uneven = bool((rows != index.shape[2]).any())
        d_rows = _device.to_device(rows, dtype=torch.int32)[0] if uneven else None
        losses = torch.empty((self.training_steps,), dtype=torch.float32, device=x.device)
        x_val = y_val = None
        if val_idx.shape[0] > 0:
            x_val, _ = _device.to_device(inputs[val_idx])
            y_val, _ = _device.to_device(targets[val_idx])
        report = max(int(self.training_steps / 10), 1)
        self.validation_losses = []
        step = 0
        while step < self.training_steps:
            n = min(report - step % report, self.training_steps - step)
            _lib.check(self._lib.simba_trainer_fit(
                t, _device.ptr(x), _device.ptr(y), x.shape[0],
                C.c_void_p(d_index.data_ptr() + step * index.shape[1] * index.shape[2] * 4),
                C.c_void_p(0 if d_rows is None else d_rows.data_ptr() + step * 4), n,
                C.c_void_p(losses.data_ptr() + step * 4), _device.stream_ptr()))
            step += n
            if step % report == 0 and x_val is not None:
                self.validation_losses.append((step, self.validation_step(x_val, y_val)))
        self._trained_ahead = True
        out = losses.cpu().numpy().astype(np.float64)
        self.validation_losses = [(s, float(v)) for s, v in self.validation_losses]
        return out
