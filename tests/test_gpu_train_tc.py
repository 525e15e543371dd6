"""bf16 tcgen05 ensemble training (MlpEnsemble(train_precision='bf16'), SIMBA_PREC_BF16_TC) against
oracle/train_oracle.py and against the fp32 trainer.

The GEMMs take bf16 operands (fp32 accumulation), so the bounds are the bf16 path's own, pinned at about
twice the worst value measured on a B200 over these shapes (DESIGN.md section 5, "bf16 training"):
  * one step: relative error of the loss, and per variable ||g - g_ref||_2 / ||g_ref||_2;
  * weights after n steps: |dw| <= 2 lr n (Adam moves a weight by about lr per step whatever its gradient's
    size, so a tiny gradient whose sign flips in bf16 costs 2 lr);
  * fit: the mean training loss over the last 10 % of the steps and the final validation loss differ
    from the fp32 trainer's by at most FIT_FRACTION of the fp32 run's loss drop.
Everything the step does in fp32 (NLL, clip, Adam, the fixed-order reductions) keeps the fp32 path's
determinism: fit equals the same batches fed one training_step at a time, and two runs are bit-identical."""
import ctypes as C

import numpy as np
import pytest

from oracle import train_oracle as T
from simba_b200 import _lib
from simba_b200.models import MlpEnsemble, TransitionModel
from tests.test_abi import _print_from_c

gpu = pytest.mark.gpu

LOSS_REL = 1.5e-3      # one step: |loss - loss_ref| / |loss_ref|  (worst measured 6.3e-4)
GRAD_REL = 0.3         # one step: ||g - g_ref|| / ||g_ref|| per variable  (worst measured 0.147)
FIT_FRACTION = 0.08    # fit: |bf16 - fp32| <= FIT_FRACTION * (fp32 loss drop)  (measured 0.027 at C5)

ONE_STEP_SHAPES = [(62, 60, 5, 64, 4, 128), (12, 10, 3, 16, 2, 40), (7, 5, 2, 9, 1, 33),
                   (62, 60, 2, 32, 2, 400), (20, 18, 2, 24, 3, 200), (9, 7, 1, 5, 2, 130)]


def _ensemble(n_in, n_out, members, batch, layers, units, lr=0.00025, schedule=False, steps=5000,
              epochs=1, seed=0, precision='bf16', dropout_rate=0.0):
    return MlpEnsemble(n_in, n_out, members, batch_size=batch, learning_rate=lr,
                       learning_rate_schedule=schedule, training_steps=steps, train_epochs=epochs,
                       mlp_params=dict(n_layers=layers, units=units, dropout_rate=dropout_rate), seed=seed,
                       train_precision=precision)


def _oracle(ens, dropout_rate=0.0, dropout_seed=0):
    return T.EnsembleTrainer([m.get_weights() for m in ens.ensemble], batch_size=ens.batch_size,
                             learning_rate=ens.learning_rate,
                             learning_rate_schedule=ens.learning_rate_schedule,
                             training_steps=ens.training_steps, train_epochs=ens.train_epochs,
                             dropout_rate=dropout_rate, dropout_seed=dropout_seed)


def _data(rng, members, rows, n_in, n_out, scale=1.0):
    x = rng.uniform(0, 1, (members, rows, n_in)).astype(np.float32)
    y = (rng.normal(0, 0.1, (members, rows, n_out)) * scale).astype(np.float32)
    return x, y


def _rel(got, ref):
    ref = np.asarray(ref, np.float64)
    return float(np.linalg.norm(np.asarray(got, np.float64) - ref) / max(np.linalg.norm(ref), 1e-30))


def _check_step(ens, ora, x, y, n_var):
    loss = float(ens.training_step(x, y))
    want = float(ora.training_step(x, y))
    assert abs(loss - want) <= LOSS_REL * abs(want), (loss, want)
    for e in range(ens.ensemble_size):
        for i, (got, ref) in enumerate(zip(ens.trainer_arrays('grads', e),
                                           ora.last_grads[e * n_var:(e + 1) * n_var])):
            assert _rel(got, ref) <= GRAD_REL, (e, i, _rel(got, ref))


def _check_weights(ens, ora, steps):
    for e in range(ens.ensemble_size):
        for got, ref in zip(ens.trainer_arrays('weights', e), ora.nets[e].arrays):
            assert np.abs(got - ref).max() <= 2 * ens.learning_rate * steps * (1 + 1e-3)


def test_trainer_config_size_matches_ctypes():
    assert _print_from_c('%zu', 'sizeof(simba_trainer_config_t)') == [C.sizeof(_lib.TrainerConfig)]


def test_train_precision_is_validated():
    with pytest.raises(ValueError):
        MlpEnsemble(12, 10, 2, train_precision='fp16')
    assert MlpEnsemble(12, 10, 2).train_precision == 'fp32'


@gpu
@pytest.mark.parametrize('shape', ONE_STEP_SHAPES)
def test_one_step_matches_oracle(shape):
    n_in, n_out, E, B, L, U = shape
    ens = _ensemble(n_in, n_out, E, B, L, U)
    ora = _oracle(ens)
    x, y = _data(np.random.default_rng(1), E, B, n_in, n_out)
    _check_step(ens, ora, x, y, 2 * L + 4)
    _check_weights(ens, ora, 1)
    assert ens.iterations == 1


@gpu
@pytest.mark.parametrize('shape,rate', [((62, 60, 3, 64, 4, 128), 0.1), ((12, 10, 2, 16, 2, 40), 0.5)])
def test_dropout_step_matches_oracle(shape, rate):
    """The bf16 chain draws the same Philox stream-4 keep masks as the fp32 chain (train_common.cuh)."""
    n_in, n_out, E, B, L, U = shape
    ens = _ensemble(n_in, n_out, E, B, L, U, lr=1e-3, seed=7, dropout_rate=rate)
    ora = _oracle(ens, rate, 7)
    rng = np.random.default_rng(12)
    for _ in range(2):
        x, y = _data(rng, E, B, n_in, n_out)
        _check_step(ens, ora, x, y, 2 * L + 4)
    _check_weights(ens, ora, 2)


@gpu
def test_clipvalue_and_schedule_over_several_steps():
    n_in, n_out, E, B, L, U = 12, 10, 3, 16, 2, 40
    ens = _ensemble(n_in, n_out, E, B, L, U, lr=1e-3, schedule=True, steps=3, epochs=4)
    ora = _oracle(ens)
    rng = np.random.default_rng(2)
    clipped = False
    for s in range(12):
        x, y = _data(rng, E, B, n_in, n_out, scale=300.0 if s < 4 else 1.0)
        got = float(ens.training_step(x, y))
        want = float(ora.training_step(x, y))
        clipped |= any(np.abs(g).max() > 1.0 for g in ora.last_grads)
        assert abs(got - want) <= LOSS_REL * abs(want), s
    assert clipped
    _check_weights(ens, ora, 12)
    # after 12 steps the schedule is at 0: further steps must not move anything
    before = [a.copy() for a in ens.trainer_arrays('weights', 0)]
    ens.training_step(*_data(rng, E, B, n_in, n_out))
    for a, b in zip(before, ens.trainer_arrays('weights', 0)):
        np.testing.assert_array_equal(a, b)
    assert ens.iterations == 13


@gpu
def test_training_step_with_fewer_rows_than_batch_size():
    n_in, n_out, E, B, L, U = 20, 18, 2, 200, 3, 200       # 2 row tiles allocated, 1 partly used
    ens = _ensemble(n_in, n_out, E, B, L, U)
    ora = _oracle(ens)
    x, y = _data(np.random.default_rng(8), E, 37, n_in, n_out)
    _check_step(ens, ora, x, y, 2 * L + 4)
    x, y = _data(np.random.default_rng(9), E, 160, n_in, n_out)  # two row tiles
    _check_step(ens, ora, x, y, 2 * L + 4)
    _check_weights(ens, ora, 2)


@gpu
def test_fit_equals_the_same_batches_one_step_at_a_time():
    n_in, n_out, E, B, L, U = 12, 10, 3, 16, 2, 40
    rng = np.random.default_rng(3)
    x = rng.uniform(0, 1, (50, n_in)).astype(np.float32)          # 50 rows / 16 -> batches 13,13,12,12
    y = rng.normal(0, 0.1, (50, n_out)).astype(np.float32)
    fitted = _ensemble(n_in, n_out, E, B, L, U, lr=5e-4, steps=25, seed=4)
    fitted.validation_split = 0.0
    stepped = _ensemble(n_in, n_out, E, B, L, U, lr=5e-4, steps=25, seed=4)
    np.random.seed(11)
    losses = fitted.fit(x, y)
    np.random.seed(11)
    train_idx, _ = fitted._split_indices(50)
    index, rows = fitted.batch_schedule(50, 25)
    assert sorted(set(rows.tolist())) == [12, 13]
    want = []
    for s in range(25):
        idx = train_idx[index[s, :, :rows[s]]]
        want.append(float(stepped.training_step(np.ascontiguousarray(x[idx]), np.ascontiguousarray(y[idx]))))
    np.testing.assert_array_equal(losses.astype(np.float32), np.array(want, np.float32))
    for e in range(E):
        for a, b in zip(fitted.trainer_arrays('weights', e), stepped.trainer_arrays('weights', e)):
            np.testing.assert_array_equal(a, b)
    assert fitted.iterations == 25


@gpu
def test_two_identical_fits_are_bit_identical():
    n_in, n_out, E, B, L, U = 62, 60, 5, 64, 4, 128
    rng = np.random.default_rng(6)
    x = rng.uniform(0, 1, (700, n_in)).astype(np.float32)
    y = rng.normal(0, 0.1, (700, n_out)).astype(np.float32)
    out = []
    for _ in range(2):
        ens = _ensemble(n_in, n_out, E, B, L, U, steps=40, seed=3, dropout_rate=0.1)
        np.random.seed(2)
        losses = ens.fit(x, y)
        out.append((losses, ens.trainer_arrays('weights', 1), ens.validation_losses))
    np.testing.assert_array_equal(out[0][0], out[1][0])
    for a, b in zip(out[0][1], out[1][1]):
        np.testing.assert_array_equal(a, b)
    assert out[0][2] == out[1][2]


@gpu
def test_validation_step_chunks_are_close_to_oracle():
    n_in, n_out, E, L, U = 12, 10, 3, 2, 40
    ens = _ensemble(n_in, n_out, E, 16, L, U)
    ora = _oracle(ens)
    rng = np.random.default_rng(4)
    for rows in (5, 64, 200, MlpEnsemble.EVAL_ROWS + 777):
        x = rng.uniform(0, 1, (rows, n_in)).astype(np.float32)
        y = rng.normal(0, 0.1, (rows, n_out)).astype(np.float32)
        got, want = float(ens.validation_step(x, y)), float(ora.validation_step(x, y))
        assert abs(got - want) <= LOSS_REL * abs(want), rows


def _dynamics(rng, n, O, A):
    obs = rng.uniform(-1, 1, (n, O)).astype(np.float32)
    act = rng.uniform(-1, 1, (n, A)).astype(np.float32)
    delta = 0.1 * np.tanh(obs) + 0.05 * np.pad(act, ((0, 0), (0, O - A))) + \
        0.02 * np.roll(obs, 1, axis=1) * act[:, :1]
    return np.concatenate([obs, act], axis=1), delta.astype(np.float32)


def _fit_pair(O, A, E, L, U, steps, n=3000):
    rng = np.random.default_rng(10)
    x, y = _dynamics(rng, n, O, A)
    out = {}
    for precision in ('fp32', 'bf16'):
        ens = _ensemble(O + A, O, E, 64, L, U, lr=1e-3, steps=steps, seed=5, precision=precision)
        np.random.seed(1)
        losses = ens.fit(x, y)
        out[precision] = (losses, ens.validation_losses[-1][1])
    return out


def _check_fit(out, steps):
    f_loss, f_val = out['fp32']
    b_loss, b_val = out['bf16']
    tail = max(steps // 10, 1)
    start = f_loss[:tail].mean()
    drop = start - f_loss[-tail:].mean()
    assert drop > 1.0, drop                               # the fp32 trainer learned the dynamics
    assert np.isfinite(b_loss).all()
    assert abs(b_loss[-tail:].mean() - f_loss[-tail:].mean()) <= FIT_FRACTION * drop
    assert abs(b_val - f_val) <= FIT_FRACTION * drop
    assert b_loss[-tail:].mean() < start - 0.5 * drop and b_val < start - 0.5 * drop


@gpu
def test_c5_shape_fit_meets_the_fit_bound():
    steps = 300
    _check_fit(_fit_pair(60, 2, 10, 4, 400, steps), steps)


@gpu
def test_wide_observation_fit_meets_the_fit_bound():
    steps = 300
    _check_fit(_fit_pair(92, 2, 5, 4, 128, steps), steps)


@gpu
def test_bf16_trained_weights_reach_the_model_handle():
    """After a bf16 fit, the model handle (through simba_trainer_sync_model) predicts exactly what a fresh
    model built on the trained weights predicts, on both rollout precisions."""
    from simba_b200.spaces import Box
    O, A = 6, 2
    kw = dict(ensemble_size=3, batch_size=32, learning_rate=2e-3, learning_rate_schedule=False,
              training_steps=200, mlp_params=dict(n_layers=2, units=64), train_epochs=1)
    obs_space, act_space = Box([-2.0] * O, [2.0] * O), Box([-1.0] * A, [1.0] * A)
    tm = TransitionModel('mlp_ensemble', obs_space, act_space, True, True, train_precision='bf16', **kw)
    x, y = _dynamics(np.random.default_rng(5), 600, O, A)
    before = tm.predict(x[:90])
    np.random.seed(0)
    losses = tm.fit(x, x[:, :O] + y)
    assert np.isfinite(losses).all() and losses[-20:].mean() < losses[:20].mean() - 0.5
    after = tm.predict(x[:90])
    assert np.abs(after - before).max() > 1e-3
    fresh = TransitionModel('mlp_ensemble', obs_space, act_space, True, True, **kw)
    fresh.model.load_state_arrays(tm.model.state_arrays())
    fresh.model._set_scaler(*tm.model._scaler)
    for precision in ('fp32', 'bf16'):
        np.testing.assert_array_equal(tm.predict(x[:90], precision=precision),
                                      fresh.predict(x[:90], precision=precision))


@gpu
@pytest.mark.parametrize('obs,act,layers,units', [(60, 2, 4, 417), (125, 1, 2, 64), (60, 2, 7, 128),
                                                  (122, 5, 2, 64)])
def test_shapes_outside_coverage_are_rejected_not_run_in_fp32(obs, act, layers, units):
    ens = _ensemble(obs + act, obs, 1, 8, layers, units)
    x, y = _data(np.random.default_rng(0), 1, 8, obs + act, obs)
    with pytest.raises(_lib.SimbaError) as err:
        ens.training_step(x, y)
    assert err.value.code == -6
    for limit in ('416', '126', '124', 'n_layers <= 6', 'fp32'):
        assert limit in str(err.value)
    plain = _ensemble(obs + act, obs, 1, 8, layers, units, precision='fp32')
    assert np.isfinite(float(plain.training_step(x, y)))
