"""The swish forms of the oracles (tests/swish_ref.py, tf.nn.swish = z * sigmoid(z)): the numpy and torch
restatements agree, the training oracle's analytic gradients match float64 central differences with and without
dropout and drive the training oracle's steps, and MlpEnsemble accepts exactly the swish spellings the reference's
eval() of mlp_params['activation'] would turn into tf.nn.swish."""
import numpy as np
import pytest
import torch

from oracle import simba_oracle as so
from oracle import train_oracle as T
from tests import swish_ref
from tests.test_train_oracle import _member


def _members(rng, E, n_in, n_out, units, layers, dtype=np.float32):
    return [_member(rng, n_in, n_out, units, layers, dtype) for _ in range(E)]


def test_numpy_and_torch_swish_forward_agree():
    rng = np.random.default_rng(0)
    members = _members(rng, 3, 9, 7, 32, 3)
    x = rng.normal(0, 1.5, (3 * 40, 9)).astype(np.float32)
    mu, var = swish_ref.MlpEnsemble(members).forward(x)
    mu_t, var_t = swish_ref.TorchEnsemble(members).forward(torch.from_numpy(x))
    np.testing.assert_allclose(mu, mu_t.numpy(), rtol=1e-5, atol=1e-6)
    np.testing.assert_allclose(var, var_t.numpy(), rtol=1e-5, atol=1e-7)
    relu_mu, _ = so.MlpEnsemble(members).forward(x)
    assert np.abs(relu_mu - mu).max() > 1e-2                  # the activation is applied


def test_training_oracle_steps_swish_members():
    rng = np.random.default_rng(1)
    members = _members(rng, 2, 5, 3, 8, 2)
    x = rng.uniform(0, 1, (2, 6, 5)).astype(np.float32)
    y = rng.normal(0, 0.1, (2, 6, 3)).astype(np.float32)
    ora = swish_ref.EnsembleTrainer(members, batch_size=6, learning_rate_schedule=False)
    want = sum(swish_ref.MemberNet(m).loss_and_grads(x[e], y[e], 0.5)[0] for e, m in enumerate(members))
    assert ora.training_step(x, y) == pytest.approx(want, rel=1e-6)
    relu = T.EnsembleTrainer(members, batch_size=6, learning_rate_schedule=False)
    assert abs(relu.training_step(x, y) - want) > 1e-4


def test_swish_matches_its_definition():
    z = np.linspace(-30, 30, 601).astype(np.float64)
    np.testing.assert_allclose(swish_ref.swish(z), z / (1 + np.exp(-z)), rtol=1e-15)
    assert swish_ref.swish(np.float32(-200.0)) == 0.0


@pytest.mark.parametrize("rate", [0.0, 0.1])
def test_swish_gradients_match_central_differences(rate):
    rng = np.random.default_rng(2)
    net = swish_ref.MemberNet(_member(rng, 5, 3, 8, 2, np.float64), np.float64)
    x = rng.normal(size=(7, 5))
    y = rng.normal(size=(7, 3))
    keep = None
    if rate > 0:
        keep = [(rng.uniform(size=(7, 8)) >= rate) / (1.0 - rate) for _ in range(2)]
        assert any((k == 0).any() for k in keep)

    def loss():
        return T.negative_log_likelihood(y, *net.forward(x, keep)[:2]) * 0.2

    got, grads = net.loss_and_grads(x, y, 0.2, keep)
    assert got == pytest.approx(loss())
    h = 1e-6
    for a, g in zip(net.arrays, grads):
        flat = a.reshape(-1)
        for j in rng.choice(flat.size, size=min(flat.size, 6), replace=False):
            v = flat[j]
            flat[j] = v + h
            up = loss()
            flat[j] = v - h
            dn = loss()
            flat[j] = v
            assert g.reshape(-1)[j] == pytest.approx((up - dn) / (2 * h), rel=2e-5, abs=1e-9)


@pytest.mark.parametrize("spelling", ['tf.nn.swish', 'tf.nn.silu', 'swish', 'silu'])
def test_mlp_ensemble_accepts_swish_spellings(spelling):
    from simba_b200 import _lib
    from simba_b200.models import MlpEnsemble
    ens = MlpEnsemble(12, 10, 2, mlp_params=dict(n_layers=2, units=16, activation=spelling))
    assert ens.activation == _lib.ACT_SWISH
    assert MlpEnsemble(12, 10, 2, mlp_params=dict(activation='tf.nn.relu')).activation == _lib.ACT_RELU


@pytest.mark.parametrize("spelling", ['tf.nn.tanh', 'tf.nn.elu', 'tf.nn.gelu'])
def test_other_activations_are_still_rejected(spelling):
    from simba_b200 import _lib
    from simba_b200.models import MlpEnsemble
    with pytest.raises(_lib.SimbaError) as e:
        MlpEnsemble(12, 10, 2, mlp_params=dict(activation=spelling))
    assert e.value.code == -6 and 'swish' in str(e.value)
