"""oracle/mppi_oracle.py: the MPPI update against an independent float64 restatement and its limits, and whole CPU
plans (no GPU)."""
import numpy as np
import pytest
from scipy.special import softmax

from oracle import mppi_oracle as mo
from oracle import simba_oracle as so
from tests import helpers


def _data(N=300, H=6, A=2, seed=0):
    rng = np.random.default_rng(seed)
    return (rng.normal(0.0, 1.0, N).astype(np.float32), rng.uniform(-1, 1, (N, H, A)).astype(np.float32),
            rng.uniform(-0.5, 0.5, (H, A)).astype(np.float32))


def _f64_update(mu, scores, acts, temperature, smoothing):
    """float64, written differently: scipy's softmax over the non-NaN scores, a tensordot for the mean."""
    keep = ~np.isnan(scores)
    if not keep.any():
        return np.asarray(mu, np.float64)
    p = softmax(np.asarray(scores[keep], np.float64) / temperature)
    mean = np.tensordot(p, np.asarray(acts[keep], np.float64), axes=1)
    return smoothing * np.asarray(mu, np.float64) + (1.0 - smoothing) * mean


@pytest.mark.parametrize("temperature", [0.05, 0.5, 5.0])
@pytest.mark.parametrize("smoothing", [0.0, 0.5])
def test_update_agrees_with_float64_restatement(temperature, smoothing):
    scores, acts, mu = _data()
    scores[::11] = np.nan
    got = mo.mppi_update(mu, scores, acts, temperature, smoothing)
    assert got.dtype == np.float32
    assert np.allclose(got, _f64_update(mu, scores, acts, temperature, smoothing), rtol=1e-6, atol=1e-6)
    got64 = mo.mppi_update(mu, scores, acts, temperature, smoothing, dtype=np.float64)
    assert np.allclose(got64, _f64_update(mu, scores, acts, temperature, smoothing), rtol=1e-12, atol=1e-12)


def test_low_temperature_gives_the_best_sequence_and_high_the_plain_mean():
    scores, acts, mu = _data()
    best = int(np.argmax(scores))
    assert np.array_equal(mo.mppi_mean(scores, acts, 1e-6), acts[best])
    assert np.allclose(mo.mppi_mean(scores, acts, 1e30), acts.mean(0, dtype=np.float64), rtol=0, atol=1e-6)


def test_smoothing():
    scores, acts, mu = _data()
    mean = mo.mppi_mean(scores, acts, 0.5)
    assert np.array_equal(mo.mppi_update(mu, scores, acts, 0.5, 0.0), mean)
    assert np.array_equal(mo.mppi_update(mu, scores, acts, 0.5, 0.5),
                          np.float32(0.5) * mu + np.float32(0.5) * mean)


def test_nan_scores():
    scores, acts, mu = _data()
    scores[:] = np.nan
    assert mo.mppi_mean(scores, acts, 1.0) is None and mo.best_candidate(scores) is None
    assert np.array_equal(mo.mppi_update(mu, scores, acts, 1.0, 0.3), mu)
    scores, acts, mu = _data()
    scores[5] = np.nan
    keep = np.arange(len(scores)) != 5
    assert np.allclose(mo.mppi_mean(scores, acts, 1.0), mo.mppi_mean(scores[keep], acts[keep], 1.0), rtol=0, atol=1e-7)


def test_unsafe_candidates_weigh_nothing_at_small_temperature():
    scores, acts, mu = _data()
    scores[:10] -= np.float32(100.0)
    keep = np.arange(len(scores)) >= 10
    assert np.allclose(mo.mppi_mean(scores, acts, 1.0), mo.mppi_mean(scores[keep], acts[keep], 1.0), atol=1e-7)


def _planner(c, objective, temperature=0.5):
    ens = so.MlpEnsemble(c['weights'])
    tm = so.TransitionModel(ens, c['smin'], c['smax'], True, True)
    env = so.Environment(so.Scorer(None, c['table']), so.Box([-1.0] * c['A'], [1.0] * c['A']), None)
    return mo.MppiPlanner(tm, env, c['H'], c['I'], 0.0, c['N'], c['P'], 0.01, temperature,
                          posterior_mean_threashold=0.15, objective=helpers.OBJ[objective])


@pytest.mark.parametrize("objective", ['reward', 'penalty', 'least_cost'])
def test_whole_plan_runs_every_iteration_and_acts_from_the_mean(objective):
    from simba_b200 import synthetic
    c = helpers.workload('tiny')
    z, eps, zf = synthetic.make_draws(c['I'], 1, c['N'], c['H'], c['A'], c['P'], c['O'])
    tr = so.Trace()
    action, score, iters = _planner(c, objective).do_generate_action(c['state'], z[:, 0], eps[:, 0], zf[0], tr)
    assert iters == c['I'] == len(tr)
    assert np.array_equal(action, tr[-1]['mu'][0] + zf[0] * np.float32(0.01))
    assert score == max(np.nanmax(t['scores']) for t in tr)
    # the first iteration's mean is the weighted mean of its candidates (smoothing 0)
    assert np.array_equal(tr[0]['mu'], mo.mppi_mean(tr[0]['scores'], tr[0]['actions'], 0.5))


def test_feasible_first_has_no_scalar_score():
    with pytest.raises(ValueError):
        _planner(helpers.workload('tiny'), 'feasible_first')
