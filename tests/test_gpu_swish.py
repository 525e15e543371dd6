"""Swish ensembles (mlp_params['activation'] = 'tf.nn.swish', SIMBA_ACT_SWISH) on every path a ReLU ensemble runs,
against the swish forms of the oracles (tests/swish_ref.py).

  1  fp32 planning: rows within 1e-4 relative of the oracle, a whole SafeCemMpc plan with the oracle's elite indices
  2  bf16 planning on every tcgen05 variant: the same kernel and work items as the ReLU model of the shape, rows
     within DESIGN.md section 5's bf16 rules, a C1 plan within 5e-2 of the fp32 plan
  3  the bit-identities of the ReLU kernels: pair vs NO_PAIR, two-tile vs NO_TAIL_SPLIT, NO_PDL / NO_FUSE plans,
     batched vs per-state plans
  4  trajectories and forward: simba_unfold_tc scored = the bf16 planner's pairs, H = 1 forward identities,
     fp32 unfold / forward against the oracle
  5  training: one fp32 step against the swish training oracle (dropout 0 and 0.1), bf16 steps within pinned bounds, a fit
     that lowers the loss and whose weights reach a planner
  6  the boundary: simba_model_set_activation after a commit or with an unknown value
"""
import ctypes as C

import numpy as np
import pytest

from oracle import simba_oracle as so
from tests import helpers
from tests import swish_ref
from tests.test_gpu_dispatch_variants import _one_state, _pick_S, _set_switches
from tests.test_gpu_kernels import _oracle_rows, dev, P
from tests.test_gpu_tc_obs_wide import SCORERS, SENSORS

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")

SWISH = 'tf.nn.swish'


def _lib():
    from simba_b200 import _lib
    return _lib


def _oracle(c, objective='penalty', **kw):
    return swish_ref.planner(c, objective, **kw)


def _policy(c, objective='penalty', precision='bf16', activation=SWISH, **kw):
    return helpers.cuda_policy(c, objective, precision=precision, activation=activation, **kw)


def _choice(c, activation, switches=(), scorer_config=None):
    """simba_planner_rollout_kernel of a fresh planner -> (kernel constant, work items)."""
    L = _lib()
    kernel, items = C.c_int32(-1), C.c_int32(-1)
    with pytest.MonkeyPatch.context() as mp:
        _set_switches(mp, *switches)
        pol = _policy(c, activation=activation, scorer_config=scorer_config)
        L.check(L.load().simba_planner_rollout_kernel(pol._ensure_planner(), C.byref(kernel), C.byref(items)))
    return kernel.value, items.value


def _rows(pol, c, acts, eps):
    """simba_rollout_score of the planner for c['S'] copies of c's first state, each with the same actions and
    draws -> (return, cost mask, cost sum) of state 0's rows, after checking every state's rows are equal."""
    L = _lib()
    S, B = c['S'], c['P'] * c['N']
    state = np.asarray(c['state'], np.float32).reshape(-1, c['O'])[:1]
    ret = torch.zeros(S * B, dtype=torch.float32, device='cuda')
    mask = torch.zeros(S * B, dtype=torch.int64, device='cuda')
    csum = torch.zeros(S * B, dtype=torch.float32, device='cuda')
    d_state = dev(np.repeat(state, S, 0))
    d_acts = dev(np.repeat(acts[None], S, 0))
    d_eps = dev(np.repeat(eps[None], S, 0))
    L.check(L.load().simba_rollout_score(pol._ensure_planner(), P(d_state), P(d_acts), P(d_eps), 0, 0, None,
                                         P(ret), P(mask), P(csum), None))
    torch.cuda.synchronize()
    ret, mask, csum = (x.cpu().numpy().reshape(S, B) for x in (ret, mask, csum))
    for s in range(1, S):
        assert np.array_equal(ret[s], ret[0]) and np.array_equal(mask[s], mask[0])
    return ret[0], mask[0].view(np.uint64), csum[0]


def _draws(c, seed=6):
    rng = np.random.default_rng(seed)
    acts = rng.uniform(-1, 1, (c['N'], c['H'], c['A'])).astype(np.float32)
    eps = rng.standard_normal((c['H'], c['P'] * c['N'], c['O'])).astype(np.float32)
    return acts, eps


# ---- 1: fp32 planning ----------------------------------------------------------------------------------------------
@pytest.mark.parametrize("cfg,objective", [('tiny', 'penalty'), ('tiny', 'reward'), ('c1', 'penalty')])
def test_fp32_rows_match_oracle(cfg, objective):
    c = helpers.workload(cfg)
    pol = _policy(c, objective, precision='fp32')
    acts, eps = _draws(c)
    ret, mask, csum = _rows(pol, dict(c, S=1), acts, eps)
    _, cum0, mask0, csum0 = _oracle_rows(c, _oracle(c, objective), acts, eps, objective)
    relu = helpers.cuda_policy(c, objective, precision='fp32')
    ret_relu, _, _ = _rows(relu, dict(c, S=1), acts, eps)
    print("fp32 swish rows: max|dret| %.3g, rows differing from the ReLU model %.2f"
          % (np.abs(ret - cum0).max(), (ret != ret_relu).mean()))
    np.testing.assert_allclose(ret, cum0, rtol=1e-4, atol=1e-5)
    np.testing.assert_allclose(csum, csum0, rtol=1e-4, atol=1e-5)
    assert np.array_equal(mask, mask0)
    assert (ret != ret_relu).mean() > 0.5                 # the activation reached the kernel


def test_fp32_safe_plan_matches_oracle():
    from simba_b200 import synthetic
    L = _lib()
    c = helpers.workload('tiny')
    z, eps, zf = synthetic.make_draws(c['I'], 1, c['N'], c['H'], c['A'], c['P'], c['O'])
    tr = so.Trace()
    a0, s0, _ = _oracle(c).do_generate_action(c['state'], z[:, 0], eps[:, 0], zf[0], tr)
    pol = _policy(c, precision='fp32')
    pol.set_external_draws(z, eps, zf)
    action, score = pol.do_generate_action(c['state'])
    elite = pol.buffer(L.BUF_ELITE, torch.int32).cpu().numpy()
    assert np.array_equal(elite, tr[-1]['elite'])
    np.testing.assert_allclose(action, a0, rtol=1e-4, atol=1e-5)
    assert abs(score - s0) <= 1e-4 * max(1.0, abs(s0))


# ---- 2: bf16 planning on every tcgen05 variant ---------------------------------------------------------------------
def _variant_case(name):
    """-> (workload, switches, scorer_config, expected kernel constant)"""
    L = _lib()
    if name == 'pair':
        return helpers.workload('tiny'), (), None, L.ROLLOUT_TC_PAIR
    if name == 'one-cta':
        return helpers.workload('tiny'), ('SIMBA_B200_NO_PAIR',), None, L.ROLLOUT_TC_ONE_CTA
    if name == 'two-tile':
        c = helpers.workload('c1', H=8)
        S, _ = _pick_S(c, lambda v: v['kernel'] == 'two', 2)
        return helpers.workload('c1', H=8, S=S), (), None, L.ROLLOUT_TC_TWO_TILE
    if name == 'wide64':
        return helpers.workload('c5', H=10), (), None, L.ROLLOUT_TC_WIDE
    return helpers.workload('tiny', sensors=SENSORS[92]), (), SCORERS['goal4'], L.ROLLOUT_TC_WIDE_OBS


VARIANTS = ['pair', 'one-cta', 'two-tile', 'wide64', 'wide128-obs92']


@pytest.mark.parametrize("name", VARIANTS)
def test_bf16_rows_close_to_oracle_on_every_variant(name, monkeypatch):
    c, switches, scorer, kernel = _variant_case(name)
    got = _choice(c, SWISH, switches, scorer)
    assert got == _choice(c, 'tf.nn.relu', switches, scorer)
    assert got[0] == kernel
    _set_switches(monkeypatch, *switches)
    pol = _policy(c, scorer_config=scorer)
    acts, eps = _draws(c)
    ret, mask, _ = _rows(pol, c, acts, eps)
    c0 = dict(c, state=np.asarray(c['state'], np.float32).reshape(-1, c['O'])[0])
    _, cum0, mask0, _ = _oracle_rows(c0, _oracle(c0, scorer_config=scorer), acts, eps, 'penalty')
    err = np.abs(ret - cum0)
    agree = (mask == mask0).mean()
    cand = np.abs(ret.reshape(c['P'], c['N']).mean(0) - cum0.reshape(c['P'], c['N']).mean(0)).max()
    print("bf16 swish %s: mean|dret| %.4g max %.4g, candidate max %.4g, mask agreement %.4f"
          % (name, err.mean(), err.max(), cand, agree))
    assert np.all(np.isfinite(ret))
    assert err.mean() < 1e-2
    assert cand < 2e-2
    assert agree >= 1.0 - 0.002 * c['H']


def test_bf16_c1_plan_close_to_fp32_plan():
    from simba_b200 import synthetic
    c = helpers.workload('c1')
    z, eps, zf = synthetic.make_draws(c['I'], 1, c['N'], c['H'], c['A'], c['P'], c['O'])
    res = {}
    for precision in ('fp32', 'bf16'):
        pol = _policy(c, precision=precision)
        pol.set_external_draws(z, eps, zf)
        res[precision] = pol.do_generate_action(c['state'])
    print("swish C1 plan: bf16 score %.5f, fp32 %.5f" % (res['bf16'][1], res['fp32'][1]))
    assert np.all(np.isfinite(res['bf16'][0]))
    assert abs(res['bf16'][1] - res['fp32'][1]) < 5e-2


# ---- 3: bit-identities ---------------------------------------------------------------------------------------------
def _plan(c, monkeypatch, switches=(), draws=None, scorer=None):
    L = _lib()
    _set_switches(monkeypatch, *switches)
    pol = _policy(c, scorer_config=scorer)
    if draws is not None:
        pol.set_external_draws(*draws)
    S = c['S']
    a, s = pol.do_generate_action(np.asarray(c['state'], np.float32).reshape(S, c['O']), seed=None if draws else 9)
    out = dict(action=np.asarray(a).reshape(S, -1), score=np.asarray(s).reshape(S),
               mu=pol.buffer(L.BUF_MU).cpu().numpy().reshape(S, -1),
               elite=pol.buffer(L.BUF_ELITE, torch.int32).cpu().numpy().reshape(S, -1))
    _set_switches(monkeypatch)
    return out


def _equal(a, b, s=None):
    for k in a:
        assert np.array_equal(a[k] if s is None else a[k][s:s + 1], b[k]), (k, s)


def test_pair_equals_one_cta_and_switches_change_nothing(monkeypatch):
    from simba_b200 import synthetic
    c = helpers.workload('tiny')
    draws = synthetic.make_draws(c['I'], 1, c['N'], c['H'], c['A'], c['P'], c['O'], seed=3)
    ref = _plan(c, monkeypatch, draws=draws)
    for sw in ('SIMBA_B200_NO_PAIR', 'SIMBA_B200_NO_PDL', 'SIMBA_B200_NO_FUSE'):
        _equal(_plan(c, monkeypatch, (sw,), draws), ref)


def test_two_tile_equals_no_tail_split(monkeypatch):
    c = helpers.workload('c1', H=8, I=3)
    S, _ = _pick_S(c, lambda v: v['kernel'] == 'two' and v['split'], 2)
    c = helpers.workload('c1', H=8, I=3, S=S)
    _equal(_plan(c, monkeypatch, ('SIMBA_B200_NO_TAIL_SPLIT',)), _plan(c, monkeypatch))


@pytest.mark.parametrize("sensors", [None, 92])
def test_batched_plans_equal_per_state_plans(sensors, monkeypatch):
    from simba_b200 import synthetic
    scorer = SCORERS['goal4'] if sensors else None
    c = helpers.workload('tiny', sensors=SENSORS[sensors] if sensors else None, S=3, H=8, I=3, N=40)
    draws = synthetic.make_draws(c['I'], c['S'], c['N'], c['H'], c['A'], c['P'], c['O'], seed=5)
    ref = _plan(c, monkeypatch, draws=draws, scorer=scorer)
    for sw in ('SIMBA_B200_NO_PDL', 'SIMBA_B200_NO_FUSE'):
        _equal(_plan(c, monkeypatch, (sw,), draws, scorer), ref)
    z, eps, zf = draws
    for s in range(c['S']):
        _equal(ref, _plan(_one_state(c, s), monkeypatch, draws=(z[:, s:s + 1], eps[:, s:s + 1], zf[s:s + 1]),
                          scorer=scorer), s)


# ---- 4: trajectories and forward -----------------------------------------------------------------------------------
@pytest.mark.parametrize("cfg,sensors,scorer", [('c1', None, None), ('c5', None, None), ('c1', 92, 'goal4')])
def test_scored_trajectories_equal_the_planners_rollout_scores(cfg, sensors, scorer):
    L = _lib()
    lib = L.load()
    c = helpers.workload(cfg, sensors=SENSORS[sensors] if sensors else None)
    pol = _policy(c, scorer_config=SCORERS.get(scorer))
    pl = pol._ensure_planner()
    H, A, N, P_, O = c['H'], c['A'], c['N'], c['P'], c['O']
    B, seed = P_ * N, 7
    rng = np.random.default_rng(5)
    d_mu = dev(rng.uniform(-0.5, 0.5, (1, H, A)).astype(np.float32))
    d_sg = dev(rng.uniform(0.2, 1.0, (1, H, A)).astype(np.float32))
    acts = torch.empty((1, N, H, A), dtype=torch.float32, device='cuda')
    L.check(lib.simba_sample_actions(pl, P(d_mu), P(d_sg), None, seed, 0, None, P(acts), None))
    d_state = dev(np.asarray(c['state'], np.float32).reshape(1, O))
    ret = torch.empty((B,), dtype=torch.float32, device='cuda')
    mask = torch.empty((B,), dtype=torch.int64, device='cuda')
    csum = torch.empty((B,), dtype=torch.float32, device='cuda')
    L.check(lib.simba_rollout_score(pl, P(d_state), P(acts), None, seed, 0, None, P(ret), P(mask), P(csum), None))
    pairs_plan = torch.empty((1, N, 2), dtype=torch.float32, device='cuda')
    L.check(lib.simba_score_reduce(pl, P(ret), P(mask), P(csum), None, P(pairs_plan), None))
    traj = pol.model.unfold_sequences(d_state.expand(B, O).contiguous(), acts[0].repeat(P_, 1, 1).contiguous(),
                                      seed=seed, precision='bf16')
    scores = torch.empty((N,), dtype=torch.float32, device='cuda')
    pairs = torch.empty((N, 2), dtype=torch.float32, device='cuda')
    L.check(lib.simba_score_trajectories(pl, P(traj), P(scores), P(pairs), None))
    torch.cuda.synchronize()
    assert np.array_equal(pairs.cpu().numpy().view(np.uint32), pairs_plan[0].cpu().numpy().view(np.uint32))


def _ensemble(c, activation=SWISH):
    from simba_b200.models import MlpEnsemble
    ens = MlpEnsemble(c['O'] + c['A'], c['O'], c['E'],
                      mlp_params=dict(n_layers=c['L'], units=c['U'], activation=activation))
    for e in range(c['E']):
        ens.ensemble[e].set_weights(c['weights'][e])
    ens._ensure_handle()
    return ens


# name: (workload, sensors, overrides, rows per member, kernel)
FORWARD_CASES = {
    'c1-one-cta': ('c1', None, dict(), 600, 'TC_ONE_CTA'),
    'c1-two-tile': ('c1', None, dict(), 60 * 128 + 5, 'TC_TWO_TILE'),
    'c5-wide': ('c5', None, dict(), 300, 'TC_WIDE'),
    'c1-o92-wide-obs': ('c1', 92, dict(), 31 * 128 + 17, 'TC_WIDE_OBS'),
}


@pytest.mark.parametrize("name", list(FORWARD_CASES))
def test_forward_at_horizon_one_is_the_unfold_step(name):
    L = _lib()
    lib = L.load()
    cfg, sensors, over, per_member, kernel = FORWARD_CASES[name]
    c = helpers.workload(cfg, sensors=SENSORS[sensors] if sensors else None, var_bias=-2.0, **over)
    O, A, B = c['O'], c['A'], c['E'] * per_member
    rng = np.random.default_rng(21)
    x = rng.uniform(0, 1, (B, O + A)).astype(np.float32)
    x[:, O:] = rng.uniform(-1, 1, (B, A))
    ens = _ensemble(c)
    h = ens._ensure_handle()
    k, items = C.c_int32(-1), C.c_int32(-1)
    L.check(lib.simba_ensemble_forward_tc_kernel(h, B, C.byref(k), C.byref(items)))
    k2, items2 = C.c_int32(-1), C.c_int32(-1)
    L.check(lib.simba_ensemble_forward_tc_kernel(_ensemble(c, 'tf.nn.relu')._ensure_handle(), B, C.byref(k2),
                                                 C.byref(items2)))
    assert (k.value, items.value) == (k2.value, items2.value) and k.value == getattr(L, 'ROLLOUT_' + kernel)
    mu = torch.empty((B, O), dtype=torch.float32, device='cuda')
    var = torch.empty_like(mu)
    L.check(lib.simba_ensemble_forward_tc(h, P(dev(x)), None, B, P(mu), P(var), None, None))
    traj = torch.empty((B, 2, O), dtype=torch.float32, device='cuda')
    L.check(lib.simba_unfold_tc(h, P(dev(x[:, :O])), P(dev(x[:, O:].reshape(B, 1, A))), None, 0, B, 1, 0,
                                P(traj), None))
    torch.cuda.synchronize()
    assert np.array_equal(traj[:, 1].cpu().numpy(), x[:, :O] + mu.cpu().numpy())
    ref_mu, ref_var = swish_ref.MlpEnsemble(c['weights'], dtype=np.float64).forward(
        x.astype(np.float64))
    rel = np.abs(mu.cpu().numpy() - ref_mu).max() / np.abs(ref_mu).max()
    print("%s: bf16 swish forward mu normwise max error %.3g" % (name, rel))
    assert rel < 3e-2


def test_fp32_unfold_and_forward_match_oracle():
    L = _lib()
    lib = L.load()
    c = helpers.workload('tiny')
    O, A, H, B = c['O'], c['A'], c['H'], 4 * c['E']
    rng = np.random.default_rng(2)
    s0 = rng.uniform(0, 1, (B, O)).astype(np.float32)
    acts = rng.uniform(-1, 1, (B, H, A)).astype(np.float32)
    eps = rng.standard_normal((H, B, O)).astype(np.float32)
    pol = _policy(c, precision='fp32')
    traj = pol.model.unfold_sequences(dev(s0), dev(acts), eps=dev(eps))
    tm_o = _oracle(c).model
    want = tm_o.unfold_sequences(s0, acts, eps)
    np.testing.assert_allclose(traj.cpu().numpy(), want, rtol=1e-4, atol=1e-5)
    x = rng.uniform(0, 1, (B, O + A)).astype(np.float32)
    ens = _ensemble(c)
    mu = torch.empty((B, O), dtype=torch.float32, device='cuda')
    var = torch.empty_like(mu)
    L.check(lib.simba_ensemble_forward(ens._ensure_handle(), P(dev(x)), None, B, P(mu), P(var), None, None))
    torch.cuda.synchronize()
    ref_mu, ref_var = swish_ref.MlpEnsemble(c['weights']).forward(x)
    np.testing.assert_allclose(mu.cpu().numpy(), ref_mu, rtol=1e-4, atol=1e-5)
    np.testing.assert_allclose(var.cpu().numpy(), ref_var, rtol=1e-4, atol=1e-6)


# ---- 5: training ---------------------------------------------------------------------------------------------------
# bf16 swish training, pinned at about twice the worst value measured on a B200 (1000 W) over the shapes below with
# dropout 0 and 0.1 (DESIGN.md section 5): one step's loss relative error (measured 1.95e-5) and per-variable
# ||g - g_ref|| / ||g_ref|| (measured 5.9e-3)
BF16_LOSS_REL = 4e-5
BF16_GRAD_REL = 1.2e-2


def _trained(n_in, n_out, E, B, L, U, precision='fp32', rate=0.0, lr=1e-3, steps=5000, seed=7):
    from simba_b200.models import MlpEnsemble
    ens = MlpEnsemble(n_in, n_out, E, batch_size=B, learning_rate=lr, learning_rate_schedule=False,
                      training_steps=steps, mlp_params=dict(n_layers=L, units=U, dropout_rate=rate,
                                                            activation=SWISH),
                      seed=seed, train_precision=precision)
    ora = swish_ref.EnsembleTrainer([m.get_weights() for m in ens.ensemble], batch_size=B, learning_rate=lr,
                            learning_rate_schedule=False, training_steps=steps, dropout_rate=rate,
                            dropout_seed=seed)
    return ens, ora


def _data(rng, E, B, n_in, n_out):
    return (rng.uniform(0, 1, (E, B, n_in)).astype(np.float32),
            rng.normal(0, 0.1, (E, B, n_out)).astype(np.float32))


def _rel(got, ref):
    ref = np.asarray(ref, np.float64)
    return float(np.linalg.norm(np.asarray(got, np.float64) - ref) / max(np.linalg.norm(ref), 1e-30))


@pytest.mark.parametrize("shape", [(62, 60, 5, 64, 4, 128), (12, 10, 3, 16, 2, 40), (9, 7, 1, 5, 2, 130)])
@pytest.mark.parametrize("rate", [0.0, 0.1])
def test_fp32_step_matches_oracle(shape, rate):
    n_in, n_out, E, B, L, U = shape
    ens, ora = _trained(n_in, n_out, E, B, L, U, rate=rate)
    rng = np.random.default_rng(1)
    n_var = 2 * L + 4
    for _ in range(2):
        x, y = _data(rng, E, B, n_in, n_out)
        loss, want = float(ens.training_step(x, y)), float(ora.training_step(x, y))
        assert loss == pytest.approx(want, rel=1e-4)
        for e in range(E):
            for got, ref in zip(ens.trainer_arrays('grads', e), ora.last_grads[e * n_var:(e + 1) * n_var]):
                np.testing.assert_allclose(got, ref, rtol=1e-4, atol=1e-7)
            for got, ref in zip(ens.trainer_arrays('m', e), ora.optimizer.m[e * n_var:(e + 1) * n_var]):
                np.testing.assert_allclose(got, ref, rtol=1e-4, atol=1e-8)
    for e in range(E):
        for got, ref in zip(ens.trainer_arrays('weights', e), ora.nets[e].arrays):
            np.testing.assert_allclose(got, ref, rtol=1e-4, atol=ens.learning_rate * 0.04)


@pytest.mark.parametrize("shape", [(62, 60, 5, 64, 4, 128), (12, 10, 3, 16, 2, 40), (62, 60, 2, 32, 2, 400)])
@pytest.mark.parametrize("rate", [0.0, 0.1])
def test_bf16_step_within_pinned_bounds(shape, rate):
    n_in, n_out, E, B, L, U = shape
    ens, ora = _trained(n_in, n_out, E, B, L, U, precision='bf16', rate=rate, lr=0.00025)
    rng = np.random.default_rng(1)
    n_var = 2 * L + 4
    x, y = _data(rng, E, B, n_in, n_out)
    loss, want = float(ens.training_step(x, y)), float(ora.training_step(x, y))
    g_err = max(_rel(g, r) for e in range(E)
                for g, r in zip(ens.trainer_arrays('grads', e), ora.last_grads[e * n_var:(e + 1) * n_var]))
    print("bf16 swish step %s rate %.1f: loss rel %.3g, grad rel max %.3g"
          % (shape, rate, abs(loss - want) / abs(want), g_err))
    assert abs(loss - want) <= BF16_LOSS_REL * abs(want)
    assert g_err <= BF16_GRAD_REL
    for e in range(E):
        for got, ref in zip(ens.trainer_arrays('weights', e), ora.nets[e].arrays):
            assert np.abs(got - ref).max() <= 2 * ens.learning_rate * (1 + 1e-3)


def test_validation_step_matches_oracle():
    ens, ora = _trained(12, 10, 3, 16, 2, 40)
    rng = np.random.default_rng(4)
    x = rng.uniform(0, 1, (100, 12)).astype(np.float32)
    y = rng.normal(0, 0.1, (100, 10)).astype(np.float32)
    assert float(ens.validation_step(x, y)) == pytest.approx(float(ora.validation_step(x, y)), rel=1e-4)


@pytest.mark.parametrize("precision", ['fp32', 'bf16'])
def test_fit_lowers_the_loss_and_equals_the_same_batches_one_step_at_a_time(precision):
    n_in, n_out, E, B, L, U = 12, 10, 3, 16, 2, 40
    rng = np.random.default_rng(3)
    x = rng.uniform(-1, 1, (400, n_in)).astype(np.float32)
    y = (0.3 * np.tanh(x[:, :n_out]) + 0.1 * x[:, 1:n_out + 1] * x[:, :1]).astype(np.float32)
    fitted, _ = _trained(n_in, n_out, E, B, L, U, precision, steps=2000, seed=4)
    fitted.validation_split = 0.0
    np.random.seed(11)
    losses = fitted.fit(x, y)
    first, last = float(np.mean(losses[:100])), float(np.mean(losses[-100:]))
    print("%s swish fit: mean loss of the first 100 steps %.4f, of the last 100 %.4f" % (precision, first, last))
    assert last < first - 0.2
    # the first 30 steps of the same schedule, fed one step at a time
    short, _ = _trained(n_in, n_out, E, B, L, U, precision, steps=30, seed=4)
    stepped, _ = _trained(n_in, n_out, E, B, L, U, precision, steps=30, seed=4)
    short.validation_split = 0.0
    np.random.seed(11)
    l30 = short.fit(x, y)
    np.random.seed(11)
    train_idx, _ = short._split_indices(400)
    index, rows = short.batch_schedule(400, 30)
    want = [float(stepped.training_step(np.ascontiguousarray(x[train_idx[index[s, :, :rows[s]]]]),
                                        np.ascontiguousarray(y[train_idx[index[s, :, :rows[s]]]])))
            for s in range(30)]
    np.testing.assert_array_equal(l30.astype(np.float32), np.array(want, np.float32))


def test_trained_weights_reach_the_planner():
    L = _lib()
    c = helpers.workload('tiny')
    pol = _policy(c, precision='fp32')
    acts, eps = _draws(c)
    before, _, _ = _rows(pol, dict(c, S=1), acts, eps)
    ens = pol.model.model
    rng = np.random.default_rng(8)
    x = rng.uniform(0, 1, (ens.ensemble_size, ens.batch_size, c['O'] + c['A'])).astype(np.float32)
    y = rng.normal(0, 0.1, (ens.ensemble_size, ens.batch_size, c['O'])).astype(np.float32)
    for _ in range(5):
        ens.training_step(x, y)
    ens._ensure_handle()                                   # the trainer's weights -> the model handle
    after, _, _ = _rows(pol, dict(c, S=1), acts, eps)
    assert not np.array_equal(before, after)
    _, cum0, _, _ = _oracle_rows(c, _oracle(dict(c, weights=[m.get_weights() for m in ens.ensemble])), acts, eps,
                                 'penalty')
    np.testing.assert_allclose(after, cum0, rtol=1e-4, atol=1e-5)
    assert L.ACT_SWISH == ens.activation


# ---- 6: the boundary -----------------------------------------------------------------------------------------------
def test_set_activation_after_commit_or_unknown_is_rejected():
    L = _lib()
    lib = L.load()
    c = helpers.workload('tiny')
    ens = _ensemble(c, 'tf.nn.relu')
    h = ens._ensure_handle()
    assert lib.simba_model_set_activation(h, L.ACT_SWISH) == -1           # committed already
    cfg = L.ModelConfig(c['O'], c['A'], c['E'], c['L'], c['U'])
    m = C.c_void_p()
    L.check(lib.simba_model_create(C.byref(cfg), C.byref(m)))
    try:
        assert lib.simba_model_set_activation(m, 2) == -1
        assert lib.simba_model_set_activation(m, -1) == -1
        assert lib.simba_model_set_activation(m, L.ACT_SWISH) == 0
        assert lib.simba_model_set_activation(m, L.ACT_RELU) == 0          # until the first commit
    finally:
        lib.simba_model_destroy(m)
