"""MPPI planning (simba_planner_set_update_rule(SIMBA_UPDATE_MPPI), MppiMpc / SafeMppiMpc) against the numpy oracle
of oracle/mppi_oracle.py, on external and Philox draws, on the fused and the separate update kernels."""
import os

import numpy as np
import pytest

from oracle import mppi_oracle, philox
from oracle import simba_oracle as so
from tests import helpers

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")

TEMPERATURE = 0.5

# bf16 rollouts against fp32 ones, same external draws, penalty objective, temperature 0.5: max |d mu| (BUF_MU after
# the plan), max |d action| and |d score|. Measured on one B200 at a 1000 W power limit by tools/mppi_bench.py
# (profiles/r10_mppi_bench.json, "bf16_errors"); the bounds are twice the measured values. At C1 a bf16 score moves
# by up to 7e-4, which at temperature 0.5 reweights the candidates enough to move mu by 0.07.
BF16_BOUNDS = {
    'c1': (0.141, 0.141, 0.0014),        # measured 0.0705, 0.0705, 0.00069
    'c5': (0.003, 0.00054, 0.00048),     # measured 0.00149, 0.00027, 0.00024
}


def _policy(c, objective='reward', **kw):
    kw.setdefault('temperature', TEMPERATURE)
    kw.setdefault('precision', 'fp32')
    return helpers.cuda_policy(c, objective, **kw)


def _oracle(c, objective='reward', temperature=TEMPERATURE, smoothing=0.0, member_map='split'):
    ens = so.MlpEnsemble(c['weights'])
    tm = so.TransitionModel(ens, c['smin'], c['smax'], True, True)
    env = so.Environment(so.Scorer(None, c['table']), so.Box([-1.0] * c['A'], [1.0] * c['A']), None)
    return mppi_oracle.MppiPlanner(tm, env, c['H'], c['I'], smoothing, c['N'], c['P'], 0.01, temperature,
                                   posterior_mean_threashold=0.15, objective=helpers.OBJ[objective],
                                   member_map=member_map)


def _plan_external(c, objective, smoothing=0.0, member_map='split', precision='fp32'):
    from simba_b200 import _lib, synthetic
    z, eps, zf = synthetic.make_draws(c['I'], c['S'], c['N'], c['H'], c['A'], c['P'], c['O'])
    pol = _policy(c, objective, smoothing=smoothing, member_map=member_map, precision=precision)
    pol.set_external_draws(z, eps, zf)
    action, score = pol.do_generate_action(c['state'])
    mu = pol.buffer(_lib.BUF_MU).cpu().numpy().reshape(c['S'], c['H'], c['A'])
    return pol, (z, eps, zf), (np.asarray(action), np.asarray(score), mu)


def _check_against_oracle(c, objective, draws, got, smoothing=0.0, member_map='split'):
    z, eps, zf = draws
    action, score, mu = got
    tr = so.Trace()
    a0, s0, n0 = _oracle(c, objective, smoothing=smoothing, member_map=member_map).do_generate_action(
        c['state'], z, eps, zf, tr)
    assert np.allclose(mu[0], tr[-1]['mu'], rtol=1e-4, atol=1e-5), np.abs(mu[0] - tr[-1]['mu']).max()
    assert np.allclose(action, a0, rtol=1e-4, atol=1e-5)
    assert np.isclose(score, s0, rtol=1e-4, atol=1e-5)
    return n0


@pytest.mark.parametrize("cfg,objective", [('tiny', 'reward'), ('tiny', 'penalty'), ('tiny', 'least_cost'),
                                           ('c1', 'reward'), ('c1', 'penalty'), ('c1', 'least_cost')])
def test_plan_matches_oracle_fp32(cfg, objective):
    c = helpers.workload(cfg)
    pol, draws, got = _plan_external(c, objective)
    n0 = _check_against_oracle(c, objective, (draws[0][:, 0], draws[1][:, 0], draws[2][0]), got)
    assert int(pol.iterations_run[0]) == n0 == c['I']                     # no early exit


def test_plan_smoothing_and_member_map_particle():
    c = helpers.workload('tiny', E=3)
    pol, draws, got = _plan_external(c, 'penalty', smoothing=0.5, member_map='particle')
    _check_against_oracle(c, 'penalty', (draws[0][:, 0], draws[1][:, 0], draws[2][0]), got, smoothing=0.5,
                          member_map='particle')


def test_plan_philox_mode_matches_oracle_fed_with_contract_normals():
    c = helpers.workload('tiny')
    seed = 0x5EED
    pol = _policy(c, 'penalty')
    action, score = pol.do_generate_action(c['state'], seed=seed)
    B = c['P'] * c['N']
    z = np.stack([philox.action_normals(seed, it, c['N'], c['H'], c['A']) for it in range(c['I'])])
    eps = np.stack([philox.noise_normals(seed, it, c['H'], np.arange(B), c['O']) for it in range(c['I'])])
    zf = philox.final_normals(seed, c['A'])
    a0, s0, _ = _oracle(c, 'penalty').do_generate_action(c['state'], z, eps, zf)
    assert np.allclose(action, a0, rtol=1e-4, atol=1e-5) and np.isclose(score, s0, rtol=1e-4, atol=1e-5)
    a1, _ = pol.do_generate_action(c['state'], seed=seed)
    a2, _ = pol.do_generate_action(c['state'], seed=seed + 1)
    assert np.array_equal(a1, action) and not np.array_equal(a2, action)


@pytest.mark.parametrize("N", [4096, 65536])
def test_large_populations_on_the_separate_update_match_oracle(N):
    """N > 1024 runs score_reduce + mppi_refit; at N = 65536 the refit is a cluster of eight CTAs."""
    c = helpers.workload('tiny', N=N, P=2, I=2)
    pol, draws, got = _plan_external(c, 'reward')
    assert pol.launches_per_plan == 1 + 4 * c['I'] + 2
    _check_against_oracle(c, 'reward', (draws[0][:, 0], draws[1][:, 0], draws[2][0]), got)


def _update_once(N, S=2, H=6, A=2, objective='reward', nan_every=0, all_nan_state=False, seed=0):
    """simba_mppi_update on random pairs and actions -> (inputs, outputs)."""
    from simba_b200 import _lib
    c = helpers.workload('tiny', N=N, S=S, H=H, P=2)
    pol = _policy(c, objective)
    lib = _lib.load()
    rng = np.random.default_rng(seed)
    pairs = np.stack([rng.normal(0.0, 1.0, (S, N)), rng.integers(0, 3, (S, N))], -1).astype(np.float32)
    if nan_every:
        pairs[:, ::nan_every, 0] = np.nan
    if all_nan_state:
        pairs[0, :, 0] = np.nan
    acts = rng.uniform(-1.0, 1.0, (S, N, H, A)).astype(np.float32)
    mu = rng.uniform(-0.5, 0.5, (S, H, A)).astype(np.float32)
    best_a = np.zeros((S, A), np.float32)
    best_s = np.full((S,), -np.inf, np.float32)
    dev = [torch.from_numpy(x).cuda() for x in (pairs, acts, mu, best_a, best_s)]
    _lib.check(lib.simba_mppi_update(pol._ensure_planner(), dev[0].data_ptr(), dev[1].data_ptr(), None,
                                     dev[2].data_ptr(), dev[3].data_ptr(), dev[4].data_ptr(), None))
    torch.cuda.synchronize()
    return pol, (pairs, acts, mu), [x.cpu().numpy() for x in dev[2:]]


@pytest.mark.parametrize("N,nan_every", [(24, 0), (1000, 7), (4096, 5), (65536, 3)])
def test_mppi_update_entry_point_matches_oracle(N, nan_every):
    pol, (pairs, acts, mu), (mu_d, best_a, best_s) = _update_once(N, nan_every=nan_every)
    for s in range(pairs.shape[0]):
        scores = pairs[s, :, 0]
        want = mppi_oracle.mppi_update(mu[s], scores, acts[s], TEMPERATURE, 0.0)
        assert np.allclose(mu_d[s], want, rtol=1e-5, atol=1e-6), np.abs(mu_d[s] - want).max()
        if nan_every:                                  # a NaN score weighs 0: the same as leaving the candidate out
            keep = ~np.isnan(scores)
            assert np.allclose(mu_d[s], mppi_oracle.mppi_update(mu[s], scores[keep], acts[s][keep], TEMPERATURE, 0.0),
                               rtol=1e-5, atol=1e-6)
        top = mppi_oracle.best_candidate(scores)
        assert best_s[s] == scores[top] and np.array_equal(best_a[s], acts[s, top, 0])


def test_mppi_update_all_nan_scores_leave_mu_unchanged():
    pol, (pairs, acts, mu), (mu_d, best_a, best_s) = _update_once(64, all_nan_state=True)
    assert np.array_equal(mu_d[0], mu[0]) and best_s[0] == -np.inf and np.all(best_a[0] == 0)
    assert not np.array_equal(mu_d[1], mu[1]) and np.isfinite(best_s[1])


@pytest.mark.parametrize("case", ['c1-fp32', 'c1-bf16', 'penalty', 'least_cost', 'states', 'unstaged', 'ragged'])
def test_fused_update_is_bit_identical_to_separate_kernels(case):
    from simba_b200 import _lib
    precision, objective, cfg, over = 'fp32', 'penalty', 'c1', {}
    if case == 'c1-bf16':
        precision = 'bf16'
    elif case in ('penalty', 'least_cost'):
        cfg, objective = 'tiny', case
    elif case == 'states':
        over = dict(S=3)
    elif case == 'unstaged':
        cfg, over = 'tiny', dict(N=1000, P=16, H=6, I=3)      # 16000 rows do not fit: rows read from global memory
    elif case == 'ragged':
        cfg, over = 'tiny', dict(N=149, P=7, H=5, I=3, E=1)
    c = helpers.workload(cfg, **over)
    res = []
    for no_fuse in (False, True):
        if no_fuse:
            os.environ['SIMBA_B200_NO_FUSE'] = '1'
        try:
            pol = _policy(c, objective, precision=precision, smoothing=0.25)
            a, s = pol.do_generate_action(c['state'], seed=123)
            res.append((np.asarray(a), np.asarray(s), pol.buffer(_lib.BUF_MU).cpu().numpy(),
                        pol.buffer(_lib.BUF_BEST_ACTION).cpu().numpy(), np.asarray(pol.iterations_run).copy(),
                        pol.launches_per_plan))
        finally:
            os.environ.pop('SIMBA_B200_NO_FUSE', None)
    f, u = res
    assert f[5] == 1 + 2 * c['I'] and u[5] == 1 + 4 * c['I'] + 2
    for x, y in zip(f[:5], u[:5]):
        assert np.array_equal(x, y)
    assert np.all(f[4] == c['I'])


def test_batched_plan_equals_single_state_plans():
    from simba_b200 import _lib, synthetic
    c = helpers.workload('tiny', S=3)
    z, eps, zf = synthetic.make_draws(c['I'], 3, c['N'], c['H'], c['A'], c['P'], c['O'])
    pol = _policy(c, 'penalty')
    pol.set_external_draws(z, eps, zf)
    acts, scores = pol.do_generate_action(c['state'])
    mu = pol.buffer(_lib.BUF_MU).cpu().numpy().reshape(3, -1)
    c1 = dict(c); c1['S'] = 1
    for s in range(3):
        p1 = _policy(c1, 'penalty')
        p1.set_external_draws(np.ascontiguousarray(z[:, s:s + 1]), np.ascontiguousarray(eps[:, s:s + 1]),
                              np.ascontiguousarray(zf[s:s + 1]))
        a, sc = p1.do_generate_action(c['state'][s])
        assert np.array_equal(a, acts[s]) and np.array_equal(sc, scores[s])
        assert np.array_equal(p1.buffer(_lib.BUF_MU).cpu().numpy(), mu[s])


@pytest.mark.parametrize("cfg", list(BF16_BOUNDS))
def test_bf16_against_fp32(cfg):
    c = helpers.workload(cfg)
    got = {p: _plan_external(c, 'penalty', precision=p)[2] for p in ('bf16', 'fp32')}
    d_mu = float(np.abs(got['bf16'][2] - got['fp32'][2]).max())
    d_act = float(np.abs(got['bf16'][0] - got['fp32'][0]).max())
    d_score = float(np.abs(got['bf16'][1] - got['fp32'][1]).max())
    print('bf16 vs fp32 %s: mu %.3g action %.3g score %.3g' % (cfg, d_mu, d_act, d_score))
    b_mu, b_act, b_score = BF16_BOUNDS[cfg]
    assert d_mu <= b_mu and d_act <= b_act and d_score <= b_score


def test_setter_errors():
    from simba_b200 import SimbaError, _lib
    lib = _lib.load()
    c = helpers.workload('tiny')
    cem = helpers.cuda_policy(c, 'reward', precision='fp32')
    h = cem._ensure_planner()
    for rule, temp in ((2, 1.0), (-1, 1.0), (_lib.UPDATE_MPPI, 0.0), (_lib.UPDATE_MPPI, -1.0),
                       (_lib.UPDATE_MPPI, float('inf')), (_lib.UPDATE_MPPI, float('nan'))):
        assert lib.simba_planner_set_update_rule(h, rule, temp) == -1, (rule, temp)
    for temp in (float('nan'), 0.0):                         # CEM ignores the temperature
        assert lib.simba_planner_set_update_rule(h, _lib.UPDATE_CEM, temp) == 0
    # the per-kernel entry point needs an MPPI planner
    assert lib.simba_mppi_update(h, 1, 1, None, 1, 1, 1, None) == -1
    ff = helpers.cuda_policy(c, 'feasible_first', precision='fp32')
    assert lib.simba_planner_set_update_rule(ff._ensure_planner(), _lib.UPDATE_MPPI, 1.0) == -6
    pol = helpers.cuda_policy(c, 'reward', precision='fp32', world_size=2, rank=0, temperature=1.0)
    with pytest.raises(SimbaError) as e:
        pol._ensure_planner()
    assert e.value.code == -6 and pol._planner is None
    pol = _policy(c)
    pol.do_generate_action(c['state'], seed=1)
    for rule in (_lib.UPDATE_CEM, _lib.UPDATE_MPPI):
        assert lib.simba_planner_set_update_rule(pol._planner, rule, 1.0) == -1
    with pytest.raises(ValueError):
        helpers.cuda_policy(c, 'feasible_first', temperature=1.0)   # SafeMppiMpc takes penalty or least_cost only


def test_cem_planner_is_unchanged_by_the_update_rule_setter():
    """A CEM planner: the same launches and bit-identical plans whether the rule is left alone, set to CEM, or set to
    MPPI and back to CEM before the first plan."""
    from simba_b200 import _lib
    lib = _lib.load()
    c = helpers.workload('c1')
    out = []
    for mode in ('default', 'cem', 'mppi-then-cem'):
        pol = helpers.cuda_policy(c, 'penalty', precision='bf16')
        h = pol._ensure_planner()
        if mode != 'default':
            if mode == 'mppi-then-cem':
                _lib.check(lib.simba_planner_set_update_rule(h, _lib.UPDATE_MPPI, 1.0))
            _lib.check(lib.simba_planner_set_update_rule(h, _lib.UPDATE_CEM, 0.0))
        a, s = pol.do_generate_action(c['state'], seed=7)
        out.append((np.asarray(a), np.asarray(s), pol.launches_per_plan,
                    pol.buffer(_lib.BUF_ELITE, torch.int32).cpu().numpy()))
    assert out[0][2] == 1 + 2 * c['I']
    for o in out[1:]:
        assert o[2] == out[0][2]
        assert all(np.array_equal(x, y) for x, y in zip(o[:2] + o[3:], out[0][:2] + out[0][3:]))


class ToyEnv(object):
    """A deterministic environment with the planner's observation layout that ends after 5 + bias steps."""

    def __init__(self, c, seed, episode_bias=0):
        from simba_b200.spaces import Box
        self.c, self.rng, self.bias, self.t, self.obs = c, np.random.default_rng(seed), episode_bias, 0, None
        self.action_space = Box([-1.0] * c['A'], [1.0] * c['A'])

    def reset(self):
        from simba_b200 import synthetic
        self.t = 0
        self.obs = synthetic.make_state(self.c['sensors'], seed=int(self.rng.integers(1 << 30)))
        return self.obs.copy()

    def step(self, action):
        self.t += 1
        self.obs = np.clip(self.obs + 0.01 * float(np.sum(action)), 0.0, 1.0).astype(np.float32)
        return self.obs.copy(), float(action[0]), self.t >= 5 + self.bias, dict(cost=float(action[0] > 0.5))


def test_mppi_drives_the_vectorized_agent_loop():
    from simba_b200 import agents
    c = helpers.workload('tiny', S=8)
    pol = _policy(c, 'penalty', precision='bf16', seed=3, n_states=8)
    envs = [ToyEnv(c, seed=20 + i, episode_bias=i % 4) for i in range(8)]
    paths, steps = agents.sample_trajectories_vectorized(envs, pol, 60, 50, action_repeat=1)
    assert steps >= 60 and steps == sum(len(p['reward']) for p in paths)
    for p in paths:
        assert p['action'].shape[1] == c['A'] and np.all(np.isfinite(p['action']))
    assert np.all(pol.iterations_run == c['I'])
