"""bf16 trajectories on the planner's tensor-core kernels: simba_unfold_tc and
TransitionModel.unfold_sequences / simulate_trajectories / predict with precision='bf16'.

  1  kernel choice per shape, the shapes no tcgen05 kernel covers (-6, fp32 still runs them), B % E != 0 (-2)
  2  trajectories against the oracle's unfold on external draws, both propagation modes: s_0 bit for bit, a canary
     beyond the output untouched, per-step max / mean |ds| within the bounds measured on a B200
  3  the trajectories are the planner's: scored by simba_score_trajectories they give the (return, cost) pairs of
     that bf16 planner's simba_rollout_score -> simba_score_reduce on the same actions, seed and iteration, bit for bit
  4  the kernels' own Philox noise against oracle/philox.py's counter contract, with wrong-counter controls
  5  the Python surface
"""
import ctypes as C

import numpy as np
import pytest

from oracle import philox
from tests import helpers
from tests.test_gpu_dispatch_variants import NOISE_BOUNDS, SEED64
from tests.test_gpu_kernels import P, dev
from tests.test_gpu_tc_obs_wide import ROBOT, SCORERS, SENSORS

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")

SENSORS_47 = dict(ROBOT, goal_lidar=16, hazards_lidar=16, aux=3)      # O = 47: a_t at dims 47, 48 straddles 48


def _lib():
    from simba_b200 import _lib
    return _lib


def _model(c, sampling=True):
    """TransitionModel with c's weights and scaler, committed to the device."""
    tm = helpers.cuda_policy(c, sampling_propagation=sampling).model
    tm.model._ensure_handle()
    return tm


def _kernel(tm, B, H):
    """simba_unfold_tc_kernel -> (return code, kernel, work items)."""
    k, items = C.c_int32(-1), C.c_int32(-1)
    rc = _lib().load().simba_unfold_tc_kernel(tm.model._ensure_handle(), B, H, C.byref(k), C.byref(items))
    return rc, k.value, items.value


def _sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


# ---- 1: kernel choice ----------------------------------------------------------------------------------------
@pytest.mark.parametrize("B", [3000, 5 * 128 * 40, 10 ** 6])
def test_c1_dims_choose_one_cta_or_two_tile_by_tile_count(B):
    L = _lib()
    tm = _model(helpers.workload('c1'))
    tiles = 5 * -(-(B // 5) // 128)                          # 128-row tiles of the tf.split member map
    rc, k, items = _kernel(tm, B, 15)
    assert rc == 0
    if tiles > _sms():
        assert k == L.ROLLOUT_TC_TWO_TILE and tiles // 2 <= items <= tiles
    else:
        assert (k, items) == (L.ROLLOUT_TC_ONE_CTA, tiles)


@pytest.mark.parametrize("cfg,sensors,kernel", [
    ('c5', None, 'TC_WIDE'), ('tiny', 76, 'TC_WIDE_OBS'), ('tiny', 92, 'TC_WIDE_OBS'), ('tiny', 124, 'TC_WIDE_OBS'),
    ('c1', 92, 'TC_WIDE_OBS')])
def test_wide_shapes_choose_the_streaming_kernels(cfg, sensors, kernel):
    L = _lib()
    c = helpers.workload(cfg, sensors=SENSORS[sensors] if sensors else None)
    tm = _model(c)
    B = c['E'] * 300
    rc, k, items = _kernel(tm, B, c['H'])
    assert (rc, k) == (0, getattr(L, 'ROLLOUT_' + kernel))
    assert items == c['E'] * -(-300 // 128)
    assert _kernel(tm, B, 200)[:2] == (0, k)                  # no cost mask: horizons beyond 64 run


@pytest.mark.parametrize("sensors,over", [(None, dict(U=432)), (92, dict(U=400, L=2))])
def test_uncovered_shapes_are_rejected_and_fp32_still_runs_them(sensors, over):
    L = _lib()
    c = helpers.workload('tiny', sensors=SENSORS[sensors] if sensors else None, **over)
    tm = _model(c)
    B = c['E'] * 16
    assert _kernel(tm, B, c['H'])[0] == -6
    rng = np.random.default_rng(0)
    s0 = np.tile(c['state'], (B, 1)).astype(np.float32)
    acts = rng.uniform(-1, 1, (B, c['H'], c['A'])).astype(np.float32)
    with pytest.raises(L.SimbaError) as e:
        tm.unfold_sequences(s0, acts, precision='bf16')
    assert e.value.code == -6 and 'fp32' in str(e.value)
    assert np.all(np.isfinite(tm.unfold_sequences(s0, acts)))


def test_batch_not_divisible_by_ensemble_and_bad_horizon():
    L = _lib()
    c = helpers.workload('c1')
    tm = _model(c)
    assert _kernel(tm, 3001, 15)[0] == -2
    assert _kernel(tm, 3000, 0)[0] == -1 and _kernel(tm, 3000, 65536)[0] == -1
    rng = np.random.default_rng(0)
    with pytest.raises(L.SimbaError) as e:
        tm.unfold_sequences(np.tile(c['state'], (3001, 1)), rng.uniform(-1, 1, (3001, 15, c['A'])).astype(np.float32),
                            precision='bf16')
    assert e.value.code == -2


# ---- 2: against the oracle -------------------------------------------------------------------------------------
# name: (workload, sensors, overrides, batch per member)
ORACLE = {
    'tiny': ('tiny', None, dict(), 64),
    'c1': ('c1', None, dict(), 64),
    'c5-reduced': ('c5', None, dict(H=20), 32),
    'o61': ('tiny', 61, dict(), 64),
    'o63-actions-straddle-64': ('tiny', 63, dict(), 64),
    'o76': ('tiny', 76, dict(), 64),
    'o92': ('tiny', 92, dict(L=4), 64),
    'o124': ('tiny', 124, dict(), 64),
    'goal-dist-67': ('tiny', 'goal_dist', dict(), 64),
    'a1': ('tiny', None, dict(A=1), 64),
    'a3': ('tiny', 61, dict(A=3), 64),
    'a4': ('tiny', None, dict(A=4), 64),
    'o47-a2-actions-straddle-48': ('tiny', 47, dict(), 64),
    'o47-a2-u256': ('tiny', 47, dict(U=256), 64),
    'L1': ('tiny', None, dict(L=1), 64),
    'L6': ('tiny', 92, dict(L=6), 64),
    'u64': ('tiny', None, dict(U=64), 64),
    'u200': ('tiny', None, dict(U=200, L=3), 64),
    'u384': ('tiny', None, dict(U=384, L=2), 64),
    'b-not-multiple-of-128': ('tiny', None, dict(), 37),
    'two-tile': ('tiny', None, dict(E=4, H=3), 40 * 128 + 17),
    'h100': ('tiny', None, dict(H=100), 16),
}
# Bounds on |bf16 - oracle| per step, over rows and dims: at the first step and at every step of the horizon
# (H <= 20, and H = 100). Measured on a B200 (148 SMs, 1000 W) with var-head bias -5 (sigma ~0.08 per step), both
# propagation modes, every case above: step 1 max 2.9e-3, mean 1.5e-4; any step up to H = 20 max 3.8e-3, mean 7.0e-4;
# any step up to H = 100 max 3.4e-2, mean 6.0e-3. Pinned about 2x above (DESIGN.md section 5).
STEP1_MAX, STEP1_MEAN = 6e-3, 3e-4
ANY_STEP_MAX = {20: (8e-3, 1.5e-3), 100: (7e-2, 1.2e-2)}


def _oracle_case(name, sampling):
    cfg, sensors, over, per_member = ORACLE[name]
    sens = SENSORS_47 if sensors == 47 else (SENSORS[sensors] if sensors is not None else None)
    c = helpers.workload(cfg, sensors=sens, var_bias=-5.0, **over)
    B = c['E'] * per_member
    rng = np.random.default_rng(11)
    s0 = (np.tile(c['state'], (B, 1)) + rng.normal(0, 0.01, (B, c['O']))).astype(np.float32)
    acts = rng.uniform(-1, 1, (B, c['H'], c['A'])).astype(np.float32)
    eps = rng.standard_normal((c['H'], B, c['O'])).astype(np.float32)
    return c, B, s0, acts, eps


@pytest.mark.parametrize("sampling", [True, False])
@pytest.mark.parametrize("name", list(ORACLE))
def test_trajectories_close_to_oracle(name, sampling):
    L = _lib()
    c, B, s0, acts, eps = _oracle_case(name, sampling)
    H, O = c['H'], c['O']
    tm = _model(c, sampling)
    rc, kernel, _ = _kernel(tm, B, H)
    assert rc == 0
    n = B * (H + 1) * O
    canary = 4096
    out = torch.full((n + canary,), 12345.0, dtype=torch.float32, device='cuda')
    d_s0, d_acts, d_eps = dev(s0), dev(acts), dev(eps)
    L.check(L.load().simba_unfold_tc(tm.model._ensure_handle(), P(d_s0), P(d_acts), P(d_eps), 0, B, H,
                                     int(sampling), P(out), None))
    torch.cuda.synchronize()
    host = out.cpu().numpy()
    assert np.all(host[n:] == 12345.0)
    traj = host[:n].reshape(B, H + 1, O)
    assert np.array_equal(traj[:, 0].view(np.uint32), s0.view(np.uint32))
    ref = helpers.oracle_planner(c, sampling_propagation=sampling).model.unfold_sequences(s0, acts, eps)
    d = np.abs(traj.astype(np.float64) - ref)
    mx, mean = d.max(axis=(0, 2)), d.mean(axis=(0, 2))
    print("%s sampling=%d kernel %d B=%d H=%d: step 1 max %.3g mean %.3g; horizon max %.3g mean %.3g (last step)"
          % (name, sampling, kernel, B, H, mx[1], mean[1], mx.max(), mean[-1]))
    assert np.all(np.isfinite(traj))
    assert mx[1] <= STEP1_MAX and mean[1] <= STEP1_MEAN
    any_max, any_mean = ANY_STEP_MAX[20 if H <= 20 else 100]
    assert mx.max() <= any_max and mean.max() <= any_mean


# ---- 3: these are the planner's trajectories --------------------------------------------------------------------
@pytest.mark.parametrize("cfg,sensors,scorer", [('c1', None, None), ('c5', None, None), ('c1', 92, 'goal4')])
@pytest.mark.parametrize("seed", [7, SEED64])
def test_scored_trajectories_equal_the_planners_rollout_scores(cfg, sensors, scorer, seed):
    L = _lib()
    lib = L.load()
    c = helpers.workload(cfg, sensors=SENSORS[sensors] if sensors else None)
    pol = helpers.cuda_policy(c, 'penalty', precision='bf16', scorer_config=SCORERS.get(scorer))
    pl = pol._ensure_planner()
    H, A, N, P_, O = c['H'], c['A'], c['N'], c['P'], c['O']
    B = P_ * N
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
    # the same rows for the model: particle-major, row p * N + i = candidate i, the state broadcast
    acts_b = acts[0].repeat(P_, 1, 1).contiguous()
    s0 = d_state.expand(B, O).contiguous()
    traj = pol.model.unfold_sequences(s0, acts_b, seed=seed, precision='bf16')
    assert tuple(traj.shape) == (B, H + 1, O)
    scores = torch.empty((N,), dtype=torch.float32, device='cuda')
    pairs = torch.empty((N, 2), dtype=torch.float32, device='cuda')
    L.check(lib.simba_score_trajectories(pl, P(traj), P(scores), P(pairs), None))
    torch.cuda.synchronize()
    got, want = pairs.cpu().numpy(), pairs_plan[0].cpu().numpy()
    print("%s obs %d seed %d: %d of %d pairs identical, returns in [%.3f, %.3f], costs in [%g, %g]"
          % (cfg, O, seed, (got == want).all(axis=1).sum(), N, want[:, 0].min(), want[:, 0].max(),
             want[:, 1].min(), want[:, 1].max()))
    assert np.array_equal(got.view(np.uint32), want.view(np.uint32))


# ---- 4: the kernels' Philox noise against the counter contract ---------------------------------------------------
def _contract(c, B, seed, it=0, t0=0, rows=None, state=0):
    rows = np.arange(B) if rows is None else rows
    return philox.noise_normals(seed, it, c['H'] + t0, rows, c['O'], state_index=state)[t0:].astype(np.float32)


@pytest.mark.parametrize("cfg,sensors,scorer", [('tiny', None, None), ('c5', None, None), ('tiny', 92, 'goal4')])
def test_device_noise_follows_the_philox_contract(cfg, sensors, scorer):
    L = _lib()
    lib = L.load()
    c = helpers.workload(cfg, sensors=SENSORS[sensors] if sensors else None, H=8)
    pol = helpers.cuda_policy(c, 'penalty', precision='bf16', scorer_config=SCORERS.get(scorer))
    pl = pol._ensure_planner()
    N, P_, H, A = c['N'], c['P'], c['H'], c['A']
    B = P_ * N
    rng = np.random.default_rng(31)
    acts = np.tile(rng.uniform(-1, 1, (N, H, A)).astype(np.float32), (P_, 1, 1))
    s0 = np.tile(np.asarray(c['state'], np.float32).reshape(1, -1), (B, 1))

    def pairs(eps=None, seed=SEED64):
        traj = pol.model.unfold_sequences(dev(s0), dev(acts), eps=None if eps is None else dev(eps), seed=seed,
                                          precision='bf16')
        out = torch.empty((N, 2), dtype=torch.float32, device='cuda')
        sc = torch.empty((N,), dtype=torch.float32, device='cuda')
        L.check(lib.simba_score_trajectories(pl, P(traj), P(sc), P(out), None))
        torch.cuda.synchronize()
        return out.cpu().numpy()

    device = pairs()

    def compare(eps):
        got = pairs(eps)
        return np.abs(got[:, 0] - device[:, 0]).mean(), (got[:, 1] == device[:, 1]).mean()

    good = compare(_contract(c, B, SEED64))
    print("%s obs %d: contract mean|dret| %.3g, costs identical %.4f" % (cfg, c['O'], *good))
    assert np.all(np.isfinite(device))
    assert good[0] <= NOISE_BOUNDS['mean_dret'] and good[1] >= NOISE_BOUNDS['csum_same']
    r = np.arange(B)
    controls = {
        'iteration+1': lambda: _contract(c, B, SEED64, it=1),
        'other state': lambda: _contract(c, B, SEED64, state=1),
        't+1': lambda: _contract(c, B, SEED64, t0=1),
        'rows candidate-major': lambda: _contract(c, B, SEED64, rows=(r % N) * P_ + r // N),
        'rows shifted': lambda: _contract(c, B, SEED64, rows=r + 1),
        'seed high word dropped': lambda: _contract(c, B, SEED64 & 0xFFFFFFFF),
    }
    for name, make in controls.items():
        bad = compare(make())
        print("  control %-22s mean|dret| %.3g  ratio %.3g" % (name, bad[0], bad[0] / max(good[0], 1e-12)))
        assert bad[0] >= 10 * good[0] and bad[0] > 0, name


# ---- 5: the Python surface ---------------------------------------------------------------------------------------
def test_python_surface():
    c = helpers.workload('c1')
    tm = _model(c)
    rng = np.random.default_rng(3)
    B = c['E'] * 200
    x = np.concatenate([np.tile(c['state'], (B, 1)), rng.uniform(-1, 1, (B, c['A']))], axis=1).astype(np.float32)
    pred = tm.predict(x, precision='bf16')
    assert isinstance(pred, np.ndarray) and pred.shape == (B, 2, c['O'])
    assert np.array_equal(pred[:, 0], x[:, :c['O']])
    fp32 = tm.predict(x)
    assert np.array_equal(fp32.view(np.uint32), tm.predict(x, precision='fp32').view(np.uint32))
    assert 0 < np.abs(pred - fp32).max() < 5e-2
    acts = rng.uniform(-1, 1, (B, 4, c['A'])).astype(np.float32)
    sim = tm.simulate_trajectories(x[:, :c['O']], acts, seed=3, precision='bf16')
    assert sim.shape == (B, 5, c['O'])
    with pytest.raises(ValueError):
        tm.predict(x, precision='fp16')
    with pytest.raises(ValueError):
        tm.unfold_sequences(x[:, :c['O']], acts, precision='bf16x')
    with pytest.raises(TypeError):
        tm.unfold_sequences(x[:, :c['O']], acts, None, 0, 'bf16')      # keyword-only
