"""The ensemble's forward pass on the planner's bf16 tensor-core kernels: simba_ensemble_forward_tc and
MlpEnsemble.forward / __call__ with precision='bf16'.

  1  kernel choice = simba_unfold_tc_kernel at H = 1, uncovered shapes (-6, fp32 still runs them), argument errors
  2  bit-identities with the bf16 planner's arithmetic, every form: simba_unfold_tc at H = 1 gives
     s_1 == float32(s_0 + mu) in mean propagation, and s_1 == sample from s_0 = 0 with external draws
  3  mu and var against the numpy oracle and the fp32 kernel, within bounds measured on a B200; the reference fixture
  4  nothing written beyond [B, O], two calls bit-identical, a bf16 planner plans the same before and after
  5  the Python surface
"""
import ctypes as C

import numpy as np
import pytest

from oracle import simba_oracle as so
from tests import helpers
from tests.test_gpu_kernels import P, dev
from tests.test_gpu_tc_obs_wide import SENSORS
from tests.test_gpu_unfold_tc import SENSORS_47

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")


def _lib():
    from simba_b200 import _lib
    return _lib


def _ensemble(c):
    """MlpEnsemble with c's weights and no scaler (x is used as given either way), committed to the device."""
    from simba_b200.models import MlpEnsemble
    ens = MlpEnsemble(c['O'] + c['A'], c['O'], c['E'], mlp_params=dict(n_layers=c['L'], units=c['U']))
    for e in range(c['E']):
        ens.ensemble[e].set_weights(c['weights'][e])
    ens._ensure_handle()
    return ens


def _kernels(ens, B):
    """(simba_ensemble_forward_tc_kernel, simba_unfold_tc_kernel at H = 1), each (return code, kernel, items)."""
    lib = _lib().load()
    out = []
    for call in (lambda k, i: lib.simba_ensemble_forward_tc_kernel(ens._ensure_handle(), B, k, i),
                 lambda k, i: lib.simba_unfold_tc_kernel(ens._ensure_handle(), B, 1, k, i)):
        k, items = C.c_int32(-1), C.c_int32(-1)
        rc = call(C.byref(k), C.byref(items))
        out.append((rc, k.value, items.value))
    return out


def _forward(ens, x, eps=None, precision='bf16'):
    """simba_ensemble_forward(_tc) on device tensors -> (rc, mu, var, sample or None)."""
    L = _lib()
    lib = L.load()
    B, O = x.shape[0], ens.outputs_dim
    mu = torch.empty((B, O), dtype=torch.float32, device='cuda')
    var = torch.empty_like(mu)
    smp = torch.empty_like(mu) if eps is not None else None
    fn = lib.simba_ensemble_forward_tc if precision == 'bf16' else lib.simba_ensemble_forward
    rc = fn(ens._ensure_handle(), P(x), P(eps), B, P(mu), P(var), P(smp), None)
    torch.cuda.synchronize()
    return rc, mu, var, smp


def _sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


# name: (workload, sensors, overrides, rows per member, kernel)
CASES = {
    'c1-one-cta': ('c1', None, dict(), 600, 'TC_ONE_CTA'),
    'c1-two-tile-over-one-wave': ('c1', None, dict(), 60 * 128 + 5, 'TC_TWO_TILE'),
    'c5-wide': ('c5', None, dict(), 300, 'TC_WIDE'),
    'c1-o92-wide-obs-over-one-wave': ('c1', 92, dict(), 31 * 128 + 17, 'TC_WIDE_OBS'),
    'o47-a2-actions-straddle-48': ('tiny', 47, dict(), 77, 'TC_ONE_CTA'),
    'o47-a2-u256-wide': ('tiny', 47, dict(U=256), 77, 'TC_WIDE'),
    'o63-actions-straddle-64': ('tiny', 63, dict(), 77, 'TC_WIDE_OBS'),
    'b-not-multiple-of-128': ('tiny', None, dict(), 37, 'TC_ONE_CTA'),
}


def _case(name, var_bias=-2.0):
    cfg, sensors, over, per_member, kernel = CASES[name]
    sens = SENSORS_47 if sensors == 47 else (SENSORS[sensors] if sensors is not None else None)
    c = helpers.workload(cfg, sensors=sens, var_bias=var_bias, **over)
    B = c['E'] * per_member
    rng = np.random.default_rng(21)
    x = rng.uniform(0, 1, (B, c['O'] + c['A'])).astype(np.float32)     # scaled inputs lie in [0, 1]
    x[:, c['O']:] = rng.uniform(-1, 1, (B, c['A']))
    eps = rng.standard_normal((B, c['O'])).astype(np.float32)
    return c, B, x, eps, kernel


# ---- 1: kernel choice and errors ---------------------------------------------------------------------------------
@pytest.mark.parametrize("name", list(CASES))
def test_kernel_is_the_unfold_kernel_at_horizon_one(name):
    L = _lib()
    c, B, _, _, kernel = _case(name)
    ens = _ensemble(c)
    fwd, unf = _kernels(ens, B)
    assert fwd == unf and fwd[0] == 0
    assert fwd[1] == getattr(L, 'ROLLOUT_' + kernel)


@pytest.mark.parametrize("B", [3000, 5 * 128 * 40])
def test_c1_dims_choose_one_cta_or_two_tile_by_tile_count(B):
    L = _lib()
    ens = _ensemble(helpers.workload('c1'))
    tiles = 5 * -(-(B // 5) // 128)
    rc, k, items = _kernels(ens, B)[0]
    assert rc == 0
    if tiles > _sms():
        assert k == L.ROLLOUT_TC_TWO_TILE
    else:
        assert (k, items) == (L.ROLLOUT_TC_ONE_CTA, tiles)


@pytest.mark.parametrize("sensors,over", [(None, dict(U=500)), (92, dict(A=5))])
def test_uncovered_shapes_are_rejected_and_fp32_still_runs_them(sensors, over):
    L = _lib()
    c = helpers.workload('tiny', sensors=SENSORS[sensors] if sensors else None, **over)
    ens = _ensemble(c)
    B = c['E'] * 16
    assert _kernels(ens, B)[0][0] == -6
    x = np.random.default_rng(0).uniform(0, 1, (B, c['O'] + c['A'])).astype(np.float32)
    with pytest.raises(L.SimbaError) as e:
        ens.forward(x, precision='bf16')
    assert e.value.code == -6 and 'fp32' in str(e.value)
    mu, var = ens.forward(x)
    assert np.all(np.isfinite(mu)) and np.all(var > 0)


def test_argument_errors():
    c = helpers.workload('c1')
    ens = _ensemble(c)
    x = dev(np.zeros((3001, c['O'] + c['A']), np.float32))
    assert _kernels(ens, 3001)[0][0] == -2
    assert _forward(ens, x)[0] == -2
    x = dev(np.zeros((3000, c['O'] + c['A']), np.float32))
    mu = torch.empty((3000, c['O']), dtype=torch.float32, device='cuda')
    lib = _lib().load()
    h = ens._ensure_handle()
    assert lib.simba_ensemble_forward_tc(h, P(x), None, 3000, P(mu), P(mu), P(mu), None) == -1   # sample, no eps
    assert lib.simba_ensemble_forward_tc(h, P(x), None, 0, P(mu), P(mu), None, None) == -1
    assert _kernels(ens, 0)[0][0] == -1
    assert lib.simba_ensemble_forward_tc(h, None, None, 3000, P(mu), P(mu), None, None) == -1


# ---- 2: the planner's arithmetic, bit for bit ---------------------------------------------------------------------
@pytest.mark.parametrize("name", list(CASES))
def test_bit_identities_with_the_bf16_rollout(name):
    L = _lib()
    lib = L.load()
    c, B, x, eps, _ = _case(name)
    O, A = c['O'], c['A']
    ens = _ensemble(c)
    h = ens._ensure_handle()
    traj = torch.empty((B, 2, O), dtype=torch.float32, device='cuda')
    # (a) mean propagation: s_1 = s_0 + mu
    rc, mu, var, _ = _forward(ens, dev(x))
    assert rc == 0
    s0, acts = dev(x[:, :O]), dev(x[:, O:].reshape(B, 1, A))
    L.check(lib.simba_unfold_tc(h, P(s0), P(acts), None, 0, B, 1, 0, P(traj), None))
    torch.cuda.synchronize()
    s1 = traj[:, 1].cpu().numpy()
    want = x[:, :O] + mu.cpu().numpy()
    same = (s1 == want).mean()
    print("%s B=%d: s_1 == s_0 + mu on %.6f of elements" % (name, B, same))
    assert np.array_equal(s1, want)
    # (b) s_0 = 0, external draws, sampling propagation: s_1 = mu + sqrt(var) * eps
    x0 = x.copy()
    x0[:, :O] = 0.0
    d_eps = dev(eps)
    rc, mu0, var0, smp = _forward(ens, dev(x0), d_eps)
    assert rc == 0
    L.check(lib.simba_unfold_tc(h, P(dev(x0[:, :O])), P(acts), P(d_eps), 0, B, 1, 1, P(traj), None))
    torch.cuda.synchronize()
    s1 = traj[:, 1].cpu().numpy()
    smp = smp.cpu().numpy()
    print("%s B=%d: s_1 == sample on %.6f of elements" % (name, B, (s1 == smp).mean()))
    assert np.array_equal(s1, smp)
    assert np.all(var0.cpu().numpy() >= 1e-4)                        # softplus(raw) + 1e-4


# ---- 3: accuracy ---------------------------------------------------------------------------------------------------
# Normwise relative errors max|d| / max|ref| and mean|d| / mean|ref| of mu and var against the oracle (fp64 reference
# arithmetic on the fp32 weights). Measured on a B200 (148 SMs, 1000 W), every case above, var-head bias -2, worst
# case: mu max 7.4e-3, mean 5.5e-3; var max 6.4e-3, mean 1.5e-3 (the same against the fp32 kernel). Pinned about 2x
# above (DESIGN.md section 5).
MU_MAX, MU_MEAN = 1.5e-2, 1.1e-2
VAR_MAX, VAR_MEAN = 1.3e-2, 3e-3


def _rel(got, ref):
    d = np.abs(got.astype(np.float64) - ref)
    return d.max() / np.abs(ref).max(), d.mean() / np.abs(ref).mean()


@pytest.mark.parametrize("name", list(CASES))
def test_mu_and_var_close_to_the_oracle_and_to_fp32(name):
    c, B, x, eps, _ = _case(name)
    ens = _ensemble(c)
    rc, mu, var, _ = _forward(ens, dev(x))
    assert rc == 0
    mu, var = mu.cpu().numpy(), var.cpu().numpy()
    assert np.all(np.isfinite(mu)) and np.all(np.isfinite(var))
    ref = so.MlpEnsemble(c['weights'], dtype=np.float64)
    rmu, rvar = ref.forward_rows(x.astype(np.float64), np.repeat(np.arange(c['E']), B // c['E']))
    f_mu, f_var = ens.forward(x)
    m_mu, m_var = _rel(mu, rmu), _rel(var, rvar)
    f_mu_err, f_var_err = _rel(mu, f_mu.astype(np.float64)), _rel(var, f_var.astype(np.float64))
    print("%s B=%d: vs oracle mu max %.3g mean %.3g, var max %.3g mean %.3g; vs fp32 mu max %.3g mean %.3g, "
          "var max %.3g mean %.3g" % (name, B, *m_mu, *m_var, *f_mu_err, *f_var_err))
    assert m_mu[0] <= MU_MAX and m_mu[1] <= MU_MEAN
    assert m_var[0] <= VAR_MAX and m_var[1] <= VAR_MEAN
    assert f_mu_err[0] <= MU_MAX and f_mu_err[1] <= MU_MEAN
    assert f_var_err[0] <= VAR_MAX and f_var_err[1] <= VAR_MEAN


# Against tests/bf16_ref.py, which repeats every rounding of the kernels: what is left is the fp32 accumulation order,
# the MUFU ex2 / lg2 / sqrt and the rare bf16 flip they cause. The cases get N(0, 0.1) hidden and mu biases
# (_ref_case), so that every bias block has a lo half. Normwise max / mean of mu, var and the sample, and the fraction
# of rows with an element beyond bf16_ref.ROW_RTOL. Measured on a B200 (148 SMs, 1000 W), every case above, worst
# case: mu max 4.2e-4, mean 2.6e-6; var max 1.09e-3, mean 4.4e-6; sample max 3.8e-4, mean 2.4e-6; rows off 0.023
# (c5-wide). Pinned about 2x above. The means are 1500-4000x inside the oracle bounds, mu max 17x. The var max is only
# 6x: the maxima come from the rows off, where the accumulation order rounded one hidden activation to the other bf16
# neighbour, and one bf16 ulp of one activation moves a head output by up to that ulp times its weight. A second
# fp32 accumulation order of the same arithmetic reaches maxima of this size on the same cases
# (test_bf16_ref.py::test_a_second_fp32_accumulation_order_stays_inside_the_forward_bounds); the two-layer, 128-unit
# cases have no such row and agree to 6e-7.
REF_MU = (9e-4, 6e-6)
REF_VAR = (2.2e-3, 9e-6)
REF_SMP = (8e-4, 5e-6)
REF_ROWS_OFF = 0.046


def _ref_case(name):
    """_case with N(0, 0.1) hidden and mu biases (bf16_ref.with_biases), so that every bias block carries a lo half"""
    from tests import bf16_ref
    c, B, x, eps, kernel = _case(name)
    return bf16_ref.with_biases(c), B, x, eps, kernel


def _ref_forward(c, B, x, eps, rnd=None):
    from tests import bf16_ref
    ref = bf16_ref.TcEnsemble(c['weights'], rnd or bf16_ref.RN)
    mu, var = ref.forward_rows(x.astype(np.float64), np.repeat(np.arange(c['E']), B // c['E']))
    return mu, var, ref.delta(mu, var, eps)


def _ref_errors(got, want):
    """{'mu' | 'var' | 'sample': (normwise max, normwise mean, fraction of rows off)}"""
    from tests import bf16_ref
    return {k: bf16_ref.normwise(g, w) + (bf16_ref.rows_off(g, w),) for k, g, w in zip(('mu', 'var', 'sample'), got, want)}


@pytest.mark.parametrize("name", list(CASES))
def test_mu_var_and_sample_match_the_bf16_reference(name):
    c, B, x, eps, _ = _ref_case(name)
    ens = _ensemble(c)
    rc, mu, var, smp = _forward(ens, dev(x), dev(eps))
    assert rc == 0
    got = [t.cpu().numpy() for t in (mu, var, smp)]
    err = _ref_errors(got, _ref_forward(c, B, x, eps))
    print("%s B=%d vs bf16 reference: %s" % (name, B, ", ".join(
        "%s max %.3g mean %.3g rows off %.4f" % (k, *v) for k, v in err.items())))
    for k, (mx, mean) in (('mu', REF_MU), ('var', REF_VAR), ('sample', REF_SMP)):
        assert err[k][0] <= mx and err[k][1] <= mean, (k, err[k])
        assert err[k][2] <= REF_ROWS_OFF, (k, err[k])


def test_reference_fixture_forward():
    import os
    g = np.load(os.path.join(os.path.dirname(__file__), 'golden', 'reference_tiny_pieces.npz'))
    c = helpers.workload('tiny')
    ens = _ensemble(c)
    mu, var = ens.forward(g['forward_x'], precision='bf16')
    err = _rel(mu, g['forward_mu'].astype(np.float64))
    print("reference fixture: mu max %.3g mean %.3g (normwise), max abs %.3g"
          % (*err, np.abs(mu - g['forward_mu']).max()))
    assert np.allclose(mu, g['forward_mu'], rtol=2e-2, atol=1e-3)       # measured: max |d| 3.5e-4
    assert np.allclose(var, g['forward_var'], rtol=2e-2, atol=1e-6)


# ---- 4: memory and determinism -------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", ['c1-one-cta', 'c1-two-tile-over-one-wave', 'c5-wide', 'o63-actions-straddle-64',
                                  'o47-a2-actions-straddle-48'])
def test_nothing_beyond_the_outputs_and_two_calls_identical(name):
    c, B, x, eps, _ = _case(name)
    O = c['O']
    ens = _ensemble(c)
    lib = _lib().load()
    canary = 4096
    outs = []
    for _ in range(2):
        bufs = [torch.full((B * O + canary,), 12345.0, dtype=torch.float32, device='cuda') for _ in range(3)]
        assert lib.simba_ensemble_forward_tc(ens._ensure_handle(), P(dev(x)), P(dev(eps)), B, P(bufs[0]),
                                             P(bufs[1]), P(bufs[2]), None) == 0
        torch.cuda.synchronize()
        host = [b.cpu().numpy() for b in bufs]
        for hb in host:
            assert np.all(hb[B * O:] == 12345.0)
            assert not np.any(hb[:B * O] == 12345.0)
        outs.append(np.stack([hb[:B * O] for hb in host]))
    assert np.array_equal(outs[0].view(np.uint32), outs[1].view(np.uint32))


@pytest.mark.parametrize("cfg,sensors", [('c1', None), ('c5', None), ('c1', 92)])
def test_planner_plans_the_same_before_and_after_a_forward_call(cfg, sensors):
    c = helpers.workload(cfg, sensors=SENSORS[sensors] if sensors else None)
    pol = helpers.cuda_policy(c, 'penalty', precision='bf16')
    pol.build()
    a0, s0 = pol.do_generate_action(c['state'], seed=5)
    B = c['E'] * 500
    x = np.random.default_rng(2).uniform(0, 1, (B, c['O'] + c['A'])).astype(np.float32)
    pol.model.model.forward(x, precision='bf16')
    pol.model.model(x, np.ones((B, c['O']), np.float32), precision='bf16')
    a1, s1 = pol.do_generate_action(c['state'], seed=5)
    assert np.array_equal(np.asarray(a0).view(np.uint32), np.asarray(a1).view(np.uint32))
    assert np.float32(s0).view(np.uint32) == np.float32(s1).view(np.uint32)


# ---- 5: the Python surface -----------------------------------------------------------------------------------------
def test_python_surface():
    c = helpers.workload('c1', var_bias=-2.0)
    ens = _ensemble(c)
    rng = np.random.default_rng(3)
    B = c['E'] * 200
    x = rng.uniform(0, 1, (B, c['O'] + c['A'])).astype(np.float32)
    eps = rng.standard_normal((B, c['O'])).astype(np.float32)
    mu, var = ens.forward(x, precision='bf16')
    assert isinstance(mu, np.ndarray) and mu.shape == (B, c['O']) and var.shape == (B, c['O'])
    tmu, tvar = ens.forward(torch.from_numpy(x).cuda(), precision='bf16')
    assert isinstance(tmu, torch.Tensor) and tmu.is_cuda
    assert np.array_equal(tmu.cpu().numpy(), mu) and np.array_equal(tvar.cpu().numpy(), var)
    cmu, _ = ens.forward(torch.from_numpy(x), precision='bf16')
    assert isinstance(cmu, torch.Tensor) and not cmu.is_cuda
    mean, std, smp = ens(x, eps, precision='bf16')
    assert all(isinstance(a, np.ndarray) and a.shape == (B, c['O']) for a in (mean, std, smp))
    assert np.array_equal(mean, mu)
    assert np.array_equal(std, np.sqrt(var))                          # IEEE sqrt, as on the device
    rc, _, _, smp2 = _forward(ens, dev(x), dev(eps))
    assert rc == 0 and np.array_equal(smp, smp2.cpu().numpy())
    assert ens(x, precision='bf16')[2].shape == (B, c['O'])            # eps drawn with torch
    # the default is the fp32 call, byte for byte
    f_mu, f_var = ens.forward(x)
    _, r_mu, r_var, _ = _forward(ens, dev(x), precision='fp32')
    assert np.array_equal(f_mu.view(np.uint32), r_mu.cpu().numpy().view(np.uint32))
    assert np.array_equal(f_var.view(np.uint32), r_var.cpu().numpy().view(np.uint32))
    assert np.array_equal(ens.forward(x, precision='fp32')[0].view(np.uint32), f_mu.view(np.uint32))
    f_mean, f_std, f_smp = ens(x, eps)
    _, _, _, r_smp = _forward(ens, dev(x), dev(eps), precision='fp32')
    assert np.array_equal(f_smp.view(np.uint32), r_smp.cpu().numpy().view(np.uint32))
    assert 0 < np.abs(mu - f_mu).max() < 5e-2
    with pytest.raises(ValueError):
        ens.forward(x, precision='fp16')
    with pytest.raises(ValueError):
        ens(x, eps, precision='bf16x')
    with pytest.raises(TypeError):
        ens.forward(x, 'bf16')                                         # keyword-only
