"""tests/bf16_ref.py on the CPU: its rounding agrees with torch's bf16 bit for bit, without its roundings it is the fp64
oracles again, and the bounds of the GPU tests against it can see the arithmetic faults it is there to catch.

The sensitivity guard runs a mutated reference (one rounding wrong: the bias lo half dropped, round toward zero in an
activation or dZ conversion, the var head rounded before its log2(e) pre-scale, dZ not rounded) on the GPU tests' own
cases and protocol and asks that it land at least 3x beyond one of the bounds those tests pin (2x for unrounded dZ in
training). A bound loosened until a fault of this kind passes fails here, without a GPU. The module needs neither a
GPU nor the built library."""
import numpy as np
import pytest

from oracle import simba_oracle as so
from oracle import train_oracle as T
from tests import bf16_ref as R
from tests import swish_ref
from tests import test_gpu_forward_tc as FWD
from tests import test_gpu_train_tc as TRN
from tests import test_gpu_unfold_tc as UNF

torch = pytest.importorskip("torch")


# ---- rounding -----------------------------------------------------------------------------------------------------
def _grid():
    f32 = np.finfo(np.float32)
    base = np.array([0.0, 1.0, 1.5, 3.0, 1e-3, 0.1, 255.5, 65504.0, 3.4e38, f32.max, f32.tiny, 1e-40, 1e-45,
                     f32.smallest_subnormal, np.inf, np.nan], dtype=np.float32)
    u = base.view(np.uint32)
    # exact ties (low half 0x8000) with an even and an odd kept half, one ulp either side, and the low-half extremes
    near = np.concatenate([u + d for d in (0x7fff, 0x8000, 0x8001, 0x18000, 0x17fff, 0x18001, 0xffff, 0x10000)])
    rnd = np.random.default_rng(0).integers(0, 2 ** 32, 200000, dtype=np.uint64).astype(np.uint32)
    bits = np.concatenate([u, near, rnd, np.array([0x7f7f8000, 0x7f7fffff, 0x7f7f7fff, 0x007f8000, 0x00008000,
                                                   0x00018000, 0x7f800001, 0x7fc00000, 0x7fffffff], np.uint32)])
    bits = np.concatenate([bits, bits | np.uint32(0x80000000)])                      # and the negatives
    return bits.view(np.float32)


def test_bf16_rn_equals_torch_bit_for_bit():
    x = _grid()
    got = R.bf16_rn(x)
    want = torch.from_numpy(x.copy()).to(torch.bfloat16).float().numpy()
    nan = np.isnan(x)
    assert np.array_equal(got[~nan].view(np.uint32), want[~nan].view(np.uint32))
    # NaN payloads differ (torch-CPU makes 0xffff, cvt.rn.bf16.f32 the canonical 0x7fff): NaN stays NaN
    assert nan.sum() > 4 and np.all(np.isnan(got[nan])) and np.all(np.isnan(want[nan]))
    assert np.isinf(R.bf16_rn(np.float32(np.finfo(np.float32).max)))                # rounds above the largest bf16
    assert R.bf16_rn(np.float32(1e-45)) == 0.0 and R.bf16_rn(np.float32(-1e-45)).view(np.uint32) == 0x80000000
    assert R.bf16_rn(np.float32(1.0 + 2 ** -8)) == 1.0                               # tie to even (down)
    assert R.bf16_rn(np.float32(1.0 + 3 * 2 ** -8)) == 1.0 + 2 ** -6                # tie to even (up)


def test_bf16_split_is_hi_plus_a_rounded_residual():
    v = np.random.default_rng(1).normal(0, 1, 10000).astype(np.float32)
    hi, lo = R.bf16_split(v)
    assert np.array_equal(hi, R.bf16_rn(v)) and np.array_equal(lo, R.bf16_rn(v - hi))
    err = np.abs((hi.astype(np.float64) + lo) - v) / np.abs(v)
    assert err.max() <= 2.0 ** -16 and np.abs(v - hi).max() > 0                   # hi + lo carries ~16 bits
    assert np.array_equal(R.bf16_rz(v), (v.view(np.uint32) & 0xffff0000).view(np.float32))


# ---- without its roundings the reference is the fp64 oracles --------------------------------------------------------
def _close(a, b, tol=1e-10):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    return np.abs(a - b).max() <= tol * max(np.abs(b).max(), 1e-30)


@pytest.mark.parametrize("name", ['o47-a2-actions-straddle-48', 'c5-wide', 'b-not-multiple-of-128'])
def test_exact_forward_is_the_oracle(name):
    c, B, x, eps, _ = FWD._ref_case(name)
    rows = np.repeat(np.arange(c['E']), B // c['E'])
    mu, var = so.MlpEnsemble(c['weights'], dtype=np.float64).forward_rows(x.astype(np.float64), rows)
    emu, evar = R.TcEnsemble(c['weights'], R.EXACT).forward_rows(x.astype(np.float64), rows)
    assert _close(emu, mu) and _close(evar, var)
    _, _, smp = so.MlpEnsemble(c['weights'], dtype=np.float64)(x.astype(np.float64), eps.astype(np.float64), rows)
    assert _close(R.TcEnsemble(c['weights'], R.EXACT)(x.astype(np.float64), eps, rows)[2], smp)


def _oracle_unfold(c, s0, acts, eps, sampling):
    ens = so.MlpEnsemble(c['weights'], dtype=np.float64)
    tm = so.TransitionModel(ens, c['smin'], c['smax'], True, sampling, dtype=np.float64)
    return tm.unfold_sequences(s0, acts, eps)


@pytest.mark.parametrize("sampling", [True, False])
def test_exact_trajectories_are_the_oracle(sampling):
    c, B, s0, acts, eps = UNF._ref_case('o47-a2-actions-straddle-48', sampling)
    want = _oracle_unfold(c, s0, acts, eps, sampling)
    got = R.TcTransitionModel(c['weights'], c['smin'], c['smax'], sampling, R.EXACT).unfold_sequences(s0, acts, eps)
    assert _close(got, want)


@pytest.mark.parametrize("swish", [False, True])
@pytest.mark.parametrize("rate", [0.0, 0.5])
def test_exact_loss_and_grads_are_the_oracle(swish, rate):
    shape = TRN.REF_CASES['l6' if not swish else 'swish-u130'][0]
    n_in, n_out, E, rows, L, U = shape
    arrays = TRN._ref_weights(shape)[0]
    x, y = TRN._data(np.random.default_rng(13), 1, rows, n_in, n_out)
    keep = None
    if rate:
        rng = np.random.default_rng(2)
        keep = [(rng.uniform(size=(rows, U)) >= rate).astype(np.float32) / np.float32(1 - rate) for _ in range(L)]
    base = swish_ref.MemberNet if swish else T.MemberNet
    loss, grads = base(arrays, np.float64).loss_and_grads(x[0], y[0], 1.0 / 3, keep)
    cls = R.TcSwishMemberNet if swish else R.TcMemberNet
    eloss, egrads = cls(arrays, np.float64, R.EXACT).loss_and_grads(x[0], y[0], 1.0 / 3, keep)
    assert abs(eloss - loss) <= 1e-10 * abs(loss)
    for g, w in zip(egrads, grads):
        assert _close(g, w)
    # and the roundings are what moves it: the RN reference is no closer than bf16 allows, and not further
    _, rgrads = cls(arrays, np.float32, R.RN).loss_and_grads(x[0], y[0], 1.0 / 3, keep)
    worst = max(TRN._rel(g, w) for g, w in zip(rgrads, grads))
    assert 1e-4 < worst < 0.3


# ---- the forward maxima are accumulation-order flips ----------------------------------------------------------------
@pytest.mark.parametrize("name", list(FWD.CASES))
def test_a_second_fp32_accumulation_order_stays_inside_the_forward_bounds(name):
    """The same arithmetic accumulated in fp32 in numpy's order, not exactly: an implementation that differs from the
    reference only where the kernels may. It stays inside the pinned bounds, and on the wide cases it reaches a
    normwise max of the size the B200 measured, which is why the max bounds sit above the means."""
    c, B, x, eps, _ = FWD._ref_case(name)
    err = FWD._ref_errors(FWD._ref_forward(c, B, x, eps, R.ACC32), FWD._ref_forward(c, B, x, eps))
    print("%s fp32-accumulated: %s" % (name, err))
    for k, (mx, mean) in (('mu', FWD.REF_MU), ('var', FWD.REF_VAR), ('sample', FWD.REF_SMP)):
        assert err[k][0] <= mx and err[k][1] <= mean and err[k][2] <= FWD.REF_ROWS_OFF, (k, err[k])
    if c['L'] * c['U'] >= 512:                           # enough activations for flips on these batches
        assert err['mu'][2] > 0 and max(err['mu'][0], err['var'][0]) > FWD.REF_MU[0] / 20


# ---- sensitivity guard ------------------------------------------------------------------------------------------
def _worst_ratio(errs, bounds):
    """max over the asserted quantities of error / bound"""
    return max(e / b for e, b in zip(errs, bounds))


FORWARD_MUTANTS = ['lo-dropped', 'activation-toward-zero', 'var-head-rounded-before-scale']


@pytest.mark.parametrize("name", list(FWD.CASES))
def test_forward_bounds_see_every_fault(name):
    c, B, x, eps, _ = FWD._ref_case(name)
    ref = FWD._ref_forward(c, B, x, eps)
    bounds = FWD.REF_MU + (FWD.REF_ROWS_OFF,) + FWD.REF_VAR + (FWD.REF_ROWS_OFF,) + FWD.REF_SMP + (FWD.REF_ROWS_OFF,)
    for m in FORWARD_MUTANTS:
        err = FWD._ref_errors(FWD._ref_forward(c, B, x, eps, R.MUTANTS[m]), ref)
        ratio = _worst_ratio(err['mu'] + err['var'] + err['sample'], bounds)
        print("%s %s: %s, worst error / bound %.3g" % (name, m, err, ratio))
        assert ratio >= 3.0, (m, err)
        if m == 'lo-dropped':                            # seen in mu too, not only through the var head
            assert _worst_ratio(err['mu'], FWD.REF_MU + (FWD.REF_ROWS_OFF,)) >= 3.0, err


@pytest.mark.parametrize("sampling", [True, False])
@pytest.mark.parametrize("name", list(UNF.ORACLE))
def test_trajectory_bounds_see_every_fault(name, sampling):
    c, B, s0, acts, eps = UNF._ref_case(name, sampling)
    ref = UNF._ref_trajectories(c, s0, acts, eps, sampling)
    bounds = UNF.REF_STEP1 + UNF.REF_ANY_STEP + (UNF.REF_ROWS_OFF,)
    for m in FORWARD_MUTANTS:
        if m == 'var-head-rounded-before-scale' and not sampling:
            continue                                     # mean propagation never reads the variance
        err = UNF._ref_traj_errors(UNF._ref_trajectories(c, s0, acts, eps, sampling, R.MUTANTS[m]), ref)
        ratio = _worst_ratio(err, bounds)
        print("%s sampling=%d %s: %s, worst error / bound %.3g" % (name, sampling, m, err, ratio))
        assert ratio >= 3.0, (m, err)


# mutant: the margin it must keep beyond the bounds. Unrounded dZ differs from bf16(dZ) by errors that average out
# over the batch, about as 1 / sqrt(rows): at 300 rows it lands 2.5x beyond the bounds, at 128 rows 3.2x.
TRAIN_MUTANTS = {'lo-dropped': 3.0, 'activation-toward-zero': 3.0, 'dz-toward-zero': 3.0, 'dz-not-rounded': 2.0}


@pytest.mark.parametrize("name", list(TRN.REF_CASES))
def test_training_bounds_see_every_fault(name):
    """The GPU test's protocol with a mutated reference in the kernels' place: every step, the RN reference starts
    from the mutant's weights and Adam slots, and all five quantities are compared."""
    shape, rate, steps, act = TRN.REF_CASES[name]
    members = TRN._ref_weights(shape)
    batches = TRN._ref_batches(shape, steps)
    for m, margin in TRAIN_MUTANTS.items():
        mut = TRN._ref_trainer(members, shape, rate, act, R.MUTANTS[m])
        ref = TRN._ref_trainer(members, shape, rate, act)

        def step(x, y):
            return float(mut.training_step(x, y)), mut.last_grads

        def state():
            return [a for n in mut.nets for a in n.arrays], mut.optimizer.m, mut.optimizer.v
        worst = TRN._ref_run(step, state, ref, batches, mut.optimizer.lr0, '%s %s' % (name, m))
        ratio = (worst / TRN._bounds(act)).max()
        print("%s %s: worst error / bound %.3g" % (name, m, ratio))
        assert ratio >= margin, (m, worst)
