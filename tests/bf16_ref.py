"""The bf16 tensor-core kernels' arithmetic, restated in float64 with every rounding the kernels make, for the tight
bf16 tests (tests/test_bf16_ref.py on the CPU, the *_tc GPU tests against the device).

The fp64 oracles (oracle/simba_oracle.py, oracle/train_oracle.py) compute what the model means; the bf16 kernels
compute it from bf16 operands with fp32 accumulation, so a bound against the oracles has to absorb the whole bf16
error. The classes here subclass those oracles and apply, at the point where a kernel applies it, each rounding the
kernel makes (DESIGN.md section 5): bf16 operands (round to nearest even), the bias as bf16 hi + lo, fp32 results of
every accumulator and epilogue operation. What is left between a kernel and this reference is the order of the fp32
accumulation inside the tensor cores, the MUFU approximations (ex2 / lg2 / sqrt .approx, treated as exact here) and
the rare bf16 rounding flip those two cause.

Every rounding goes through a `Rounding` object: `RN` is the kernels', `EXACT` replaces each rounding (and each fp32
constant) by the identity, which turns these classes back into the fp64 oracles (tests/test_bf16_ref.py holds them to
1e-10). The `Rounding` fields `drop_lo`, `act_rz`, `dz_rz`, `dz_exact` and `var_scale_after` build the mutants of
the sensitivity tests: arithmetic faults that the GPU bounds must be able to see.
"""
import dataclasses

import numpy as np

from oracle import simba_oracle as so
from oracle import train_oracle as T
from tests import swish_ref


# ---- roundings ----------------------------------------------------------------------------------------------------
def bf16_rn(x):
    """float32 -> bf16 -> float32, round to nearest even, as __float2bfloat16_rn / cvt.rn.bf16.f32 and the host
    packer's bf16_bits (internal.h:17): NaN stays NaN (the canonical NaN 0x7fff that cvt.rn.bf16.f32 makes), values
    that round above the largest bf16 become inf, subnormals round like normal numbers (bf16 has fp32's exponent
    range)."""
    u = np.asarray(x, dtype=np.float32).view(np.uint32).astype(np.uint64)
    nan = (u & 0x7fffffff) > 0x7f800000
    r = ((u + 0x7fff + ((u >> 16) & 1)) >> 16) << 16
    r = np.where(nan, np.uint64(0x7fff0000), r)
    return r.astype(np.uint32).view(np.float32)


def bf16_rz(x):
    """float32 -> bf16 -> float32 toward zero (truncation): the fault the sensitivity tests plant."""
    u = np.asarray(x, dtype=np.float32).view(np.uint32)
    return (u & np.uint32(0xffff0000)).view(np.float32)


def bf16_split(v):
    """(hi, lo) of a bias as the kernels carry it (internal.h:31): hi = bf16(v), lo = bf16(v - hi)."""
    v = np.asarray(v, dtype=np.float32)
    hi = bf16_rn(v)
    return hi, bf16_rn(v - hi)


@dataclasses.dataclass(frozen=True)
class Rounding:
    exact: bool = False              # EXACT: every rounding and fp32 constant is the identity
    drop_lo: bool = False            # mutant: biases lose their lo half
    act_rz: bool = False             # mutant: hidden activations (forward A operands) converted toward zero
    dz_rz: bool = False              # mutant: dZ converted toward zero for the backward and update GEMMs
    dz_exact: bool = False           # mutant: dZ enters the backward and update GEMMs unrounded
    var_scale_after: bool = False    # mutant: var head rounded to bf16 before its log2(e) pre-scale
    acc32: bool = False              # the forward GEMMs accumulated in fp32 in numpy's order, not exactly

    @property
    def dt(self):
        """the type the kernels' fp32 library math (softplus, swish) runs in"""
        return np.float64 if self.exact else np.float32

    def f32(self, x):
        x = np.asarray(x, dtype=np.float64)
        return x if self.exact else x.astype(np.float32).astype(np.float64)

    def const(self, v):
        """an fp32 constant of the kernels (1e-4f, kLog2e, ln 2)"""
        return float(v) if self.exact else float(np.float32(v))

    def bf16(self, x, rz=False):
        """an fp32 value converted to a bf16 operand"""
        x = np.asarray(x, dtype=np.float64)
        if self.exact:
            return x
        return (bf16_rz if rz else bf16_rn)(x.astype(np.float32)).astype(np.float64)

    def bias(self, b):
        """hi + lo, the two bias rows of a GEMM that the A operand multiplies by constant ones"""
        b = np.asarray(b, dtype=np.float64)
        if self.exact:
            return b
        hi, lo = bf16_split(b.astype(np.float32))
        return hi.astype(np.float64) + (0.0 if self.drop_lo else lo.astype(np.float64))

    def gemm(self, a, w, b):
        """fp32 accumulator of a . w + hi + lo: exact, then rounded once to fp32 (acc32: accumulated in fp32, so a
        different summation order than the kernel's, as a second kernel would have)"""
        if not self.acc32:
            return self.f32(a @ w + b)
        acc = np.asarray(a, np.float32) @ np.asarray(w, np.float32)
        return (acc + np.asarray(b, np.float32)).astype(np.float64)     # hi + lo is exact in fp32

    def dz(self, d):
        """dZ as the backward and update GEMMs read it: bf16 of the fp32 value (trainer_tc.cu:345, :469)"""
        return self.f32(d) if self.dz_exact else self.bf16(d, rz=self.dz_rz)


RN = Rounding()
EXACT = Rounding(exact=True)
MUTANTS = {
    'lo-dropped': Rounding(drop_lo=True),
    'activation-toward-zero': Rounding(act_rz=True),
    'var-head-rounded-before-scale': Rounding(var_scale_after=True),
    'dz-toward-zero': Rounding(dz_rz=True),
    'dz-not-rounded': Rounding(dz_exact=True),
}
ACC32 = Rounding(acc32=True)


def with_biases(c, seed=5, scale=0.1):
    """workload c with N(0, scale) hidden and mu-head biases: the synthetic workloads' are zero, and a zero bias is
    packed as hi = lo = 0 whatever the packer does"""
    rng = np.random.default_rng(seed)
    members = []
    for m in c['weights']:
        m = [a.copy() for a in m]
        for i in range(1, len(m) - 2, 2):                # b_1 .. b_L and b_mu; the var bias stays
            m[i] = rng.normal(0, scale, m[i].shape).astype(np.float32)
        members.append(m)
    return dict(c, weights=members)

LOG2E = 1.4426950408889634          # kLog2e (internal.h:40)
LN2 = 0.6931471805599453            # tc_head.cuh:153, :371


# ---- forward: simba_ensemble_forward_tc (rollout_tc.cu / rollout_tc_wide.cu packers, tc_head.cuh) ----------------
class TcEnsemble(so.MlpEnsemble):
    """so.MlpEnsemble with the bf16 rollout kernels' roundings. `mlp` takes the fp32 layer-0 input x_scaled (the
    forward form's identity tables make it x itself) and returns (mu, var) as the kernels store them."""

    def __init__(self, members, rnd=RN):
        super().__init__(members, dtype=np.float64)
        self.r = rnd

    def mlp(self, e, x):
        r, w = self.r, self.members[e]
        n_layers = (len(w) - 4) // 2
        h = r.bf16(x)                                    # A operand of layer 0: bf16(fma(x, a, b)), tc_head.cuh:191
        for l in range(n_layers):
            # bf16 weights, bias hi + lo (rollout_tc.cu:1009-1013, :1029; rollout_tc_wide.cu:648-652), fp32 accumulator
            z = r.gemm(h, r.bf16(w[2 * l]), r.bias(w[2 * l + 1]))
            h = r.bf16(np.maximum(z, 0.0), rz=r.act_rz)  # cvt.rn.relu.bf16x2 (tc_ptx.cuh:147)
        mu = r.gemm(h, r.bf16(w[-4]), r.bias(w[-3]))    # the mu head's fp32 accumulator (tc_head.cuh:266)
        log2e = r.const(LOG2E)
        if r.var_scale_after:
            raw = r.f32(log2e * r.gemm(h, r.bf16(w[-2]), r.bias(w[-1])))
        else:                                            # bf16(fp32(log2e W)), split(fp32(log2e b)): rollout_tc.cu:1015, :1027
            raw = r.gemm(h, r.bf16(r.f32(log2e * w[-2])), r.bias(r.f32(log2e * w[-1])))
        return mu, self.variance(raw)

    def variance(self, raw):
        """fma(lg2(1 + ex2(min(raw, 120))), ln 2, 1e-4) with ex2 / lg2 exact and each result fp32 (tc_head.cuh:377-382)"""
        r = self.r
        e = r.f32(np.exp2(np.minimum(raw, 120.0)))
        l = r.f32(np.log2(r.f32(1.0 + e)))
        return r.f32(l * r.const(LN2) + r.const(1e-4))

    def delta(self, mu, var, eps):
        """mu + sqrt(var) * bf16(eps) as one fp32 FMA (tc_head.cuh:384-392)"""
        r = self.r
        return r.f32(r.f32(np.sqrt(var)) * r.bf16(eps) + mu)

    def __call__(self, x, eps, member_of_row=None):
        mu, var = self.forward(x) if member_of_row is None else self.forward_rows(x, member_of_row)
        return mu, np.sqrt(var), self.delta(mu, var, eps)


# ---- trajectories: simba_unfold_tc --------------------------------------------------------------------------------
class TcTransitionModel(so.TransitionModel):
    """so.TransitionModel over a TcEnsemble: x_t = bf16(fma(s_t, a, b)) with the model's fp32 scale tables
    (api.cu:207-208, tc_head.cuh:187-191), s_{t+1} = fp32(s_t + mu) or fp32(s_t + fp32(mu + sqrt(var) bf16(eps)))
    (tc_head.cuh:390, :398)."""

    def __init__(self, members, inputs_min, inputs_max, sampling_propagation=True, rnd=RN):
        super().__init__(TcEnsemble(members, rnd), inputs_min, inputs_max, True, sampling_propagation,
                         dtype=np.float64)
        self.r = rnd

    def scale(self, x):
        r = self.r
        delta = self.inputs_max - self.inputs_min
        delta = np.where(delta < r.const(1e-5), r.const(1.01), r.f32(delta))
        a = r.f32(1.0 / delta)
        b = r.f32(-self.inputs_min * a)
        return r.f32(x * a + b)                           # one fp32 FMA

    def unfold_sequences(self, s_0, action_sequences, eps, member_of_row=None):
        r = self.r
        horizon = action_sequences.shape[1]
        traj = np.empty((s_0.shape[0], horizon + 1, s_0.shape[1]), dtype=np.float64)
        s_t = np.asarray(s_0, dtype=np.float64).copy()
        for t in range(horizon):
            traj[:, t] = s_t
            x = self.scale(np.concatenate([s_t, action_sequences[:, t]], axis=1))
            mus, _, d_s_t = self.model(x, np.asarray(eps[t], dtype=np.float64), member_of_row)
            s_t = r.f32(s_t + (d_s_t if self.sampling_propagation else mus))
        traj[:, horizon] = s_t
        return traj


# ---- training: train_tc_chain_kernel + train_tc_update_kernel (trainer_tc.cu) ------------------------------------
class TcMemberNet(T.MemberNet):
    """T.MemberNet with the bf16 trainer's roundings. The variables (Adam's master weights) stay in `dtype`; the
    step computes in float64 from bf16(theta) and returns gradients in `dtype`.

      A operand of layer 0      bf16(x), ones at k = K, K + 1 carry the bias hi + lo (trainer_tc.cu:196, :633-634)
      hidden                    H = fp32(relu(Z) keep) kept in fp32, next A operand bf16(H) (:285-316)
      head                      mu, raw var = the fp32 accumulator; nll_terms in fp32 (train_common.cuh:176-185)
      back-propagation          dZ_{l-1} = fp32(fp32(bf16(dZ_l) . bf16(theta_l)^T) keep) where H_l > 0 (:350-375)
      weight gradients          fp32(bf16([H, 1])^T . bf16(dZ)) (:445-498)
    """
    swish = False

    def __init__(self, arrays, dtype=np.float32, rnd=RN):
        super().__init__(arrays, dtype)
        self.r = rnd

    def act(self, z, keep):
        """(H, multiplier of the backward pass) of an fp32 pre-activation Z"""
        r = self.r
        if self.swish:
            zt = z.astype(r.dt)
            h, g = swish_ref.swish(zt).astype(np.float64), swish_ref.swish_grad(zt).astype(np.float64)
            if keep is not None:
                k = keep.astype(np.float64)
                h, g = r.f32(h * k), r.f32(k * g)
            return h, g
        h = np.maximum(z, 0.0)
        if keep is not None:
            h = r.f32(h * keep.astype(np.float64))
        return h, None

    def operand(self, hs, l):
        """bf16 of layer l's fp32 input, as the chain's A tile and the update kernel's staging hold it"""
        return self.r.bf16(hs[l], rz=self.r.act_rz and l > 0)

    def forward(self, x, keep=None):
        r, L = self.r, self.n_layers
        w = [np.asarray(a, dtype=np.float64) for a in self.arrays]
        hs, mults = [np.asarray(x, dtype=np.float64)], []
        for l in range(L):
            z = r.f32(self.operand(hs, l) @ r.bf16(w[2 * l]) + r.bias(w[2 * l + 1]))
            h, m = self.act(z, None if keep is None else keep[l])
            hs.append(h)
            mults.append(m)
        a = self.operand(hs, L)
        mu = r.f32(a @ r.bf16(w[2 * L]) + r.bias(w[2 * L + 1]))
        raw = r.f32(a @ r.bf16(w[2 * L + 2]) + r.bias(w[2 * L + 3]))
        var = r.f32(so.tf_softplus(raw.astype(r.dt)).astype(np.float64) + r.const(1e-4))
        return mu, var, (hs, raw, mults, w)

    def loss_and_grads(self, x, y, loss_scale=1.0, keep=None):
        r, L = self.r, self.n_layers
        mu, var, (hs, raw, mults, w) = self.forward(x, keep)
        y = np.asarray(y, dtype=np.float64)
        loss = T.negative_log_likelihood(y, mu, var) * loss_scale
        c = r.f32(loss_scale / mu.size)
        diff = mu - y
        d_mu = r.f32(c * diff / var)
        d_var = 0.5 * c * (1.0 / var - np.square(diff) / np.square(var))
        d_raw = r.f32(d_var / (1.0 + np.exp(-raw)))
        grads = [None] * len(self.arrays)
        zmu, zraw = r.dz(d_mu), r.dz(d_raw)
        a = self.operand(hs, L)
        grads[2 * L] = a.T @ zmu
        grads[2 * L + 1] = zmu.sum(axis=0)
        grads[2 * L + 2] = a.T @ zraw
        grads[2 * L + 3] = zraw.sum(axis=0)
        d_h = r.f32(zmu @ r.bf16(w[2 * L]).T + zraw @ r.bf16(w[2 * L + 2]).T)
        for l in range(L - 1, -1, -1):
            if self.swish:
                d_z = r.f32(d_h * mults[l])
            else:
                back = keep[l].astype(np.float64) if keep is not None else 1.0
                d_z = np.where(hs[l + 1] > 0, r.f32(d_h * back), 0.0)
            zl = r.dz(d_z)
            grads[2 * l] = self.operand(hs, l).T @ zl
            grads[2 * l + 1] = zl.sum(axis=0)
            if l > 0:
                d_h = r.f32(zl @ r.bf16(w[2 * l]).T)
        return self.dtype.type(loss), [r.f32(g).astype(self.dtype) for g in grads]


class TcSwishMemberNet(TcMemberNet):
    """TcMemberNet with the swish trainer's fp32 epilogue: H = swish_f32(Z) keep, M = keep swish_grad_f32(Z)
    (trainer_tc.cu:276-297), back-propagation multiplies by M (:364)."""
    swish = True


class TcEnsembleTrainer(T.EnsembleTrainer):
    """T.EnsembleTrainer over TcMemberNets: float32 master weights, clip and Adam (T.Adam), bf16(theta) re-read
    every step. validation_step is the training forward pass without dropout."""

    def __init__(self, members, dtype=np.float32, rnd=RN, swish=False, **kw):
        super().__init__(members, dtype=dtype, **kw)
        cls = TcSwishMemberNet if swish else TcMemberNet
        self.nets = [cls(n.arrays, dtype, rnd) for n in self.nets]


# ---- metrics of the tests against this reference ------------------------------------------------------------------
# A row "agrees" when every element is within ROW_RTOL of the reference's normwise scale max|ref|: the fp32
# accumulation order moves an element by about 1e-7 of it, one bf16 rounding flip upstream by 1e-5 or more.
ROW_RTOL = 1e-5


def normwise(got, ref):
    """(max|d| / max|ref|, mean|d| / mean|ref|)"""
    ref = np.asarray(ref, np.float64)
    d = np.abs(np.asarray(got, np.float64) - ref)
    return float(d.max() / np.abs(ref).max()), float(d.mean() / np.abs(ref).mean())


def rows_off(got, ref, scale=None, rtol=ROW_RTOL):
    """fraction of rows (first axis) with an element further than rtol * scale (default max|ref|) from ref"""
    ref = np.asarray(ref, np.float64)
    d = np.abs(np.asarray(got, np.float64) - ref).reshape(ref.shape[0], -1)
    scale = np.abs(ref).max() if scale is None else scale
    return float((d.max(axis=1) > rtol * scale).mean())
