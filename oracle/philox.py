"""TEST INFRASTRUCTURE ONLY — the RNG contract of the planner, restated on the CPU.

The reference draws its normals with TensorFlow's stateful generators
(`tf.random.normal` at simba/policies/cem_mpc.py:44,68 and
`tfp.distributions.Normal.sample` at simba/models/mlp_ensemble.py:192-193). That draw
order is TF-internal and cannot be reproduced without TensorFlow, so parity is defined
"given identical draws". This module defines the draws of the CUDA kernels' *production*
mode (counter-based Philox4x32-10, Salmon et al. SC'11 / Random123) so that the oracle can
be fed exactly the normals a kernel will generate on the device.

Counter map (must match csrc/philox.cuh):
    key     = (seed_lo, seed_hi)
    counter = (c0, c1, c2, c3)
        c0 = block index j: the 4 outputs of one Philox call are elements 4j .. 4j+3
        c1 = row index (candidate i for ACTION, global row r = p*N + i for NOISE, 0 for FINAL)
        c2 = t | (iteration << 16)
        c3 = state index s | (stream << 28)
    streams: ACTION = 1 (elements = flattened (h, a)), NOISE = 2 (elements = observation
    dims o), FINAL = 3 (elements = action dims a).
ACTION / FINAL streams (4 normals per Philox block, 24-bit uniforms):
  Uniforms:  u = ((x >> 8) + 0.5) * 2**-24   (fp32 arithmetic, never 0)
  Normals :  Box-Muller on (x0, x1) and (x2, x3):
             z_even = sqrt(-2 ln u_a) * cos(2 pi u_b),  z_odd = sqrt(-2 ln u_a) * sin(2 pi u_b)
NOISE stream (8 normals per Philox block, 16-bit uniforms — the rollout draws 60 of these per
transition, so the Philox cost per normal is halved): every 32-bit word x gives one pair
  u_a = ((x & 0xffff) + 0.5) * 2**-16,  u_b = ((x >> 16) + 0.5) * 2**-16   (exact in fp32)
  z_even = sqrt(-2 ln u_a) * cos(2 pi u_b),  z_odd = sqrt(-2 ln u_a) * sin(2 pi u_b)
  c0 is then the index of the block of 8 consecutive observation dims; |z| <= 4.85.
The oracle evaluates the Box-Muller formula in float64 and rounds once to float32; the
device evaluates it in fp32 (a few ulp away) — tests state that tolerance.
"""
import numpy as np

PHILOX_M0 = np.uint64(0xD2511F53)
PHILOX_M1 = np.uint64(0xCD9E8D57)
PHILOX_W0 = 0x9E3779B9
PHILOX_W1 = 0xBB67AE85

STREAM_ACTION = 1
STREAM_NOISE = 2
STREAM_FINAL = 3
STREAM_DROPOUT = 4      # training only: counter (column block, batch row, iteration, member | layer << 8 | 4 << 28)

_MASK32 = np.uint64(0xFFFFFFFF)


def philox4x32(counter, key, rounds=10):
    """Philox4x32-R. counter: (..., 4) uint32, key: (2,) or (..., 2) uint32 -> (..., 4) uint32."""
    counter = np.asarray(counter, dtype=np.uint32)
    key = np.asarray(key, dtype=np.uint32)
    c0 = counter[..., 0].astype(np.uint64)
    c1 = counter[..., 1].astype(np.uint64)
    c2 = counter[..., 2].astype(np.uint64)
    c3 = counter[..., 3].astype(np.uint64)
    k0 = np.broadcast_to(key[..., 0], c0.shape).astype(np.uint64)
    k1 = np.broadcast_to(key[..., 1], c0.shape).astype(np.uint64)
    for _ in range(rounds):
        p0 = PHILOX_M0 * c0
        p1 = PHILOX_M1 * c2
        hi0, lo0 = p0 >> np.uint64(32), p0 & _MASK32
        hi1, lo1 = p1 >> np.uint64(32), p1 & _MASK32
        c0, c1, c2, c3 = (hi1 ^ c1 ^ k0) & _MASK32, lo1, (hi0 ^ c3 ^ k1) & _MASK32, lo0
        k0 = (k0 + np.uint64(PHILOX_W0)) & _MASK32
        k1 = (k1 + np.uint64(PHILOX_W1)) & _MASK32
    return np.stack([c0, c1, c2, c3], axis=-1).astype(np.uint32)


def uniform_from_bits(x):
    """u = ((x >> 8) + 0.5) * 2^-24 in fp32 (round-to-nearest-even on the add, exact scale)."""
    return ((x >> np.uint32(8)).astype(np.float32) + np.float32(0.5)) * np.float32(2.0 ** -24)


def normals_from_bits(x):
    """(..., 4) uint32 -> (..., 4) float32 normals (Box-Muller contract, f64 math, one rounding)."""
    u = uniform_from_bits(np.asarray(x, dtype=np.uint32)).astype(np.float64)
    ra = np.sqrt(-2.0 * np.log(u[..., 0]))
    rb = np.sqrt(-2.0 * np.log(u[..., 2]))
    ta = 2.0 * np.pi * u[..., 1]
    tb = 2.0 * np.pi * u[..., 3]
    z = np.stack([ra * np.cos(ta), ra * np.sin(ta), rb * np.cos(tb), rb * np.sin(tb)], axis=-1)
    return z.astype(np.float32)


def normals8_from_bits(x):
    """(..., 4) uint32 -> (..., 8) float32 normals: the NOISE-stream contract (16-bit uniforms)."""
    x = np.asarray(x, dtype=np.uint32)
    ua = ((x & np.uint32(0xFFFF)).astype(np.float64) + 0.5) * 2.0 ** -16
    ub = ((x >> np.uint32(16)).astype(np.float64) + 0.5) * 2.0 ** -16
    r = np.sqrt(-2.0 * np.log(ua))
    th = 2.0 * np.pi * ub
    z = np.stack([r * np.cos(th), r * np.sin(th)], axis=-1)          # (..., 4, 2)
    return z.reshape(x.shape[:-1] + (8,)).astype(np.float32)


def _key(seed):
    seed = int(seed) & 0xFFFFFFFFFFFFFFFF
    return np.array([seed & 0xFFFFFFFF, seed >> 32], dtype=np.uint32)


def _normals(seed, n_elems, c1, c2, c3, per_block=4):
    """Normals for elements 0..n_elems-1 over broadcast index arrays c1/c2/c3 -> (..., n_elems)."""
    nblk = (n_elems + per_block - 1) // per_block
    c1, c2, c3 = np.broadcast_arrays(np.asarray(c1, np.uint32), np.asarray(c2, np.uint32),
                                     np.asarray(c3, np.uint32))
    shape = c1.shape
    ctr = np.empty(shape + (nblk, 4), dtype=np.uint32)
    ctr[..., 0] = np.arange(nblk, dtype=np.uint32)
    ctr[..., 1] = c1[..., None]
    ctr[..., 2] = c2[..., None]
    ctr[..., 3] = c3[..., None]
    bits = philox4x32(ctr, _key(seed))
    z = normals_from_bits(bits) if per_block == 4 else normals8_from_bits(bits)
    return z.reshape(shape + (nblk * per_block,))[..., :n_elems]


def action_normals(seed, iteration, n_samples, horizon, act_dim, state_index=0, first_candidate=0):
    """z for cem_mpc.py:44 — shape [n_samples, horizon, act_dim]; candidate index is global."""
    cand = np.arange(first_candidate, first_candidate + n_samples, dtype=np.uint32)
    z = _normals(seed, horizon * act_dim, cand, np.uint32(iteration << 16),
                 np.uint32(state_index | (STREAM_ACTION << 28)))
    return z.reshape(n_samples, horizon, act_dim)


def noise_normals(seed, iteration, horizon, rows, obs_dim, state_index=0):
    """eps for mlp_ensemble.py:193 — shape [horizon, len(rows), obs_dim]; rows are GLOBAL row ids."""
    rows = np.asarray(rows, dtype=np.uint32)
    t = np.arange(horizon, dtype=np.uint32)[:, None]
    return _normals(seed, obs_dim, rows[None, :], t | np.uint32(iteration << 16),
                    np.uint32(state_index | (STREAM_NOISE << 28)), per_block=8)


def final_normals(seed, act_dim, state_index=0):
    """nu for cem_mpc.py:68 — shape [act_dim]."""
    return _normals(seed, act_dim, np.uint32(0), np.uint32(0),
                    np.uint32(state_index | (STREAM_FINAL << 28)))


def dropout_keep(seed, iteration, member, layer, rows, units, rate):
    """Dropout keep mask of the trainer (csrc/train_common.cuh): [rows, units] bool, keep = u >= rate with
    u = uniform_from_bits(philox(column block j, batch row r, iteration, member | layer << 8 | 4 << 28))."""
    nblk = (units + 3) // 4
    ctr = np.empty((rows, nblk, 4), dtype=np.uint32)
    ctr[..., 0] = np.arange(nblk, dtype=np.uint32)[None, :]
    ctr[..., 1] = np.arange(rows, dtype=np.uint32)[:, None]
    ctr[..., 2] = np.uint32(iteration)
    ctr[..., 3] = np.uint32(member | (layer << 8) | (STREAM_DROPOUT << 28))
    u = uniform_from_bits(philox4x32(ctr, _key(seed)))
    return (u >= np.float32(rate)).reshape(rows, nblk * 4)[:, :units]
