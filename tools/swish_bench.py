#!/usr/bin/env python
"""What a swish ensemble costs against a ReLU ensemble of the same shape, in both precisions, measured in one run.

Planning: whole SafeCemMpc plans (simba_plan, one CUDA graph per plan, device Philox draws), plans/s (states planned
per second) at
  c1        C1 dims (E=5, L=4x128, O=60, A=2, N=150, P=20, I=5, H=15), one state per plan
  c1-256    the same with 256 states per plan
  c5        C5 dims (E=10, L=4x400), one state per plan
Training: simba_trainer_fit steps/s at C1 and C5 (batch 64, 800 steps per timed call).
The two activations alternate call by call in one process, each call timed with CUDA events after warm-up calls of
the same shape. Also recorded: the bf16 swish errors of the rollout rows (mean |d return| against the oracle at C1)
and of the forward pass (normwise mu error) that tests/test_gpu_swish.py bounds, and the GPU's name, SM count and
power limit, read in the same run.

  python tools/swish_bench.py [--out profiles/r09_swish_bench.json]
"""
import argparse
import ctypes as C
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, 'ethz-safe-learning_b200')]

import numpy as np  # noqa: E402

from tools.obs_width_bench import gpu_info  # noqa: E402
from tools.train_tc_bench import CONFIGS as TRAIN_CONFIGS, dynamics  # noqa: E402

ACTS = {'relu': 'tf.nn.relu', 'swish': 'tf.nn.swish'}
PLAN_CASES = [('c1', 'c1', 1), ('c1-256', 'c1', 256), ('c5', 'c5', 1)]


def time_alternating(torch, calls, steps, warmup):
    """calls: {key: fn} -> {key: [ms per call]}, the keys alternating call by call"""
    for _ in range(warmup):
        for fn in calls.values():
            fn()
    torch.cuda.synchronize()
    ev = {k: [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
          for k in calls}
    for i in range(steps):
        for k, fn in calls.items():
            ev[k][i][0].record()
            fn()
            ev[k][i][1].record()
    torch.cuda.synchronize()
    return {k: [a.elapsed_time(b) for a, b in ev[k]] for k in calls}


def plans(torch, steps, warmup):
    from simba_b200 import _lib, synthetic
    lib = _lib.load()
    names = {getattr(_lib, k): k[len('ROLLOUT_'):] for k in dir(_lib) if k.startswith('ROLLOUT_')}
    out = []
    for name, cfg, S in PLAN_CASES:
        c = synthetic.make_workload(cfg, S=S)
        states = torch.from_numpy(np.ascontiguousarray(np.asarray(c['state'], np.float32).reshape(S, c['O']))).cuda()
        for precision in ('bf16', 'fp32'):
            pols = {a: synthetic.build_policy(c, 'penalty', precision=precision, seed=3, activation=spelling)
                    for a, spelling in ACTS.items()}
            n = steps if S == 1 else max(steps // 5, 3)
            ms = time_alternating(torch, {a: (lambda p=p: p.plan_device(states)) for a, p in pols.items()}, n, warmup)
            case = {"case": name, "precision": precision, "states": S, "E": c['E'], "L": c['L'], "U": c['U'],
                    "H": c['H'], "N": c['N'], "P": c['P'], "I": c['I'], "plans": n}
            for a, p in pols.items():
                kernel, items = C.c_int32(-1), C.c_int32(-1)
                _lib.check(lib.simba_planner_rollout_kernel(p._ensure_planner(), C.byref(kernel), C.byref(items)))
                m = float(np.mean(ms[a]))
                case[a] = {"rollout_kernel": names.get(kernel.value, kernel.value), "work_items": items.value,
                           "ms_per_plan": m, "ms_min": float(np.min(ms[a])), "ms_max": float(np.max(ms[a])),
                           "plans_per_s": S * 1e3 / m}
            case["swish_over_relu_time"] = case['swish']['ms_per_plan'] / case['relu']['ms_per_plan']
            print(json.dumps(case), flush=True)
            out.append(case)
            del pols
    return out


def fits(torch, steps, repeats):
    from simba_b200 import _device, _lib
    from simba_b200.models import MlpEnsemble
    lib = _lib.load()
    out = []
    rng = np.random.default_rng(10)
    for name, cfg in TRAIN_CONFIGS.items():
        E, O, A, L, U = cfg['E'], cfg['O'], cfg['A'], cfg['L'], cfg['U']
        x, y = dynamics(rng, 20000, O, A)
        rs = np.random.RandomState(5)
        index = np.stack([np.stack([rs.randint(0, x.shape[0], 64) for _ in range(E)]) for _ in range(steps)])
        dx, _ = _device.to_device(x)
        dy, _ = _device.to_device(y)
        di, _ = _device.to_device(index.astype(np.int32), dtype=torch.int32)
        losses = torch.empty((steps,), dtype=torch.float32, device='cuda')
        for precision in ('bf16', 'fp32'):
            trainers = {}
            for a, spelling in ACTS.items():
                ens = MlpEnsemble(O + A, O, E, batch_size=64, learning_rate=1e-3, learning_rate_schedule=False,
                                  training_steps=steps, mlp_params=dict(n_layers=L, units=U, activation=spelling),
                                  seed=5, train_precision=precision)
                trainers[a] = (ens, ens._ensure_trainer())

            def fit(t):
                _lib.check(lib.simba_trainer_fit(t, _device.ptr(dx), _device.ptr(dy), x.shape[0], _device.ptr(di),
                                                 None, steps, _device.ptr(losses), _device.stream_ptr()))
            ms = time_alternating(torch, {a: (lambda t=t: fit(t)) for a, (_, t) in trainers.items()}, repeats, 1)
            case = {"case": name, "precision": precision, "E": E, "L": L, "U": U, "batch": 64,
                    "steps_per_call": steps, "calls": repeats}
            for a in trainers:
                med = float(np.median(ms[a]))
                case[a] = {"ms_per_call": sorted(ms[a]), "steps_per_s": steps * 1e3 / med}
            case["swish_over_relu_time"] = case['relu']['steps_per_s'] / case['swish']['steps_per_s']
            print(json.dumps(case), flush=True)
            out.append(case)
            del trainers
    return out


def bf16_errors(torch):
    """The bf16 swish rollout rows against the oracle (C1, external draws) and the bf16 forward pass against the
    float64 oracle: what tests/test_gpu_swish.py bounds."""
    from simba_b200 import _lib, synthetic
    from tests import helpers, swish_ref
    from tests.test_gpu_kernels import _oracle_rows
    from tests.test_gpu_swish import FORWARD_CASES, _draws, _ensemble, _oracle, _rows
    from tests.test_gpu_tc_obs_wide import SENSORS
    lib = _lib.load()
    out = {}
    for cfg in ('c1', 'c5'):
        c = synthetic.make_workload(cfg)
        acts, eps = _draws(c)
        ret = {}
        for precision in ('bf16', 'fp32'):
            pol = synthetic.build_policy(c, 'penalty', precision=precision, activation=ACTS['swish'])
            ret[precision], _, _ = _rows(pol, c, acts, eps)
        _, cum0, _, _ = _oracle_rows(c, _oracle(c), acts, eps, 'penalty')
        out['rows_%s' % cfg] = {p: {"mean_abs_dreturn": float(np.abs(r - cum0).mean()),
                                    "max_abs_dreturn": float(np.abs(r - cum0).max())} for p, r in ret.items()}
    for name, (cfg, sensors, over, per_member, _) in FORWARD_CASES.items():
        c = helpers.workload(cfg, sensors=SENSORS[sensors] if sensors else None, var_bias=-2.0, **over)
        O, A, B = c['O'], c['A'], c['E'] * per_member
        rng = np.random.default_rng(21)
        x = rng.uniform(0, 1, (B, O + A)).astype(np.float32)
        x[:, O:] = rng.uniform(-1, 1, (B, A))
        ens = _ensemble(c)
        mu = torch.empty((B, O), dtype=torch.float32, device='cuda')
        var = torch.empty_like(mu)
        xd = torch.from_numpy(x).cuda()
        _lib.check(lib.simba_ensemble_forward_tc(ens._ensure_handle(), C.c_void_p(xd.data_ptr()), None, B,
                                                 C.c_void_p(mu.data_ptr()), C.c_void_p(var.data_ptr()), None, None))
        torch.cuda.synchronize()
        ref_mu, ref_var = swish_ref.MlpEnsemble(c['weights'], dtype=np.float64).forward(x.astype(np.float64))
        m, v = mu.cpu().numpy(), var.cpu().numpy()
        out['forward_%s' % name] = {"mu_max_rel": float(np.abs(m - ref_mu).max() / np.abs(ref_mu).max()),
                                    "mu_mean_rel": float(np.abs(m - ref_mu).mean() / np.abs(ref_mu).mean()),
                                    "var_max_rel": float(np.abs(v - ref_var).max() / np.abs(ref_var).max())}
    print(json.dumps(out), flush=True)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--out', help='also write the JSON result to this file')
    ap.add_argument('--steps', type=int, default=20, help='timed plans per case and activation')
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--fit-steps', type=int, default=800)
    ap.add_argument('--fit-repeats', type=int, default=5)
    args = ap.parse_args()
    import torch
    assert torch.cuda.is_available(), "this benchmark needs a GPU"
    result = {"gpu": gpu_info(torch), "plans": plans(torch, args.steps, args.warmup),
              "fit": fits(torch, args.fit_steps, args.fit_repeats), "bf16_errors": bf16_errors(torch)}
    result["gpu_after"] = gpu_info(torch)
    text = json.dumps(result, indent=1)
    print(text)
    if args.out:
        with open(args.out, 'w') as f:
            f.write(text + '\n')


if __name__ == '__main__':
    main()
