#!/usr/bin/env python
"""What the MPPI update costs against CEM's selection and refit, in both precisions, measured in one run.

Planning: whole SafeMppiMpc and SafeCemMpc plans (penalty objective, simba_plan, one CUDA graph per plan, device
Philox draws), plans/s (states planned per second) at
  c1        C1 dims (E=5, L=4x128, O=60, A=2, N=150, P=20, I=5, H=15), one state per plan
  c1-256    the same with 256 states per plan
  c5        C5 dims (E=10, L=4x400, H=50), one state per plan
  n65536    configs[2] dims (H=30, N=65536, P=32, member_map 'particle') on one GPU: the separate update kernels
The two rules alternate call by call in one process, each call timed with CUDA events after warm-up calls.
Update kernel: the time of one iteration's update, CUDA events around 50 launches on the plan's own pairs and
actions: simba_mppi_update (mppi_refit_kernel) against simba_select_elites + simba_refit. At N <= 1024 a plan fuses
either update with the reduction and the next sampling, so this is the separate kernels' time.
Also recorded: bf16 against fp32 MPPI plans on the same external draws (max |d mu|, |d action|, |d score|) at C1
and C5, which tests/test_gpu_mppi.py bounds, and the GPU's name, SM count and power limit, read in the same run.

  python tools/mppi_bench.py [--out profiles/r10_mppi_bench.json]
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
from tools.swish_bench import time_alternating  # noqa: E402

TEMPERATURE = 0.5
PLAN_CASES = [('c1', 'c1', 1, {}), ('c1-256', 'c1', 256, {}), ('c5', 'c5', 1, {}),
              ('n65536', 'c3', 1, dict(member_map='particle'))]


def _policy(c, rule, precision, **kw):
    from simba_b200 import synthetic
    if rule == 'mppi':
        kw['temperature'] = TEMPERATURE
    return synthetic.build_policy(c, 'penalty', precision=precision, seed=3, **kw)


def update_ms(torch, lib, pols, c, S, launches=50):
    """ms per launch of each rule's separate update kernels on the plan's own buffers (scratch mu / best copies)."""
    from simba_b200 import _lib
    out = {}
    for rule, p in pols.items():
        h = p._ensure_planner()
        pairs, acts = p.buffer(_lib.BUF_PAIRS_LOCAL), p.buffer(_lib.BUF_ACTIONS)
        mu, sigma = p.buffer(_lib.BUF_MU), p.buffer(_lib.BUF_SIGMA)
        best_a, best_s = p.buffer(_lib.BUF_BEST_ACTION), p.buffer(_lib.BUF_BEST_SCORE)
        elite = torch.empty((S * c['K'],), dtype=torch.int32, device='cuda')
        if rule == 'mppi':
            def call():
                _lib.check(lib.simba_mppi_update(h, pairs.data_ptr(), acts.data_ptr(), None, mu.data_ptr(),
                                                 best_a.data_ptr(), best_s.data_ptr(), None))
        else:
            def call():
                _lib.check(lib.simba_select_elites(h, pairs.data_ptr(), acts.data_ptr(), None, elite.data_ptr(), None,
                                                   best_a.data_ptr(), best_s.data_ptr(), None))
                _lib.check(lib.simba_refit(h, acts.data_ptr(), elite.data_ptr(), mu.data_ptr(), sigma.data_ptr(),
                                           None, None, None))
        for _ in range(5):
            call()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(launches):
            call()
        b.record()
        torch.cuda.synchronize()
        out[rule] = a.elapsed_time(b) / launches
    return out


def plans(torch, steps, warmup):
    from simba_b200 import _lib, synthetic
    lib = _lib.load()
    out = []
    for name, cfg, S, kw in PLAN_CASES:
        c = synthetic.make_workload(cfg, S=S)
        states = torch.from_numpy(np.ascontiguousarray(np.asarray(c['state'], np.float32).reshape(S, c['O']))).cuda()
        for precision in ('bf16', 'fp32'):
            pols = {r: _policy(c, r, precision, **kw) for r in ('mppi', 'cem')}
            n = (steps if S == 1 else max(steps // 5, 3)) if c['N'] <= 1024 else 2
            w = warmup if c['N'] <= 1024 else 1
            ms = time_alternating(torch, {r: (lambda p=p: p.plan_device(states)) for r, p in pols.items()}, n, w)
            case = {"case": name, "precision": precision, "states": S, "E": c['E'], "L": c['L'], "U": c['U'],
                    "H": c['H'], "N": c['N'], "P": c['P'], "I": c['I'], "K_cem": c['K'], "plans": n,
                    "temperature": TEMPERATURE}
            upd = update_ms(torch, lib, pols, c, S)
            for r, p in pols.items():
                m = float(np.mean(ms[r]))
                case[r] = {"launches_per_plan": p.launches_per_plan, "ms_per_plan": m, "ms_min": float(np.min(ms[r])),
                           "ms_max": float(np.max(ms[r])), "plans_per_s": S * 1e3 / m,
                           "separate_update_ms_per_iteration": upd[r]}
            case["mppi_over_cem_time"] = case['mppi']['ms_per_plan'] / case['cem']['ms_per_plan']
            print(json.dumps(case), flush=True)
            out.append(case)
            del pols
    return out


def bf16_errors():
    from simba_b200 import _lib, synthetic
    out = {}
    for cfg in ('c1', 'c5'):
        c = synthetic.make_workload(cfg)
        z, eps, zf = synthetic.make_draws(c['I'], 1, c['N'], c['H'], c['A'], c['P'], c['O'])
        got = {}
        for precision in ('bf16', 'fp32'):
            p = _policy(c, 'mppi', precision)
            p.set_external_draws(z, eps, zf)
            a, s = p.do_generate_action(c['state'])
            got[precision] = (np.asarray(a), np.asarray(s), p.buffer(_lib.BUF_MU).cpu().numpy())
        b, f = got['bf16'], got['fp32']
        out[cfg] = {"max_abs_dmu": float(np.abs(b[2] - f[2]).max()), "max_abs_daction": float(np.abs(b[0] - f[0]).max()),
                    "abs_dscore": float(np.abs(b[1] - f[1]).max()), "fp32_score": float(f[1])}
        print(json.dumps({cfg: out[cfg]}), flush=True)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--out', help='also write the JSON result to this file')
    ap.add_argument('--steps', type=int, default=20, help='timed plans per case and rule (fewer for large cases)')
    ap.add_argument('--warmup', type=int, default=3)
    args = ap.parse_args()
    import torch
    assert torch.cuda.is_available(), "this benchmark needs a GPU"
    result = {"gpu": gpu_info(torch), "bf16_errors": bf16_errors(), "plans": plans(torch, args.steps, args.warmup)}
    result["gpu_after"] = gpu_info(torch)
    text = json.dumps(result, indent=1)
    print(text)
    if args.out:
        with open(args.out, 'w') as f:
            f.write(text + '\n')


if __name__ == '__main__':
    main()
