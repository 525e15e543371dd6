#!/usr/bin/env python
"""Planning throughput across horizons, in both precisions: whole SafeCemMpc plans (simba_plan, one CUDA graph per
plan, device Philox draws) at horizons on both sides of 64 steps, where the per-row cost history grows from one
64-bit plane to several.

Shapes:
  c1        C1 dims (E=5, L=4x128, O=60, A=2, N=150, P=20, I=5), one state per plan, H in {15, 64, 65, 128, 256}
  c1-256    the same with 256 states per plan
  c5        C5 dims (E=10, L=4x400), one state per plan, H in {50, 100}

Each case reports plans/s (states planned per second), the rollout kernel, the update path the plan took (fused:
one update kernel per iteration; separate: reduce, select and refit kernels) with its launch count, and the GPU's
name, SM count and power limit, read in the same run. The two precisions alternate plan by plan in one process, each
plan timed with CUDA events on the current stream after warm-up plans of the same shape.

  python tools/long_horizon_bench.py [--out profiles/r08_long_horizon_bench.json] [--steps K]
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

CASES = [('c1', 'c1', 1, H) for H in (15, 64, 65, 128, 256)] + \
        [('c1-256', 'c1', 256, H) for H in (15, 64, 65, 128, 256)] + \
        [('c5', 'c5', 1, H) for H in (50, 100)]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--out', help='also write the JSON result to this file')
    ap.add_argument('--steps', type=int, default=20, help='timed plans per case and precision')
    ap.add_argument('--warmup', type=int, default=3)
    args = ap.parse_args()
    import torch
    from simba_b200 import _lib, synthetic
    assert torch.cuda.is_available(), "this benchmark needs a GPU"
    lib = _lib.load()
    names = {getattr(_lib, k): k[len('ROLLOUT_'):] for k in dir(_lib) if k.startswith('ROLLOUT_')}
    result = {"gpu": gpu_info(torch), "cases": []}
    precisions = ('bf16', 'fp32')
    for name, cfg, S, H in CASES:
        c = synthetic.make_workload(cfg, S=S, H=H)
        pols = {p: synthetic.build_policy(c, 'penalty', precision=p, seed=3) for p in precisions}
        states = torch.from_numpy(np.ascontiguousarray(np.asarray(c['state'], np.float32).reshape(S, c['O']))).cuda()
        for _ in range(args.warmup):
            for p in precisions:
                pols[p].plan_device(states)
        torch.cuda.synchronize()
        ev = {p: [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))
                  for _ in range(args.steps)] for p in precisions}
        for k in range(args.steps):
            for p in precisions:
                ev[p][k][0].record()
                pols[p].plan_device(states)
                ev[p][k][1].record()
        torch.cuda.synchronize()
        for p in precisions:
            ms = np.array([a.elapsed_time(b) for a, b in ev[p]])
            kernel, items = C.c_int32(-1), C.c_int32(-1)
            _lib.check(lib.simba_planner_rollout_kernel(pols[p]._ensure_planner(), C.byref(kernel), C.byref(items)))
            launches = pols[p].launches_per_plan
            case = {"case": name, "precision": p, "H": H, "states": S, "E": c['E'], "L": c['L'], "U": c['U'],
                    "N": c['N'], "P": c['P'], "I": c['I'], "cost_mask_planes": (H + 63) // 64,
                    "rollout_kernel": names.get(kernel.value, kernel.value), "work_items": items.value,
                    "update_path": "fused" if launches == 1 + 2 * c['I'] else "separate",
                    "launches_per_plan": launches,
                    "ms_per_plan": float(ms.mean()), "ms_min": float(ms.min()), "ms_max": float(ms.max()),
                    "plans": args.steps, "plans_per_s": S * 1e3 / float(ms.mean())}
            print(json.dumps(case), flush=True)
            result["cases"].append(case)
        del pols
    text = json.dumps(result, indent=1)
    print(text)
    if args.out:
        with open(args.out, 'w') as f:
            f.write(text + '\n')


if __name__ == '__main__':
    main()
