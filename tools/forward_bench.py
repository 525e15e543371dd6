#!/usr/bin/env python
"""The ensemble's forward pass (MlpEnsemble.forward / __call__) on the bf16 tensor-core kernels against the fp32
kernel: simba_ensemble_forward_tc against simba_ensemble_forward, mean and variance only (no sample).

Shapes:
  c1        C1 model (E=5, L=4x128, O=60, A=2) over 10^6 rows
  c5        C5 model (E=10, L=4x400, O=60, A=2) over 10^6 rows
  c1-o92    the goal + four constrained lidars layout (O = 92) at C1 dims over 10^6 rows

Each case reports rows/s, the algorithmic TFLOP/s (synthetic.flops_per_transition x B over the call time), the kernel
the call chose and the GPU's name, SM count and power limit, read in the same run. The two precisions alternate call
by call in one process, each timed with CUDA events around the C entry point on the current stream, so a call
includes what a caller pays besides the kernel: the tile-list upload (after a device synchronise) and the launch. A
256 MB buffer is overwritten before every timed call, so no call starts with the previous call's data in L2.

  python tools/forward_bench.py [--out results.json] [--steps K]
"""
import argparse
import ctypes as C
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, 'ethz-safe-learning_b200')]

import numpy as np  # noqa: E402

from tools.obs_width_bench import LAYOUTS, gpu_info  # noqa: E402

CASES = {                  # name: (config, sensors, batch)
    'c1': ('c1', None, 10 ** 6),
    'c5': ('c5', None, 10 ** 6),
    'c1-o92': ('c1', LAYOUTS[92], 10 ** 6),
}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--out', help='also write the JSON result to this file')
    ap.add_argument('--steps', type=int, default=20, help='timed calls per case and precision')
    args = ap.parse_args()
    import torch
    from simba_b200 import _lib, synthetic
    assert torch.cuda.is_available(), "this benchmark needs a GPU"
    lib = _lib.load()
    names = {getattr(_lib, k): k[len('ROLLOUT_'):] for k in dir(_lib) if k.startswith('ROLLOUT_')}
    flush = torch.empty(64 * 2 ** 20, dtype=torch.int32, device='cuda')
    result = {"gpu": gpu_info(torch), "cases": []}
    entries = (('bf16', lib.simba_ensemble_forward_tc), ('fp32', lib.simba_ensemble_forward))
    for name, (cfg, sensors, B) in CASES.items():
        c = synthetic.make_workload(cfg, sensors=sensors)
        O, A = c['O'], c['A']
        ens = synthetic.build_policy(c, 'penalty', precision='fp32').model.model
        h = ens._ensure_handle()
        rng = np.random.default_rng(1)
        x = torch.from_numpy(rng.uniform(0, 1, (B, O + A)).astype(np.float32)).cuda()
        mu = {p: torch.empty((B, O), dtype=torch.float32, device='cuda') for p, _ in entries}
        var = {p: torch.empty((B, O), dtype=torch.float32, device='cuda') for p, _ in entries}
        kernel, items = C.c_int32(-1), C.c_int32(-1)
        _lib.check(lib.simba_ensemble_forward_tc_kernel(h, B, C.byref(kernel), C.byref(items)))
        stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)

        def call(p, entry):
            _lib.check(entry(h, C.c_void_p(x.data_ptr()), None, B, C.c_void_p(mu[p].data_ptr()),
                             C.c_void_p(var[p].data_ptr()), None, stream))
        for _ in range(3):
            for p, entry in entries:
                call(p, entry)
        torch.cuda.synchronize()
        ev = {p: [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))
                  for _ in range(args.steps)] for p, _ in entries}
        for k in range(args.steps):
            for p, entry in entries:
                flush.fill_(k & 0xff)
                ev[p][k][0].record()
                call(p, entry)
                ev[p][k][1].record()
        torch.cuda.synchronize()
        flops = synthetic.flops_per_transition(O, A, c['L'], c['U']) * B
        for p, _ in entries:
            ms = np.array([a.elapsed_time(b) for a, b in ev[p]])
            case = {"case": name, "precision": p, "E": c['E'], "L": c['L'], "U": c['U'], "O": O, "A": A, "batch": B,
                    "kernel": names.get(kernel.value, kernel.value) if p == 'bf16' else 'FP32',
                    "work_items": items.value if p == 'bf16' else None,
                    "ms_per_call": float(ms.mean()), "ms_min": float(ms.min()), "ms_max": float(ms.max()),
                    "calls": args.steps, "rows_per_s": B * 1e3 / float(ms.mean()),
                    "algorithmic_tflops": flops / (float(ms.mean()) * 1e-3) / 1e12}
            if p == 'bf16':
                dm = (mu['bf16'] - mu['fp32']).abs()
                dv = (var['bf16'] - var['fp32']).abs()
                case["vs_fp32"] = {"mu_max_abs": float(dm.max()), "mu_mean_abs": float(dm.mean()),
                                   "var_max_rel": float((dv / var['fp32']).max()),
                                   "var_mean_rel": float((dv / var['fp32']).mean())}
            print(json.dumps(case), flush=True)
            result["cases"].append(case)
        del ens
    by = {(r["case"], r["precision"]): r for r in result["cases"]}
    result["bf16_over_fp32"] = {n: by[(n, 'bf16')]["rows_per_s"] / by[(n, 'fp32')]["rows_per_s"] for n in CASES}
    text = json.dumps(result, indent=1)
    print(text)
    if args.out:
        with open(args.out, 'w') as f:
            f.write(text + '\n')


if __name__ == '__main__':
    main()
