#!/usr/bin/env python
"""Model rollouts (TransitionModel.unfold_sequences / predict) on the bf16 tensor-core kernels against the fp32
kernel: simba_unfold_tc against simba_unfold, Philox noise, sampling propagation on.

Shapes:
  c1          C1 model (E=5, L=4x128, O=60, A=2), B = 3000 rows, H = 15
  c1-predict  predict (H = 1) on the C1 model over 10^6 rows
  c5          C5 model (E=10, L=4x400), B = 3000, H = 50
  c1-o92      the goal + four constrained lidars layout (O = 92) at C1 dims, B = 3000, H = 15

Each case reports rows/s, the algorithmic TFLOP/s (synthetic.flops_per_transition x B x H over the call time), the
bytes of trajectory written, the kernel the call chose and the GPU's name, SM count and power limit, read in the
same run. A call is timed with CUDA events around the C entry point on the current stream, so it includes what a
caller pays besides the kernel: the tile-list upload (after a device synchronise) and the launch. A 256 MB buffer is
overwritten before every timed call, so no call starts with the previous call's data in L2.

  python tools/unfold_bench.py [--out results.json] [--steps K]
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

CASES = {                  # name: (config, sensors, batch, horizon)
    'c1': ('c1', None, 3000, 15),
    'c1-predict': ('c1', None, 10 ** 6, 1),
    'c5': ('c5', None, 3000, 50),
    'c1-o92': ('c1', LAYOUTS[92], 3000, 15),
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
    for name, (cfg, sensors, B, H) in CASES.items():
        c = synthetic.make_workload(cfg, sensors=sensors)
        O, A = c['O'], c['A']
        tm = synthetic.build_policy(c, 'penalty', precision='fp32').model
        h = tm.model._ensure_handle()
        rng = np.random.default_rng(1)
        s0 = torch.from_numpy(np.tile(c['state'], (B, 1)).astype(np.float32)).cuda()
        acts = torch.from_numpy(rng.uniform(-1, 1, (B, H, A)).astype(np.float32)).cuda()
        out = torch.empty((B, H + 1, O), dtype=torch.float32, device='cuda')
        kernel, items = C.c_int32(-1), C.c_int32(-1)
        _lib.check(lib.simba_unfold_tc_kernel(h, B, H, C.byref(kernel), C.byref(items)))
        stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)
        outs = {}
        for precision, entry in (('bf16', lib.simba_unfold_tc), ('fp32', lib.simba_unfold)):
            def call(k):
                _lib.check(entry(h, C.c_void_p(s0.data_ptr()), C.c_void_p(acts.data_ptr()), None, 17 + k, B, H, 1,
                                 C.c_void_p(out.data_ptr()), stream))
            for k in range(3):
                call(k)
            torch.cuda.synchronize()
            ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))
                  for _ in range(args.steps)]
            for k in range(args.steps):
                flush.fill_(k & 0xff)
                ev[k][0].record()
                call(k)
                ev[k][1].record()
            torch.cuda.synchronize()
            outs[precision] = out[:, -1].clone()
            ms = np.array([a.elapsed_time(b) for a, b in ev])
            flops = synthetic.flops_per_transition(O, A, c['L'], c['U']) * B * H
            case = {"case": name, "precision": precision, "E": c['E'], "L": c['L'], "U": c['U'], "O": O, "A": A,
                    "batch": B, "horizon": H,
                    "kernel": names.get(kernel.value, kernel.value) if precision == 'bf16' else 'FP32',
                    "work_items": items.value if precision == 'bf16' else None,
                    "ms_per_call": float(ms.mean()), "ms_min": float(ms.min()), "ms_max": float(ms.max()),
                    "calls": args.steps, "rows_per_s": B * 1e3 / float(ms.mean()),
                    "algorithmic_tflops": flops / (float(ms.mean()) * 1e-3) / 1e12,
                    "bytes_written": B * (H + 1) * O * 4,
                    "write_gb_per_s": B * (H + 1) * O * 4 / (float(ms.mean()) * 1e-3) / 1e9}
            print(json.dumps(case), flush=True)
            result["cases"].append(case)
        d = (outs['bf16'] - outs['fp32']).abs()
        result["cases"][-2]["last_state_vs_fp32"] = {"max_abs": float(d.max()), "mean_abs": float(d.mean())}
        del tm
    by = {(r["case"], r["precision"]): r for r in result["cases"]}
    result["bf16_over_fp32"] = {n: by[(n, 'bf16')]["rows_per_s"] / by[(n, 'fp32')]["rows_per_s"] for n in CASES}
    text = json.dumps(result, indent=1)
    print(text)
    if args.out:
        with open(args.out, 'w') as f:
            f.write(text + '\n')


if __name__ == '__main__':
    main()
