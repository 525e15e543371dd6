#!/usr/bin/env python
"""Planning throughput against observation width: C1 dims (E=5, L=4x128, A=2, H=15, N=150, P=20, I=5) at
obs_dim 60, 76, 92 and 124, one and 256 states per call, bf16 and fp32.

The observation is a goal task with 16-bin lidars: PointGoal1's 60 dims (goal, hazards, vases), goal + hazards,
pillars and vases (76), goal + all four constrained classes (92), and the 92 plus 32 more robot dims (124). Every
observed lidar class is constrained. For each case the script reports plans/s, the algorithmic TFLOP/s of the call
(synthetic.flops_per_transition x I x H x P x N x S over the CUDA-event time of the call) and the rollout kernel
the planner chose, with the GPU's name and power limit read in the same run. A 256 MB buffer is overwritten
before every timed call, so no call starts with the previous call's data in L2.

  python tools/obs_width_bench.py [--out results.json] [--steps K]
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, 'ethz-safe-learning_b200')]

import numpy as np  # noqa: E402

ROBOT = dict(accelerometer=3, gyro=3, magnetometer=3, velocimeter=3)
LAYOUTS = {
    60: dict(ROBOT, goal_lidar=16, hazards_lidar=16, vases_lidar=16),
    76: dict(ROBOT, goal_lidar=16, hazards_lidar=16, pillars_lidar=16, vases_lidar=16),
    92: dict(ROBOT, goal_lidar=16, gremlins_lidar=16, hazards_lidar=16, pillars_lidar=16, vases_lidar=16),
    124: dict(ROBOT, goal_lidar=16, gremlins_lidar=16, hazards_lidar=16, pillars_lidar=16, vases_lidar=16, joints=32),
}


def gpu_info(torch):
    info = {"name": torch.cuda.get_device_name(0), "sms": torch.cuda.get_device_properties(0).multi_processor_count}
    try:
        out = subprocess.check_output(["nvidia-smi", "-i", "0", "--query-gpu=power.limit,clocks.max.sm",
                                       "--format=csv,noheader"], timeout=20).decode().strip()
        info["power_limit"], info["max_sm_clock"] = [x.strip() for x in out.split(',')]
    except Exception as e:                                      # reported, not guessed
        info["power_limit"] = "unavailable (%s)" % e
    return info


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--out', help='also write the JSON result to this file')
    ap.add_argument('--steps', type=int, default=10, help='timed calls per case (at 256 states: a fifth of it)')
    args = ap.parse_args()
    import torch
    from simba_b200 import _lib, synthetic
    assert torch.cuda.is_available(), "this benchmark needs a GPU"
    names = {getattr(_lib, k): k[len('ROLLOUT_'):] for k in dir(_lib) if k.startswith('ROLLOUT_')}
    flush = torch.empty(64 * 2 ** 20, dtype=torch.int32, device='cuda')
    result = {"gpu": gpu_info(torch), "cases": []}
    for O, sensors in LAYOUTS.items():
        scorer = {'constrain_' + k[:-len('_lidar')]: True for k in sensors if k.endswith('_lidar') and k != 'goal_lidar'}
        for S in (1, 256):
            for precision in ('bf16', 'fp32'):
                c = synthetic.make_workload('c1', sensors=sensors, S=S)
                assert c['O'] == O
                pol = synthetic.build_policy(c, 'penalty', precision=precision, scorer_config=scorer, seed=7)
                kernel, items = C.c_int32(-1), C.c_int32(-1)
                _lib.check(_lib.load().simba_planner_rollout_kernel(pol._ensure_planner(), C.byref(kernel),
                                                                     C.byref(items)))
                st = torch.from_numpy(synthetic.make_state(sensors, seed=500, n_states=S).reshape(S, -1)).cuda()
                for _ in range(2):
                    pol.plan_device(st)
                torch.cuda.synchronize()
                K = max(2, args.steps // 5) if S > 1 else args.steps
                ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(K)]
                for k in range(K):
                    flush.fill_(k & 0xff)
                    ev[k][0].record()
                    pol.plan_device(st)
                    ev[k][1].record()
                torch.cuda.synchronize()
                ms = np.array([a.elapsed_time(b) for a, b in ev])
                flops = synthetic.flops_per_transition(O, c['A'], c['L'], c['U']) * c['I'] * c['H'] * c['P'] * c['N'] * S
                case = {"obs_dim": O, "states": S, "precision": precision, "constraints": len(scorer),
                        "rollout_kernel": names.get(kernel.value, kernel.value), "work_items": items.value,
                        "ms_per_call": float(ms.mean()), "ms_min": float(ms.min()), "ms_max": float(ms.max()),
                        "calls": K, "plans_per_s": S * 1e3 / float(ms.mean()),
                        "algorithmic_tflops": flops / (float(ms.mean()) * 1e-3) / 1e12}
                print(json.dumps(case), flush=True)
                result["cases"].append(case)
                del pol
    by = {(r["obs_dim"], r["states"], r["precision"]): r for r in result["cases"]}
    result["bf16_over_fp32"] = {"O=%d S=%d" % (O, S): by[(O, S, 'bf16')]["plans_per_s"] / by[(O, S, 'fp32')]["plans_per_s"]
                                for O in LAYOUTS for S in (1, 256)}
    text = json.dumps(result, indent=1)
    print(text)
    if args.out:
        with open(args.out, 'w') as f:
            f.write(text + '\n')


if __name__ == '__main__':
    main()
