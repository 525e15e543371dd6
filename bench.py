#!/usr/bin/env python
"""bench.py — CEM-MPC plans/sec + ensemble transitions/sec at the PointGoal1 shape (BASELINE.json).

  python bench.py --gpus N --steps K --warmup W            # this repo's CUDA planner
  python bench.py --impl reference --gpus N --steps K ...  # the reference's CPU planner (oracle port)
  python bench.py ... --dump-outputs bench_outputs         # also save the last timed plan's outputs (.npy)

A "step" is ONE planning call (policy.generate_action: 5 CEM iterations of sample -> fused ensemble
rollout + scoring -> score-reduce -> select -> refit) at BASELINE configs[1] (C1 dims: 5-member
4x128 ensemble, obs 60, act 2, horizon 15, population 150, 20 particles, 5 iterations, all of
which run: stddev_threshold = 0).
  value  = plans/sec with the state already in HBM, timed with CUDA events around each plan, L2
           flushed between plans, max over ranks.
  e2e    = plans/sec through policy.generate_action(numpy_state): host buffers in, host buffers
           out, H2D + D2H + synchronisation inside the timed region.
N > 1: one process per GPU (torchrun); every rank plans its own independent states (weak scaling,
no data-path collective — batched planning of BASELINE configs[3]); value = all ranks' plans / max
time. `--extras c3` adds the population-65536 plan sharded over the ranks with the per-iteration
NCCL all-gather (strong scaling) as extra keys.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
for _p in (ROOT, os.path.join(ROOT, 'ethz-safe-learning_b200')):
    if _p not in sys.path:
        sys.path.insert(0, _p)

import numpy as np  # noqa: E402

METRIC = "CEM-MPC plans/sec (PointGoal1 shape; ensemble transitions/sec alongside)"
UNIT = "plans/s"


def workload_config(c, precision, extra=None):
    cfg = {"workload": "BASELINE configs[1] (C1 dims): E=%d L=%dx%d O=%d A=%d H=%d N=%d P=%d I=%d K=%d, "
                       "SafeCemMpc penalty objective, stddev_threshold=0 (all iterations run)"
                       % (c['E'], c['L'], c['U'], c['O'], c['A'], c['H'], c['N'], c['P'], c['I'], c['K']),
           "rollout_precision": precision, "l2": "flushed between timed plans (256 MiB write)",
           "rng": "Philox4x32-10 on device"}
    cfg.update(extra or {})
    return cfg


# ------------------------------------------------------------------------------------------------
# clocks sampler (B200_PROFILING.md recipe)
# ------------------------------------------------------------------------------------------------
class ClockSampler(object):
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.stop_flag, self.th = index, [], False, None

    def _run_nvml(self):
        """In-process NVML polling (5 ms period) so that even a sub-second timed region is sampled
        many times; same fields as the nvidia-smi query."""
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(self.index)
        mx = pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM)
        bits = [("hw_slowdown", getattr(pynvml, 'nvmlClocksThrottleReasonHwSlowdown', 0x8)),
                ("hw_thermal_slowdown", getattr(pynvml, 'nvmlClocksThrottleReasonHwThermalSlowdown', 0x40)),
                ("sw_thermal_slowdown", getattr(pynvml, 'nvmlClocksThrottleReasonSwThermalSlowdown', 0x20)),
                ("sw_power_cap", getattr(pynvml, 'nvmlClocksThrottleReasonSwPowerCap', 0x4))]
        while not self.stop_flag:
            sm = pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM)
            try:
                mask = pynvml.nvmlDeviceGetCurrentClocksThrottleReasons(h)
            except Exception:
                mask = 0
            self.rows.append([str(sm), str(mx)] + ['Active' if mask & b else 'Not Active' for _, b in bits])
            time.sleep(0.005)

    def _run(self):
        try:
            self._run_nvml()
            return
        except Exception:
            pass
        while not self.stop_flag:
            try:
                out = subprocess.check_output(
                    ["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                     "--format=csv,noheader,nounits"], timeout=5).decode().strip()
                self.rows.append([x.strip() for x in out.split(',')])
            except Exception:
                pass
            time.sleep(0.1)

    def start(self):
        self.th = threading.Thread(target=self._run, daemon=True)
        self.th.start()

    def stop(self):
        self.stop_flag = True
        if self.th:
            self.th.join(timeout=6)
        sm = [float(r[0]) for r in self.rows if r and r[0].replace('.', '').isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) > 1 and r[1].replace('.', '').isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for r in self.rows if len(r) >= 6 for i in range(4)
                          if r[2 + i].lower().startswith('active')})
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm)}


# ------------------------------------------------------------------------------------------------
# CPU planner (the oracle port) — cpu_baseline leg and --impl reference
# ------------------------------------------------------------------------------------------------
def _cpu_planners(c, objective='penalty'):
    """The two CPU restatements of the reference planner (oracle/simba_oracle.py: numpy;
    oracle/torch_ref.py: torch-CPU, shaped like the reference) as plan(state, z, eps, zf) callables."""
    from oracle import simba_oracle as so           # the only product-side use: the CPU baseline
    from oracle import torch_ref
    from tests import helpers
    pn = helpers.oracle_planner(c, objective)
    cfg = dict(so.DEFAULT_SCORER_CONFIG)
    dyn = torch_ref.Dynamics(torch_ref.Ensemble(c['weights']), c['smin'], c['smax'], True, True)
    pt = torch_ref.Planner(dyn, torch_ref.GoalScorer(cfg, c['table']), [-1.0] * c['A'], [1.0] * c['A'], c['H'],
                           c['I'], 0.0, c['N'], c['K'], c['P'], 0.0, 0.01, posterior_mean_threashold=0.15,
                           objective=objective)
    return {"numpy": lambda st, z, eps, zf: pn.do_generate_action(st, z, eps, zf)[2],
            "torch": lambda st, z, eps, zf: pt.do_generate_action(st, z, eps, zf)[2]}


def time_cpu_planner(c, budget_s=20.0, max_plans=12, label="C1", steps=None, warmup=0):
    """Times the CPU restatements of the reference planner on this box's host cores: whole plans with
    the normal draws pre-generated outside the timed region. Both restatements (numpy and torch-CPU,
    cross-checked against each other and against fixtures produced by the unmodified reference code) get
    two plans each; the faster one is the baseline and gets the rest of the budget. With `steps`, the
    faster one instead runs `warmup` untimed plans and then exactly `steps` timed ones, with no budget."""
    from simba_b200 import synthetic
    z, eps, zf = synthetic.make_draws(c['I'], 1, c['N'], c['H'], c['A'], c['P'], c['O'], seed=2)
    z, eps, zf = z[:, 0], eps[:, 0], zf[0]
    try:
        # torchrun exports OMP_NUM_THREADS=1; the CPU planner is allowed every host thread it can use
        import threadpoolctl
        threadpoolctl.threadpool_limits(limits=os.cpu_count())
        import torch
        torch.set_num_threads(os.cpu_count())
    except Exception:
        pass
    planners = _cpu_planners(c)
    probe, n = {}, c['I']
    t_start = time.perf_counter()
    for name, fn in planners.items():
        fn(c['state'], z, eps, zf)                                          # warm-up (BLAS threads, pages)
        t0 = time.perf_counter()
        n = fn(c['state'], z, eps, zf)
        probe[name] = time.perf_counter() - t0
        if time.perf_counter() - t_start > budget_s and len(probe) == 1:  # very large workloads: one is enough
            break
    best_name = min(probe, key=probe.get)
    fn, times = planners[best_name], [probe[best_name]]
    if steps is not None:
        for _ in range(warmup):
            fn(c['state'], z, eps, zf)
        times, max_plans, budget_s = [], steps, float('inf')
    while len(times) < max_plans and time.perf_counter() - t_start < budget_s:
        t0 = time.perf_counter()
        n = fn(c['state'], z, eps, zf)
        times.append(time.perf_counter() - t0)
    best, med = min(times), float(np.median(times))
    try:
        import threadpoolctl
        threads = max([p.get('num_threads', 1) for p in threadpoolctl.threadpool_info()] or [1])
    except Exception:
        threads = os.cpu_count()
    return {"value": 1.0 / med, "unit": UNIT, "cores": int(threads), "kind": "port",
            "sample": "%d whole %s plans on the %s fp32 restatement of the TensorFlow reference (the faster of "
                      "the two restatements here: %s), threads=%d of %d host cpus; median %.1f ms, best %.1f ms per plan"
                      % (len(times), label, best_name,
                         ", ".join("%s %.0f ms" % (k, v * 1e3) for k, v in sorted(probe.items())), threads, os.cpu_count(),
                         med * 1e3, best * 1e3),
            "transitions_per_s": n * c['H'] * c['P'] * c['N'] / med, "ms_per_plan_median": med * 1e3}


def run_reference(args):
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    from simba_b200 import synthetic
    c = synthetic.make_workload('c1')
    cb = time_cpu_planner(c, steps=args.steps, warmup=args.warmup)
    line = {"impl": "reference", "metric": METRIC, "value": cb["value"], "unit": UNIT, "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": cb["ms_per_plan_median"],
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic (random-init ensemble, synthetic state; reference TensorFlow planner is not "
                    "installable here, so this is the oracle port on host cores)",
            "config": workload_config(c, "f32 (CPU)"), "cpu_baseline": cb, "gpu_launches": 0,
            "e2e": {"value": cb["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "transitions_per_s": cb["transitions_per_s"]}
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------------
# GPU arm
# ------------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=200)
    ap.add_argument('--warmup', type=int, default=10)
    ap.add_argument('--impl', default='b200', choices=['b200', 'reference'])
    ap.add_argument('--precision', default='bf16', choices=['bf16', 'fp32'])
    ap.add_argument('--extras', default=None, help="comma list of: c3, c4, c5, fp32, train, none (default: c3,c4 when N > 1, fp32,c4,c3,c5,train when N == 1)")
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--dump-outputs', metavar='DIR', default=None,
                    help="write what the last timed plan returned (device plan: action, score, iterations; "
                         "end to end: action) as DIR/<name>.npy in float32, for comparing two builds")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == 'reference':
        if args.dump_outputs:
            ap.error("--dump-outputs applies to the b200 arm")
        return run_reference(args)

    import torch
    import torch.distributed as dist
    from simba_b200 import _lib, synthetic
    import ctypes as C

    rank = int(os.environ.get('RANK', '0'))
    world = int(os.environ.get('WORLD_SIZE', '1'))
    local_rank = int(os.environ.get('LOCAL_RANK', '0'))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a B200: there is no CPU fallback (use --impl reference for the CPU planner)")
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group('nccl', device_id=torch.device('cuda', local_rank))
    lib = _lib.load()
    W, K = max(3, args.warmup), args.steps

    c = synthetic.make_workload('c1')
    precision = args.precision
    pol = synthetic.build_policy(c, 'penalty', precision=precision, seed=0x5EED + 1000 * rank)
    pol.build()                 # fails loudly if the requested precision is not offered for this shape
    n_pool = 16
    states_np = synthetic.make_state(c['sensors'], seed=100 + rank, n_states=n_pool)
    states = torch.from_numpy(states_np).cuda()
    flush = torch.empty(256 << 20, dtype=torch.uint8, device='cuda')
    out_a = torch.empty((1, c['A']), dtype=torch.float32, device='cuda')
    out_s = torch.empty((1,), dtype=torch.float32, device='cuda')
    out_i = torch.empty((1,), dtype=torch.int32, device='cuda')

    def sync_all():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    # ---- device-resident throughput --------------------------------------------------------------
    for k in range(W):
        pol.plan_device(states[k % n_pool:k % n_pool + 1], None, out_a, out_s, out_i)
    sync_all()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(K)]
    iters_total = 0
    sync_all()
    t_wall0 = time.perf_counter()
    for k in range(K):
        flush.fill_(k & 0xff)
        ev[k][0].record()
        pol.plan_device(states[k % n_pool:k % n_pool + 1], None, out_a, out_s, out_i)
        ev[k][1].record()
    sync_all()
    t_wall = time.perf_counter() - t_wall0
    ms = np.array([a.elapsed_time(b) for a, b in ev])
    last_plan = {"plan_action": out_a.cpu().numpy(), "plan_score": out_s.cpu().numpy(),
                 "plan_iterations": out_i.cpu().numpy()}
    iters_total = int(out_i.cpu()[0])
    t_rank = torch.tensor([ms.sum() / 1e3], dtype=torch.float64, device='cuda')
    if world > 1:
        dist.all_reduce(t_rank, op=dist.ReduceOp.MAX)
    t_dev = float(t_rank.cpu()[0])
    value = world * K / t_dev
    launches = pol.launches_per_plan * K

    # ---- end to end through the public API (host buffers) ----------------------------------------
    for k in range(W):
        pol.generate_action(states_np[k % n_pool])
    sync_all()
    t_e2e = 0.0
    for k in range(K):
        flush.fill_(k & 0xff)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        a = pol.generate_action(states_np[k % n_pool])
        t_e2e += time.perf_counter() - t0
    assert np.all(np.isfinite(a))
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, dict(last_plan, e2e_action=a), '_rank%d' % rank if world > 1 else '')
    t_e = torch.tensor([t_e2e], dtype=torch.float64, device='cuda')
    if world > 1:
        dist.all_reduce(t_e, op=dist.ReduceOp.MAX)
    e2e_value = world * K / float(t_e.cpu()[0])
    clocks = sampler.stop() if rank == 0 else None

    # ---- the dominant kernel alone: fused rollout, CUDA events on the launching stream -------------
    planner = pol._ensure_planner()
    B = c['P'] * c['N']
    acts = torch.empty((1, c['N'], c['H'], c['A']), dtype=torch.float32, device='cuda').uniform_(-1, 1)
    r_ret = torch.empty(B, dtype=torch.float32, device='cuda')
    r_msk = torch.empty(B, dtype=torch.int64, device='cuda')
    r_sum = torch.empty(B, dtype=torch.float32, device='cuda')
    st_ptr = C.c_void_p(torch.cuda.current_stream().cuda_stream)

    def rollout_once(it):
        _lib.check(lib.simba_rollout_score(planner, C.c_void_p(states.data_ptr()), C.c_void_p(acts.data_ptr()),
                                           None, 0x5EED, it, None, C.c_void_p(r_ret.data_ptr()),
                                           C.c_void_p(r_msk.data_ptr()), C.c_void_p(r_sum.data_ptr()), st_ptr))
    for it in range(5):
        rollout_once(it)
    torch.cuda.synchronize()
    n_roll = min(200, max(20, K))
    rev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(n_roll)]
    for k in range(n_roll):
        flush.fill_(k & 0xff)
        rev[k][0].record()
        rollout_once(k % c['I'])
        rev[k][1].record()
    torch.cuda.synchronize()
    roll_ms = float(np.mean([a.elapsed_time(b) for a, b in rev]))
    fpt = synthetic.flops_per_transition(c['O'], c['A'], c['L'], c['U'])
    flops_per_launch = fpt * c['H'] * B
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, 'MEASURED_PEAKS.json')))
    except Exception:
        pass
    peak_tf = peaks.get('bf16_tflops', 1590.0)
    achieved_tf = flops_per_launch / (roll_ms * 1e-3) / 1e12
    ms_plan = ms.mean()
    kernel_name = "rollout_tc_kernel<1,4,pair>" if precision == 'bf16' else "rollout_f32_kernel"
    roofline = {"kernel": kernel_name,
                "bound": "tensor", "achieved": achieved_tf, "peak": peak_tf, "unit": "TFLOP/s",
                # dram__bytes_read.sum + dram__bytes_write.sum of one launch of the CURRENT kernel at this shape,
                # from the committed ncu --set full capture (profiles/kernel_traffic.json, written by
                # tools/ncu_traffic.py); null when no capture of this kernel version is committed
                "frac": achieved_tf / peak_tf, "traffic": committed_traffic(kernel_name + "@c1"),
                "peak_source": "MEASURED_PEAKS.json bf16_tflops (burst)" if peaks else "fallback 1.59 PFLOP/s",
                "flops_per_launch": flops_per_launch, "launch_ms": roll_ms,
                "share_of_plan": c['I'] * roll_ms / ms_plan,
                "note": "C1 is latency-bound: %d row tiles (%s) on 148 SMs, %d dependent GEMM stages per launch"
                        % (c['E'] * ((B // c['E'] + 127) // 128) if precision == 'bf16' else (B + 31) // 32,
                           "a cluster of two CTAs each" if precision == 'bf16' else "one CTA each",
                           c['H'] * (c['L'] + 1))}

    line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W,
            "ms_per_step": float(ms_plan), "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "bf16" if precision == 'bf16' else "f32", "data": "synthetic (random-init ensemble, synthetic states)",
            "config": workload_config(c, "bf16 tcgen05, fp32 accumulate" if precision == 'bf16' else "fp32 SIMT",
                                      {"parallelism": "independent plans per GPU (no collective)" if world > 1 else "1 GPU"}),
            "transitions_per_s": world * K * iters_total * c['H'] * B / t_dev,
            "iterations_run_per_plan": iters_total,
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": c['O'] * 4 + 16,
                    "d2h_bytes_per_step": c['A'] * 4 + 8},
            "gpu_launches": launches, "launches_per_plan": pol.launches_per_plan,
            "clocks": clocks, "roofline": roofline, "wall_s_timed_loop": t_wall}

    # ---- extras -----------------------------------------------------------------------------------
    extras = {}
    if args.extras is None:
        args.extras = 'c3,c4' if world > 1 else 'fp32,c4,c3,c5,train'
    want = [x for x in args.extras.split(',') if x]
    try:
        if 'fp32' in want and precision != 'fp32':
            extras['fp32'] = bench_plain(synthetic, torch, c, 'fp32', states, flush, min(K, 50))
        if 'c4' in want:
            extras['c4'] = bench_batched(synthetic, torch, dist, precision, flush, world, rank)
        if 'c3' in want:
            extras['c3'] = bench_c3(synthetic, torch, dist, lib, _lib, precision, world, rank, flush)
        if 'c5' in want and rank == 0:
            extras['c5'] = bench_wide(synthetic, torch, flush, cpu=not args.no_cpu_baseline and world == 1)
        if 'train' in want and rank == 0:
            extras['train'] = bench_train(torch, cpu=not args.no_cpu_baseline and world == 1)
    except Exception as e:                      # extras never take the headline line down
        extras['error'] = repr(e)
    if extras:
        line['extras'] = extras
    if 'c5' in extras and 'bf16_20state' in extras.get('c5', {}):
        tfw = extras['c5']['bf16_20state']['tflops']
        line['roofline_wide'] = {"kernel": "rollout_tc_wide_kernel", "workload": "configs[4] x 20 states per call",
                                 "bound": "tensor", "achieved": tfw, "peak": peak_tf, "unit": "TFLOP/s",
                                 "frac": tfw / peak_tf, "traffic": committed_traffic("rollout_tc_wide_kernel@c5_20states"),
                                 "note": "plan-level: algorithmic flops of the call / CUDA-event time of the call; "
                                         "470 row tiles = 3.18 waves of 148 SMs (the fourth wave is 18 % full)"}
        if 'bf16_18state' in extras['c5']:
            tf18 = extras['c5']['bf16_18state']['tflops']
            line['roofline_wide']['full_waves'] = {"workload": "configs[4] x 18 states per call (430 row tiles = 2.91 waves)",
                                                   "achieved": tf18, "frac": tf18 / peak_tf}
    if 'c4' in extras and 'tflops_per_gpu' in extras['c4']:
        # the same kernel at a shape that fills the GPU (BASELINE configs[3], 1024 states per call):
        # whole planning calls, so it includes the small CEM kernels (< 1 % of the time there)
        tf = extras['c4']['tflops_per_gpu']
        line['roofline_large'] = {"kernel": "rollout_tc_kernel<2,2>" if precision == 'bf16' else "rollout_f32_kernel",
                                  "traffic_rollout_launch": committed_traffic("rollout_tc_kernel<2,2>@c4_256states"),
                                  "workload": "configs[3]: %d states x C1 per GPU" % extras['c4']['states_per_call_per_gpu'],
                                  "bound": "tensor", "achieved": tf, "peak": peak_tf, "unit": "TFLOP/s",
                                  "frac": tf / peak_tf, "traffic": None,
                                  "note": "plan-level: algorithmic flops of the call / CUDA-event time of the call"}

    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        line['cpu_baseline'] = time_cpu_planner(c)
    if rank == 0:
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def dump_outputs(out_dir, arrays, suffix=''):
    """Each array as <out_dir>/<name><suffix>.npy in float32 (iteration counts are exact in float32)."""
    os.makedirs(out_dir, exist_ok=True)
    for name, x in arrays.items():
        np.save(os.path.join(out_dir, name + suffix + '.npy'), np.asarray(x, dtype=np.float32))


def committed_traffic(key):
    """DRAM bytes per launch of a kernel from the committed ncu capture of the current kernel version."""
    try:
        rec = json.load(open(os.path.join(ROOT, 'profiles', 'kernel_traffic.json')))[key]
        return rec['dram_bytes_per_launch']
    except Exception:
        return None


def bench_plain(synthetic, torch, c, precision, states, flush, K):
    pol = synthetic.build_policy(c, 'penalty', precision=precision, seed=7)
    for k in range(3):
        pol.plan_device(states[k:k + 1])
    torch.cuda.synchronize()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(K)]
    for k in range(K):
        flush.fill_(k & 0xff)
        ev[k][0].record()
        pol.plan_device(states[k % 16:k % 16 + 1])
        ev[k][1].record()
    torch.cuda.synchronize()
    ms = float(np.mean([a.elapsed_time(b) for a, b in ev]))
    return {"plans_per_s": 1e3 / ms, "ms_per_plan": ms, "precision": precision}


def bench_wide(synthetic, torch, flush, cpu=True):
    """BASELINE configs[4]: the wide 10 x (4 x 400) ensemble, horizon 50 — safety-aware (SafeCemMpc,
    penalty) and safety-unaware (CemMpc, reward-only elites) single-state plans on the streaming tcgen05
    kernel (bf16), the fp32 kernel beside it, plus 5, 18 and 20 states per call for the kernel's throughput (one
    128-row tile per SM and wave: 20 states are 470 tiles = 3.18 waves of 148, i.e. a fourth wave that is 18 % full;
    18 states are 430 tiles = 2.91 waves, the same kernel without that tail), and one plan of the CPU restatement on
    the host cores."""
    out = {}
    fpt = None
    for objective, precision, S in (('penalty', 'bf16', 1), ('reward', 'bf16', 1), ('penalty', 'fp32', 1),
                                    ('penalty', 'bf16', 5), ('penalty', 'bf16', 18), ('penalty', 'bf16', 20),
                                    ('reward', 'bf16', 20)):
        c = synthetic.make_workload('c5', S=S, seed=0)
        pol = synthetic.build_policy(c, objective, precision=precision, seed=31)
        st = torch.from_numpy(synthetic.make_state(c['sensors'], seed=500, n_states=S).reshape(S, -1)).cuda()
        pol.plan_device(st)
        torch.cuda.synchronize()
        K = 3
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(K)]
        for k in range(K):
            flush.fill_(k & 0xff)
            ev[k][0].record()
            pol.plan_device(st)
            ev[k][1].record()
        torch.cuda.synchronize()
        ms = float(np.mean([a.elapsed_time(b) for a, b in ev]))
        fpt = synthetic.flops_per_transition(c['O'], c['A'], c['L'], c['U'])
        trans = c['I'] * c['H'] * c['P'] * c['N'] * S
        tag = "%s_%dstate" % (precision, S) if objective == 'penalty' else "%s_%dstate_reward_only" % (precision, S)
        tiles = c['E'] * ((c['P'] * c['N'] * S // c['E'] + 127) // 128)
        out[tag] = {"objective": "SafeCemMpc penalty" if objective == 'penalty' else "CemMpc reward-only",
                    "ms_per_call": ms, "plans_per_s": S * 1e3 / ms, "tflops": trans * fpt / (ms * 1e-3) / 1e12,
                    "row_tiles": tiles, "waves_of_148_sms": round(tiles / 148.0, 2)}
    out["workload"] = "configs[4]: E=10 L=4x400 O=60 A=2 H=50 N=150 P=20 I=5; %d flop per transition" % fpt
    if cpu:
        c = synthetic.make_workload('c5', S=1, seed=0)
        cb = time_cpu_planner(c, budget_s=30.0, max_plans=2, label="configs[4] (C5)")
        out["cpu_baseline"] = cb
    return out


def bench_train(torch, cpu=True, steps=1000, rows=24000):
    """SURVEY.md section 8 f1: MlpEnsemble training steps (E=5 members x batch 64, 62 -> 4x128 ->
    2x60, Adam) through simba_trainer_fit with the data and the batch schedule resident in HBM;
    beside it the numpy training oracle on the host cores."""
    from simba_b200 import _device, _lib
    from simba_b200.models import MlpEnsemble
    import ctypes as C
    E, B, IN, O = 5, 64, 62, 60
    rng = np.random.default_rng(0)
    ens = MlpEnsemble(IN, O, E, batch_size=B, training_steps=5000, mlp_params=dict(n_layers=4, units=128))
    x = rng.uniform(0, 1, (rows, IN)).astype(np.float32)
    y = rng.normal(0, 0.1, (rows, O)).astype(np.float32)
    index, _ = ens.batch_schedule(rows, steps)
    t = ens._ensure_trainer()
    dx, dy = torch.from_numpy(x).cuda(), torch.from_numpy(y).cuda()
    dindex = torch.from_numpy(index).cuda()
    losses = torch.empty(steps, device='cuda')

    def run(n):
        _lib.check(ens._lib.simba_trainer_fit(t, _device.ptr(dx), _device.ptr(dy), rows, _device.ptr(dindex),
                                              C.c_void_p(0), n, _device.ptr(losses), _device.stream_ptr()))
    run(20)
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    run(steps)
    b.record()
    torch.cuda.synchronize()
    ms = a.elapsed_time(b)
    ens._trained_ahead = True
    per_step = int(ens._lib.simba_trainer_launches_per_step(t))
    out = {"workload": "E=%d x batch %d, 62->4x128->2x60, Adam(clipvalue 1, eps 1e-5); %d steps, data in HBM" % (E, B, steps),
           "steps_per_s": steps / (ms * 1e-3), "us_per_step": ms * 1e3 / steps, "launches_per_step": per_step,
           "loss_first": float(losses[0]), "loss_last": float(losses[steps - 1])}
    if cpu:
        from oracle import train_oracle as T           # CPU baseline leg only
        try:
            import threadpoolctl
            threadpoolctl.threadpool_limits(limits=os.cpu_count())
        except Exception:
            pass
        ora = T.EnsembleTrainer([m.get_weights() for m in MlpEnsemble(IN, O, E, mlp_params=dict(n_layers=4, units=128)).ensemble],
                                batch_size=B)
        n, t0 = 0, time.perf_counter()
        while time.perf_counter() - t0 < 5.0:
            idx = index[n % steps]
            ora.training_step(x[idx], y[idx])
            n += 1
        dt = time.perf_counter() - t0
        out["cpu_port_steps_per_s"] = n / dt
        out["cpu_sample"] = "%d numpy fp32 training steps in %.1f s (all host cores available to BLAS)" % (n, dt)
    return out


def bench_batched(synthetic, torch, dist, precision, flush, world, rank, S=1024):
    """BASELINE configs[3]: S independent states per call, sharded over the ranks (no data-path
    collective). Device-timed per rank (max over ranks), and once end to end through
    simba_b200.distributed.plan_states_sharded (host states in, all S actions out on every rank)."""
    from simba_b200 import distributed as sd
    S_local = S // world
    c = synthetic.make_workload('c1', S=S_local, seed=0)
    pol = synthetic.build_policy(c, 'penalty', precision=precision, seed=11)
    states_all = synthetic.make_state(c['sensors'], seed=300, n_states=S)          # same on every rank
    lo, hi = sd.shard_bounds(S, world, rank)
    st = torch.from_numpy(np.ascontiguousarray(states_all[lo:hi])).cuda()
    for _ in range(2):
        pol.plan_device(st)
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    K = 5
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(K)]
    for k in range(K):
        flush.fill_(k & 0xff)
        ev[k][0].record()
        pol.plan_device(st)
        ev[k][1].record()
    torch.cuda.synchronize()
    t = torch.tensor([np.mean([a.elapsed_time(b) for a, b in ev])], dtype=torch.float64, device='cuda')
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t.cpu()[0])
    fpt = synthetic.flops_per_transition(c['O'], c['A'], c['L'], c['U'])
    trans = c['I'] * c['H'] * c['P'] * c['N'] * S_local
    out = {"states_per_call_per_gpu": S_local, "states_per_call_total": S, "ms_per_call": ms,
           "plans_per_s_per_gpu": S_local * 1e3 / ms, "plans_per_s_total": S * 1e3 / ms,
           "transitions_per_s_per_gpu": trans / (ms * 1e-3), "tflops_per_gpu": trans * fpt / (ms * 1e-3) / 1e12,
           "scaling": "strong (1024 states split over the ranks)"}
    if world > 1:
        # the public sharded call: every rank passes all S states, gets all S actions
        dist.barrier()
        t0 = time.perf_counter()
        acts = sd.plan_states_sharded(pol, states_all)
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        out["plan_states_sharded"] = {"ms_per_call_e2e": dt * 1e3, "actions_shape": list(acts.shape),
                                      "all_finite": bool(np.all(np.isfinite(acts)))}
    return out


def bench_c3(synthetic, torch, dist, lib, _lib, precision, world, rank, flush):
    """BASELINE configs[2]: population 65536, 32 particles, horizon 30, sharded over the ranks with one
    NCCL all-gather of (return, cost) per iteration. E=5 does not divide P=32 (the reference's tf.split
    would raise) -> member_map='particle'. Five timed plans, L2 flushed between them; a per-iteration
    breakdown from CUDA events around single launches of each stage; at N > 1 rank 0 also runs the same
    plan unsharded and reports whether the sharded plan reproduces it bit for bit."""
    import ctypes as C
    c = synthetic.make_workload('c3')
    pol, ok = None, 1.0
    try:
        pol = synthetic.build_policy(c, 'penalty', precision=precision, member_map='particle', seed=21,
                                     rank=rank, world_size=world)
        pol.build()
    except Exception:
        ok = 0.0
    if world > 1:
        # every rank must reach the collective NCCL init, or none: agree first
        flag = torch.tensor([ok], device='cuda')
        dist.all_reduce(flag, op=dist.ReduceOp.MIN)
        ok = float(flag.cpu()[0])
    if ok < 1.0:
        return {"skipped": "planner construction failed on at least one rank"}
    if world > 1:
        from simba_b200 import distributed as sd
        sd.init_population_sharding(pol)
    st = torch.from_numpy(synthetic.make_state(c['sensors'], seed=400, n_states=1).reshape(1, -1)).cuda()
    pol.plan_device(st, seed=5)
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    K = 5
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(K)]
    outs = []
    for k in range(K):
        flush.fill_(k & 0xff)
        ev[k][0].record()
        a_k, s_k = pol.plan_device(st, seed=5 + k)[:2]
        ev[k][1].record()
        outs.append(torch.cat([a_k.reshape(-1).clone(), s_k.reshape(-1).clone()]))
    torch.cuda.synchronize()
    t = torch.tensor([np.mean([a.elapsed_time(b) for a, b in ev])], dtype=torch.float64, device='cuda')
    same = torch.ones(1, device='cuda')
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ref = outs[-1].clone()
        dist.broadcast(ref, 0)
        same = (ref == outs[-1]).all().float().reshape(1)
        dist.all_reduce(same, op=dist.ReduceOp.MIN)
    ms = float(t.cpu()[0])
    fpt = synthetic.flops_per_transition(c['O'], c['A'], c['L'], c['U'])
    trans = c['I'] * c['H'] * c['P'] * c['N']
    out = {"ms_per_plan": ms, "plans_per_s": 1e3 / ms, "transitions_per_s": trans / (ms * 1e-3),
           "tflops_total": trans * fpt / (ms * 1e-3) / 1e12, "replicas_bit_identical": bool(same.cpu()[0] > 0),
           "member_map": "particle", "scaling": "strong", "timed_plans": K, "l2": "flushed between timed plans"}

    # ---- per-iteration breakdown: each stage launched alone, CUDA events, this rank's shard --------
    pl = pol._ensure_planner()
    S, N, H, A, P_, O, Kel = 1, c['N'], c['H'], c['A'], c['P'], c['O'], c['K']
    Nl = N // world
    f32 = dict(dtype=torch.float32, device='cuda')
    mu = torch.zeros((S, H, A), **f32); sg = torch.ones((S, H, A), **f32)
    acts = torch.empty((S, N, H, A), **f32)
    ret = torch.empty((S, P_, Nl), **f32); msk = torch.empty((S, P_, Nl), dtype=torch.int64, device='cuda')
    csum = torch.empty((S, P_, Nl), **f32)
    pl_local = torch.empty((S, Nl, 2), **f32); pairs = torch.empty((world, S, Nl, 2), **f32)
    elite = torch.empty((S, Kel), dtype=torch.int32, device='cuda')
    best_a = torch.zeros((S, A), **f32); best_s = torch.full((S,), -np.inf, **f32)
    active = torch.ones((S,), dtype=torch.int32, device='cuda'); iters = torch.zeros((S,), dtype=torch.int32, device='cuda')
    sp = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    p = lambda t_: C.c_void_p(t_.data_ptr())
    stages = [
        ('sample', lambda i: lib.simba_sample_actions(pl, p(mu), p(sg), None, 3, i, None, p(acts), sp)),
        ('rollout', lambda i: lib.simba_rollout_score(pl, p(st), p(acts), None, 3, i, None, p(ret), p(msk), p(csum), sp)),
        ('reduce', lambda i: lib.simba_score_reduce(pl, p(ret), p(msk), p(csum), None, p(pl_local), sp)),
        ('all_gather', lambda i: lib.simba_allgather_scores(pl, p(pl_local), p(pairs), sp)),
        ('select', lambda i: lib.simba_select_elites(pl, p(pairs), p(acts), None, p(elite), None, p(best_a), p(best_s), sp)),
        ('refit', lambda i: lib.simba_refit(pl, p(acts), p(elite), p(mu), p(sg), p(active), p(iters), sp)),
    ]
    breakdown = {}
    for name, fn in stages:
        _lib.check(fn(0))
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        ts = []
        for i in range(3):
            a_, b_ = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a_.record(); _lib.check(fn(i + 1)); b_.record(); torch.cuda.synchronize()
            ts.append(a_.elapsed_time(b_))
        breakdown[name + "_us"] = 1e3 * float(np.mean(ts))
    rest = sum(v for k_, v in breakdown.items() if k_ != 'rollout_us')
    breakdown["not_rollout_share"] = rest / max(1e-9, rest + breakdown['rollout_us'])
    breakdown["note"] = ("single launches incl. ~5-8 us launch latency each; inside the plan's CUDA graph the small "
                         "stages are shorter")
    out["per_iteration_breakdown"] = breakdown

    # ---- sharded == unsharded (rank 0 runs the whole population alone) ----------------------------
    if world > 1:
        eq = torch.ones(1, device='cuda')
        if rank == 0:
            solo = synthetic.build_policy(c, 'penalty', precision=precision, member_map='particle', seed=21)
            a1, s1 = solo.plan_device(st, seed=5 + K - 1)[:2]
            torch.cuda.synchronize()
            single = torch.cat([a1.reshape(-1), s1.reshape(-1)])
            eq = (single == outs[-1]).all().float().reshape(1)
        dist.broadcast(eq, 0)
        out["sharded_equals_single"] = bool(eq.cpu()[0] > 0)
    return out


if __name__ == '__main__':
    main()
