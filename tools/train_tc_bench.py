"""Ensemble training throughput and accuracy, fp32 SIMT trainer against the bf16 tcgen05 trainer.

For C1 (E=5, 62 -> 4x128 -> 2x60) and C5 (E=10, 62 -> 4x400 -> 2x60), batch 64: steps/s of
simba_trainer_fit timed with CUDA events, the two precisions alternating in one process; the loss curve
of each precision on the same data and batch schedule; and the one-step errors of the bf16 path against
oracle/train_oracle.py over the shapes of tests/test_gpu_train_tc.py. The card name and power limit are
read in the same run.

  python tools/train_tc_bench.py --out profiles/r05_train_tc_bench.json
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, 'ethz-safe-learning_b200')):
    if p not in sys.path:
        sys.path.insert(0, p)

import torch  # noqa: E402

from oracle import train_oracle as T  # noqa: E402
from simba_b200 import _device, _lib  # noqa: E402
from simba_b200.models import MlpEnsemble  # noqa: E402

CONFIGS = {'C1': dict(E=5, O=60, A=2, L=4, U=128), 'C5': dict(E=10, O=60, A=2, L=4, U=400)}
ONE_STEP_SHAPES = [(62, 60, 5, 64, 4, 128), (12, 10, 3, 16, 2, 40), (7, 5, 2, 9, 1, 33),
                   (62, 60, 2, 32, 2, 400), (20, 18, 2, 24, 3, 200), (9, 7, 1, 5, 2, 130)]


def card():
    out = subprocess.check_output(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm',
                                   '--format=csv,noheader', '-i', '0'], text=True).strip()
    name, power, clock = [s.strip() for s in out.split(',')]
    return dict(name=name, power_limit=power, max_sm_clock=clock)


def dynamics(rng, n, O, A):
    obs = rng.uniform(-1, 1, (n, O)).astype(np.float32)
    act = rng.uniform(-1, 1, (n, A)).astype(np.float32)
    delta = 0.1 * np.tanh(obs) + 0.05 * np.pad(act, ((0, 0), (0, O - A))) + \
        0.02 * np.roll(obs, 1, axis=1) * act[:, :1]
    return np.concatenate([obs, act], axis=1), delta.astype(np.float32)


def flops_per_step(E, B, IN, O, L, U):
    """forward + weight gradients + activation back-propagation without layer 0, 2 flop per MAC"""
    fwd = 2 * ((IN + 1) * U + (L - 1) * (U + 1) * U + (U + 1) * 2 * O)
    bwd = 2 * ((L - 1) * U * U + U * 2 * O)
    return (2 * fwd + bwd) * B * E


class Fitter:
    def __init__(self, cfg, precision, x, y, steps, seed=5):
        E, O, A, L, U = cfg['E'], cfg['O'], cfg['A'], cfg['L'], cfg['U']
        self.ens = MlpEnsemble(O + A, O, E, batch_size=64, learning_rate=1e-3, learning_rate_schedule=False,
                               training_steps=steps, mlp_params=dict(n_layers=L, units=U), seed=seed,
                               train_precision=precision)
        self.t = self.ens._ensure_trainer()
        self.lib = _lib.load()
        rs = np.random.RandomState(seed)
        index = np.stack([np.stack([rs.randint(0, x.shape[0], 64) for _ in range(E)]) for _ in range(steps)])
        self.x, _ = _device.to_device(x)
        self.y, _ = _device.to_device(y)
        self.index, _ = _device.to_device(index.astype(np.int32), dtype=torch.int32)
        self.losses = torch.empty((steps,), dtype=torch.float32, device=self.x.device)
        self.n = x.shape[0]

    def fit(self, steps):
        _lib.check(self.lib.simba_trainer_fit(self.t, _device.ptr(self.x), _device.ptr(self.y), self.n,
                                              _device.ptr(self.index), None, steps, _device.ptr(self.losses),
                                              _device.stream_ptr()))


def one_step_errors():
    rows = []
    for shape in ONE_STEP_SHAPES:
        for rate in (0.0, 0.1, 0.5):
            n_in, n_out, E, B, L, U = shape
            ens = MlpEnsemble(n_in, n_out, E, batch_size=B, learning_rate=0.00025, learning_rate_schedule=False,
                              mlp_params=dict(n_layers=L, units=U, dropout_rate=rate), seed=7,
                              train_precision='bf16')
            ora = T.EnsembleTrainer([m.get_weights() for m in ens.ensemble], batch_size=B,
                                    learning_rate=0.00025, learning_rate_schedule=False, dropout_rate=rate,
                                    dropout_seed=7)
            rng = np.random.default_rng(1)
            x = rng.uniform(0, 1, (E, B, n_in)).astype(np.float32)
            y = rng.normal(0, 0.1, (E, B, n_out)).astype(np.float32)
            got, want = float(ens.training_step(x, y)), float(ora.training_step(x, y))
            n_var = 2 * L + 4
            g_err = 0.0
            for e in range(E):
                for g, r in zip(ens.trainer_arrays('grads', e), ora.last_grads[e * n_var:(e + 1) * n_var]):
                    r = np.asarray(r, np.float64)
                    g_err = max(g_err, float(np.linalg.norm(g - r) / max(np.linalg.norm(r), 1e-30)))
            w_err = max(float(np.abs(a - b).max()) for e in range(E)
                        for a, b in zip(ens.trainer_arrays('weights', e), ora.nets[e].arrays))
            rows.append(dict(shape=list(shape), dropout_rate=rate, loss_rel=abs(got - want) / abs(want),
                             grad_rel_max=g_err, weight_abs_max_over_lr=w_err / 0.00025))
    return rows


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--steps', type=int, default=800, help='steps per timed fit call')
    ap.add_argument('--repeats', type=int, default=5)
    ap.add_argument('--curve-steps', type=int, default=2000)
    ap.add_argument('--out', default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("train_tc_bench needs a GPU")
    result = dict(card=card(), batch=64, timed_steps_per_call=args.steps, repeats=args.repeats, configs={})
    rng = np.random.default_rng(10)
    for name, cfg in CONFIGS.items():
        x, y = dynamics(rng, 20000, cfg['O'], cfg['A'])
        fl = flops_per_step(cfg['E'], 64, cfg['O'] + cfg['A'], cfg['O'], cfg['L'], cfg['U'])
        fitters = {p: Fitter(cfg, p, x, y, max(args.steps, args.curve_steps)) for p in ('fp32', 'bf16')}
        for f in fitters.values():                                  # warm-up: graph capture, module load
            f.fit(32)
        torch.cuda.synchronize()
        times = {p: [] for p in fitters}
        for _ in range(args.repeats):
            for p, f in fitters.items():                            # alternate the precisions
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record()
                f.fit(args.steps)
                b.record()
                b.synchronize()
                times[p].append(a.elapsed_time(b) / args.steps * 1e3)   # us per step
        entry = dict(cfg, flop_per_step=fl)
        for p, ts in times.items():
            med = float(np.median(ts))
            entry[p] = dict(us_per_step=sorted(ts), median_us_per_step=med, steps_per_s=1e6 / med,
                            tflops=fl / med / 1e6)
        entry['bf16_speedup'] = entry['fp32']['median_us_per_step'] / entry['bf16']['median_us_per_step']
        # loss curves: fresh trainers, the same data and batch schedule
        curves = {}
        for p in ('fp32', 'bf16'):
            f = Fitter(cfg, p, x, y, args.curve_steps, seed=6)
            f.fit(args.curve_steps)
            losses = f.losses.cpu().numpy()
            curves[p] = dict(every_50=[float(v) for v in losses[::50]],
                             last_10pct_mean=float(losses[-args.curve_steps // 10:].mean()),
                             first_10pct_mean=float(losses[:args.curve_steps // 10].mean()))
        entry['loss_curves'] = curves
        result['configs'][name] = entry
        print(name, json.dumps({p: entry[p]['steps_per_s'] for p in ('fp32', 'bf16')}), flush=True)
    result['one_step_errors'] = one_step_errors()
    worst = {k: max(r[k] for r in result['one_step_errors'])
             for k in ('loss_rel', 'grad_rel_max', 'weight_abs_max_over_lr')}
    result['one_step_worst'] = worst
    print(json.dumps(dict(card=result['card'], worst=worst,
                          speedup={n: result['configs'][n]['bf16_speedup'] for n in CONFIGS})))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, 'w') as fh:
            json.dump(result, fh, indent=1)


if __name__ == '__main__':
    main()
