#!/usr/bin/env python
"""Phase timeline of the tcgen05 rollout kernel (needs the -DSIMBA_TC_TIMELINE build:
SIMBA_B200_LIB=.../libsimba_b200_tl.so python tools/tc_timeline.py [c1|c4|c5]; c5 = wide kernel)."""
import ctypes as C
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, 'ethz-safe-learning_b200')]
import numpy as np  # noqa: E402
import torch  # noqa: E402
from simba_b200 import _lib, synthetic  # noqa: E402

wl = sys.argv[1] if len(sys.argv) > 1 else 'c1'
over = dict(S=64) if wl == 'c4' else {}
c = synthetic.make_workload({'c4': 'c4', 'c5': 'c5'}.get(wl, 'c1'), **over)
pol = synthetic.build_policy(c, 'penalty', precision='bf16', seed=1)
lib = _lib.load()
pl = pol._ensure_planner()
S, N, H, A, P_, O = c['S'], c['N'], c['H'], c['A'], c['P'], c['O']
st = torch.from_numpy(np.ascontiguousarray(synthetic.make_state(c['sensors'], 5, S)).reshape(S, O)).cuda()
acts = torch.empty((S, N, H, A), device='cuda').uniform_(-1, 1)
ret = torch.empty((S, P_, N), device='cuda'); msk = torch.empty((S, P_, N), dtype=torch.int64, device='cuda')
csum = torch.empty((S, P_, N), device='cuda')
# the timeline build stamps into prm.timeline, handed in through the env hook of the debug build
tl = torch.zeros((4, 64, 64), dtype=torch.int64, device='cuda')
os.environ['SIMBA_TC_TIMELINE_PTR'] = str(tl.data_ptr())
p = lambda t: C.c_void_p(t.data_ptr())
for it in range(3):
    _lib.check(lib.simba_rollout_score(pl, p(st), p(acts), None, 3, it, None, p(ret), p(msk), p(csum), None))
torch.cuda.synchronize()
t = tl.cpu().numpy()
L = c['L']
if wl == 'c5':                     # rollout_tc_wide.cu keeps the round-1 event layout
    for who, name in ((0, 'epilogue warp 0'), (1, 'last warp of tile')):
        print("==", name)
        for step in range(2, min(H - 1, 8)):
            ev = t[who, step]
            base = ev[0]
            line = ["step %2d" % step]
            for l in range(L):
                line.append("L%d wait->%5d epi->%5d publish->%5d |" % (l, ev[1 + 4 * l] - base, ev[2 + 4 * l] - base, ev[3 + 4 * l] - base))
            line.append("head wait->%5d pass->%5d publish->%5d score->%5d  total %5d" % (
                ev[40] - base, ev[41] - base, ev[42] - base, ev[43] - base, t[who, step + 1][0] - base))
            print(' '.join(line))
    sys.exit(0)
# rollout_tc.cu: epilogue warps stamp 0 (step start), per hidden layer l: 1+4l accumulator ready, 2+4l drained,
# 3+4l A slice published (+ deferred scoring at l = 0), 4+4l noise block done; 40 head accumulator ready,
# 41 head pass done, 42 published. The issuer warp of tile 0 (who = 2) stamps 2*layer (A ready seen) and 2*layer+1 (layer committed).
for who, name in ((0, 'epilogue warp 0 of tile 0'), (1, 'last epilogue warp of tile 0')):
    print("==", name, "(cycles since the step's start)")
    for step in range(2, min(H - 1, 8)):
        ev = t[who, step]
        base = ev[0]
        line = ["step %2d" % step]
        for l in range(L):
            line.append("L%d acc->%5d drained->%5d published->%5d noise->%5d |" % (
                l, ev[1 + 4 * l] - base, ev[2 + 4 * l] - base, ev[3 + 4 * l] - base, ev[4 + 4 * l] - base))
        line.append("head acc->%5d pass->%5d published->%5d  total %5d" % (
            ev[40] - base, ev[41] - base, ev[42] - base, t[who, step + 1][0] - base))
        print(' '.join(line))
print("== noise block detail, epilogue warp 0 (last block of the step): philox rounds / box-muller cycles")
for step in range(2, min(H - 1, 8)):
    ev = t[0, step]
    print("step %2d philox %5d  box-muller %5d" % (step, ev[51] - ev[50], ev[52] - ev[51]))
k = t[3, 0]
print("== launch anatomy, thread 0 of CTA 0 (cycles since kernel entry): setup done %d, PDL wait passed %d, first A published %d, "
      "all items done %d, exit %d" % tuple(int(k[i] - k[0]) for i in range(1, 6)))
if wl == 'c4':
    print("== issuer warp of tile 0 (cycles since epilogue warp 0's step start; layer: A-ready seen -> committed)")
    for step in range(2, min(H - 1, 8)):
        base = t[0, step][0]
        ev = t[2, step]
        print("step %2d " % step + ' | '.join("L%d %5d -> %5d" % (l, ev[2 * l] - base, ev[2 * l + 1] - base) for l in range(L + 1)))
    sys.exit(0)
# one-tile kernels: every layer is two 64-column halves. Epilogue warp 0 above drains the low half, the last warp the
# high half. The issuer stamps 2l (A low half seen), 2l+1 (K[0,64) of both halves issued; layer 0: both halves
# committed), 20+2l (A high half seen) and 21+2l (commits 0 and 1 issued) for hidden and head layers l >= 1.
print("== issuer warp (cycles since epilogue warp 0's step start; layer: A low seen -> K[0,64) issued, "
      "A high seen -> both halves committed)")
for step in range(2, min(H - 1, 8)):
    base = t[0, step][0]
    ev = t[2, step]
    parts = ["L0 %5d -> %5d" % (ev[0] - base, ev[1] - base)]
    parts += ["L%d %5d -> %5d, %5d -> %5d" % (l, ev[2 * l] - base, ev[2 * l + 1] - base, ev[20 + 2 * l] - base,
                                              ev[21 + 2 * l] - base) for l in range(1, L + 1)]
    print("step %2d " % step + ' | '.join(parts))
print("== per hidden layer: high half ready - low half ready / low half published - high half ready (cycles; the "
      "low half drains while the high half's last MMAs run)")
for step in range(2, min(H - 1, 8)):
    lo, hi = t[0, step], t[1, step]
    print("step %2d " % step + ' '.join("L%d %5d / %5d" % (l, hi[1 + 4 * l] - lo[1 + 4 * l], lo[3 + 4 * l] - hi[1 + 4 * l])
                                        for l in range(L)))
