"""bench.py --dump-outputs holds what the LAST timed step returned: the plan is recomputed here from
the same policy seed, call index and state, which also shows that --steps set the number of timed
steps (one step more or fewer changes the seed and the state of the last one)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

# bench.py: policy seed 0x5EED on rank 0, a pool of 16 states (seed 100), call k of the policy uses
# seed + k; W warm-up then K timed device plans, then W warm-up then K timed end-to-end plans.
SEED, POOL, W, K = 0x5EED, 16, 3, 5


def test_dump_outputs_hold_the_last_timed_step(tmp_path):
    out_dir = tmp_path / 'dump'
    cmd = [sys.executable, os.path.join(ROOT, 'bench.py'), '--steps', str(K), '--warmup', str(W),
           '--extras', 'none', '--no-cpu-baseline', '--dump-outputs', str(out_dir)]
    out = subprocess.run(cmd, cwd=str(tmp_path), capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-3000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert line['steps'] == K and line['warmup'] == W
    got = {n[:-len('.npy')]: np.load(out_dir / n) for n in os.listdir(out_dir)}
    assert sorted(got) == ['e2e_action', 'plan_action', 'plan_iterations', 'plan_score']
    assert all(a.dtype == np.float32 for a in got.values())

    from simba_b200 import synthetic
    c = synthetic.make_workload('c1')
    pol = synthetic.build_policy(c, 'penalty', precision='bf16', seed=SEED)
    states_np = synthetic.make_state(c['sensors'], seed=100, n_states=POOL)
    states = torch.from_numpy(states_np).cuda()

    def plan(k, call):
        a, s, i = pol.plan_device(states[k % POOL:k % POOL + 1], seed=SEED + call)
        return {'plan_action': a.cpu().numpy(), 'plan_score': s.cpu().numpy(),
                'plan_iterations': i.cpu().numpy().astype(np.float32)}

    last, first = plan(K - 1, W + K - 1), plan(0, W)
    assert not np.array_equal(last['plan_action'], first['plan_action'])   # the test can tell them apart
    for name, want in last.items():
        assert np.array_equal(got[name], want), name
    e2e, _ = pol.do_generate_action(states_np[(K - 1) % POOL], seed=SEED + 2 * W + 2 * K - 1)
    assert np.array_equal(got['e2e_action'], e2e)
