"""Synthetic workloads of the BASELINE.json shapes (SURVEY.md section 8 d). Pure numpy: the same
arrays feed the CUDA planner, the CPU oracle (tests, bench cpu_baseline) and the golden fixtures.

There are no trained checkpoints or datasets offline, so weights are Keras-default random inits
(glorot-uniform kernels, zero biases — mlp_ensemble.py:13,28-30) with two documented adjustments
that keep rollouts in the regime a trained model produces (small state deltas, small predictive
variance) instead of a random walk that saturates every threshold:
  * mu-head kernel scaled by `mu_scale`;
  * var-head bias = `var_bias` (softplus(-9) + 1e-4 ~= 2.2e-4, sigma ~= 0.015 per step);
  * first-layer rows of the action inputs scaled by `action_gain`, so that the candidate action
    sequences actually steer the rollout (otherwise 2 of 62 random inputs barely matter and every
    candidate scores alike). With the defaults a C1 plan sees a mix of safe and unsafe candidates.
"""
import numpy as np

CONFIGS = {
    # name: E, L, U, O, A, H, N, P, I, K, S
    'c1': dict(E=5, L=4, U=128, H=15, N=150, P=20, I=5, K=15, S=1),          # BASELINE configs[0]/[1]
    'c3': dict(E=5, L=4, U=128, H=30, N=65536, P=32, I=5, K=6554, S=1),      # configs[2] (member_map particle)
    'c4': dict(E=5, L=4, U=128, H=15, N=150, P=20, I=5, K=15, S=1024),       # configs[3]
    'c5': dict(E=10, L=4, U=400, H=50, N=150, P=20, I=5, K=15, S=1),         # configs[4]
    'shipped': dict(E=15, L=4, U=128, H=8, N=500, P=45, I=9, K=20, S=1),     # config/policies.yaml:11-20
    'tiny': dict(E=2, L=2, U=128, H=6, N=24, P=8, I=3, K=5, S=1),
}

POINTGOAL1_SENSORS = dict(accelerometer=3, goal_lidar=16, gyro=3, hazards_lidar=16, magnetometer=3,
                          vases_lidar=16, velocimeter=3)
POINTSIMPLEGOAL1_SENSORS = dict(accelerometer=3, goal_lidar=5, gyro=3, hazards_lidar=5,
                                magnetometer=3, velocimeter=3)


def offsets(sensors):
    table, off = {}, 0
    for k in sorted(sensors):
        table[k] = slice(off, off + sensors[k])
        off += sensors[k]
    return table, off


def make_weights(E, L, U, O, A, seed=0, mu_scale=0.05, var_bias=-9.0, action_gain=8.0):
    """members[e] = [W_1, b_1, ..., W_L, b_L, W_mu, b_mu, W_var, b_var] (Keras order, kernels [in, out])."""
    rng = np.random.default_rng(seed)
    members = []
    for _ in range(E):
        arrs, fan_in = [], O + A
        for _ in range(L):
            lim = np.sqrt(6.0 / (fan_in + U))
            w = rng.uniform(-lim, lim, (fan_in, U))
            if fan_in == O + A:
                w[O:, :] *= action_gain
            arrs += [w.astype(np.float32), np.zeros(U, np.float32)]
            fan_in = U
        lim = np.sqrt(6.0 / (U + O))
        arrs += [(rng.uniform(-lim, lim, (U, O)) * mu_scale).astype(np.float32), np.zeros(O, np.float32)]
        arrs += [rng.uniform(-lim, lim, (U, O)).astype(np.float32), np.full(O, var_bias, np.float32)]
        members.append(arrs)
    return members


def make_scaler(O, A):
    """Finite bounds (avoids the +-inf NaN of transition_model.py:85-87): obs in [-1, 2], act in [-1, 1]."""
    mn = np.concatenate([np.full(O, -1.0), np.full(A, -1.0)]).astype(np.float32)
    mx = np.concatenate([np.full(O, 2.0), np.full(A, 1.0)]).astype(np.float32)
    return mn, mx


def make_state(sensors=None, seed=1, n_states=1):
    """Sensor dims U(-1, 1); goal_lidar U(0.3, 1.0) (goal not met at t = 0); hazards_lidar
    U(0.2, 1.0) (the 0.2 / 4 = 0.05 cost threshold is reachable within a horizon, not at t = 0)."""
    sensors = sensors or POINTGOAL1_SENSORS
    table, O = offsets(sensors)
    rng = np.random.default_rng(seed)
    st = rng.uniform(-1.0, 1.0, (n_states, O)).astype(np.float32)
    for k, sl in table.items():
        n = sl.stop - sl.start
        if k == 'goal_lidar':
            st[:, sl] = rng.uniform(0.3, 1.0, (n_states, n))
        elif k == 'hazards_lidar':
            st[:, sl] = rng.uniform(0.2, 1.0, (n_states, n))
        elif k.endswith('_lidar'):
            st[:, sl] = rng.uniform(0.08, 1.0, (n_states, n))
    return st if n_states > 1 else st[0]


def make_draws(I, S, N, H, A, P, O, seed=2):
    """External N(0,1) draws for parity mode: z_actions [I,S,N,H,A], eps [I,S,H,P*N,O], z_final [S,A]."""
    rng = np.random.default_rng(seed)
    z = rng.standard_normal((I, S, N, H, A), dtype=np.float32)
    eps = rng.standard_normal((I, S, H, P * N, O), dtype=np.float32)
    zf = rng.standard_normal((S, A), dtype=np.float32)
    return z, eps, zf


def make_workload(cfg_name='c1', sensors=None, seed=0, mu_scale=0.05, var_bias=-9.0, action_gain=8.0,
                  **over):
    """Everything a planner needs for one named config: dims, weights, scaler, state(s)."""
    c = dict(CONFIGS[cfg_name])
    c.update(over)
    sensors = sensors or POINTGOAL1_SENSORS
    table, O = offsets(sensors)
    A = int(c.get('A', 2))                        # action dims (the reference's point robot has 2)
    c.update(O=O, A=A, sensors=sensors, table=table)
    c['weights'] = make_weights(c['E'], c['L'], c['U'], O, A, seed=seed, mu_scale=mu_scale,
                                var_bias=var_bias, action_gain=action_gain)
    c['smin'], c['smax'] = make_scaler(O, A)
    c['state'] = make_state(sensors, seed=seed + 1, n_states=c['S'])
    return c


def build_policy(c, objective='penalty', precision='bf16', member_map='split', threshold=0.15,
                 smoothing=0.0, stddev_threshold=0.0, noise_stddev=0.01, sampling_propagation=True,
                 scorer_config=None, seed=0, n_states=None, rank=0, world_size=1, activation='tf.nn.relu',
                 temperature=None):
    """The reference's construction sequence (mbrl_agent.py:103-118) on the B200 classes:
    environment -> TransitionModel(MlpEnsemble) -> CemMpc / SafeCemMpc, with the workload's
    weights and scaler statistics loaded. `activation`: mlp_params['activation'] of the ensemble.
    With a `temperature`, MppiMpc / SafeMppiMpc instead (no n_elite, no stddev_threshold)."""
    from .environment_utils import ScorerEnvironment
    from .models import TransitionModel
    from .policies import CemMpc, MppiMpc, SafeCemMpc, SafeMppiMpc
    env = ScorerEnvironment(c['sensors'], scorer_config, action_low=[-1.0] * c['A'], action_high=[1.0] * c['A'])
    tm = TransitionModel('mlp_ensemble', env.observation_space, env.action_space, True,
                         sampling_propagation, ensemble_size=c['E'],
                         mlp_params=dict(n_layers=c['L'], units=c['U'], activation=activation,
                                         dropout_rate=0.0))
    for e in range(c['E']):
        tm.model.ensemble[e].set_weights(c['weights'][e])
    tm.set_statistics(c['smin'], c['smax'])
    if temperature is not None:
        common = dict(horizon=c['H'], iterations=c['I'], smoothing=smoothing, n_samples=c['N'], particles=c['P'],
                      noise_stddev=noise_stddev, temperature=temperature, precision=precision,
                      member_map=member_map, seed=seed, n_states=c['S'] if n_states is None else n_states,
                      rank=rank, world_size=world_size)
        if objective == 'reward':
            return MppiMpc(tm, env, **common)
        return SafeMppiMpc(tm, env, posterior_mean_threashold=threshold, selection=objective, **common)
    common = dict(horizon=c['H'], iterations=c['I'], smoothing=smoothing, n_samples=c['N'],
                  n_elite=c['K'], particles=c['P'], stddev_threshold=stddev_threshold,
                  noise_stddev=noise_stddev, precision=precision, member_map=member_map, seed=seed,
                  n_states=c['S'] if n_states is None else n_states, rank=rank, world_size=world_size)
    if objective == 'reward':
        return CemMpc(tm, env, **common)
    return SafeCemMpc(tm, env, posterior_mean_threashold=threshold, selection=objective, **common)


def flops_per_transition(O, A, L, U):
    """Algorithmic (unpadded) flops of one ensemble transition: 2*((O+A)*U + (L-1)*U^2 + U*2*O)
    (SURVEY.md section 8 d); bias / activation / RNG / scoring excluded."""
    return 2 * ((O + A) * U + (L - 1) * U * U + U * 2 * O)
