"""MppiMpc / SafeMppiMpc — the CEM planners' sampling, rollout and objectives with the MPPI update of Williams et al.,
"Information theoretic MPC for model-based reinforcement learning" (ICRA 2017), as PDDM (Nagabandi et al., 2019)
plans with.

Each iteration weights ALL N candidates by w_i = exp((S_i - max S) / temperature) (0 for a NaN score) and moves the
mean to the weighted mean of their action sequences, with CemMpc's smoothing; sigma stays at its initial value and
there is no early exit. The action is mu[0] + noise_stddev * z, the score the best candidate's score over all
iterations. Low temperatures approach the best candidate, high ones the plain mean. With SafeMppiMpc's penalty
objective an unsafe candidate scores 100 lower and so weighs exp(-100 / temperature) as much.

Every keyword-only option of CemMpc applies (precision, seed, n_states, member_map); the population is not sharded
(world_size 1), so multi-GPU use shards states (simba_b200.distributed.plan_states_sharded).
"""
from .. import _lib
from .cem_mpc import CemMpc


class MppiMpc(CemMpc):
    _objective = _lib.OBJ_REWARD

    def __init__(self, model, environment, horizon, iterations, smoothing, n_samples, particles, noise_stddev,
                 temperature, **kwargs):
        # n_elite and stddev_threshold are CEM's: the planner config needs valid values, the MPPI update reads neither
        super().__init__(model, environment, horizon, iterations, smoothing, n_samples, 1, particles, 0.0,
                         noise_stddev, **kwargs)
        self.temperature = float(temperature)

    def _configure_planner(self, handle):
        _lib.check(self._lib.simba_planner_set_update_rule(handle, _lib.UPDATE_MPPI, self.temperature))


class SafeMppiMpc(MppiMpc):
    """SafeCemMpc's objectives under the MPPI update: selection='penalty' (safe_cem_mpc.py:96, the default) or
    'least_cost' (optimize_for_safety's score). 'feasible_first' is an order with no scalar score and is rejected."""
    _objective = _lib.OBJ_SAFE_PENALTY

    def __init__(self, model, environment, horizon, iterations, smoothing, n_samples, particles, noise_stddev,
                 temperature, posterior_mean_threashold, *, selection='penalty', **kwargs):
        objectives = {'penalty': _lib.OBJ_SAFE_PENALTY, 'least_cost': _lib.OBJ_LEAST_COST}
        if selection not in objectives:
            raise ValueError("selection must be 'penalty' or 'least_cost' under MPPI, got %r" % (selection,))
        super().__init__(model, environment, horizon, iterations, smoothing, n_samples, particles, noise_stddev,
                         temperature, objective=objectives[selection],
                         posterior_mean_threashold=posterior_mean_threashold, **kwargs)
        self.cost = environment.get_cost
        self.posterior_mean_threashold = posterior_mean_threashold
