"""TEST INFRASTRUCTURE ONLY — CPU restatement of the MPPI planning call (simba_planner_set_update_rule with
SIMBA_UPDATE_MPPI, simba_b200.policies.MppiMpc / SafeMppiMpc).

MPPI is Williams et al., "Information theoretic MPC for model-based reinforcement learning" (ICRA 2017), the update
PDDM (Nagabandi et al., 2019) plans with. Everything but the update is the CEM planner of oracle/simba_oracle.py,
reused here: the sampling clip(mu + sigma z, lb, ub), the unfold, the objectives, and the final noise. Per iteration:
  m = max_i S_i over non-NaN scores;  w_i = exp((S_i - m) / temperature), 0 for a NaN score;
  mu <- smoothing mu + (1 - smoothing) sum_i w_i a_i / sum_i w_i   (unchanged when every score is NaN);
sigma fixed; no early exit; best_score = the largest score seen (strict '>'); action = mu[0] + noise_stddev z_final.
Random draws are inputs, as in simba_oracle. The product never imports this file.
"""
import numpy as np

from . import simba_oracle as so


def mppi_mean(scores, acts, temperature, dtype=np.float32):
    """Weighted mean sum_i w_i a_i / sum_i w_i of acts [N, H, A] for scores [N]; None when every score is NaN."""
    dt = np.dtype(dtype)
    scores = np.asarray(scores, dtype=dt)
    valid = ~np.isnan(scores)
    if not valid.any():
        return None
    m = np.max(scores[valid])
    with np.errstate(invalid='ignore'):
        w = np.where(valid, np.exp((scores - m) / dt.type(temperature)), dt.type(0.0)).astype(dt)
    num = np.sum(w[:, None, None] * np.asarray(acts, dtype=dt), axis=0, dtype=dt)
    return (num / np.sum(w, dtype=dt)).astype(dt)


def mppi_update(mu, scores, acts, temperature, smoothing, dtype=np.float32):
    """One MPPI mean update with the CEM refit's smoothing (cem_mpc.py:64)."""
    dt = np.dtype(dtype)
    mu = np.asarray(mu, dtype=dt)
    mean = mppi_mean(scores, acts, temperature, dt)
    if mean is None:
        return mu.copy()
    return dt.type(smoothing) * mu + (dt.type(1.0) - dt.type(smoothing)) * mean


def best_candidate(scores):
    """First index of the largest non-NaN score, or None."""
    valid = ~np.isnan(scores)
    if not valid.any():
        return None
    return int(np.flatnonzero(valid)[np.argmax(scores[valid])])


class MppiPlanner(so.CemPlanner):
    def __init__(self, model, environment, horizon, iterations, smoothing, n_samples, particles, noise_stddev,
                 temperature, posterior_mean_threashold=None, objective=so.OBJ_REWARD, member_map='split',
                 dtype=np.float32):
        if objective == so.OBJ_FEASIBLE_FIRST:
            raise ValueError("FEASIBLE_FIRST is an order with no scalar score: MPPI cannot weight it")
        super().__init__(model, environment, horizon, iterations, smoothing, n_samples, 1, particles, 0.0,
                         noise_stddev, posterior_mean_threashold=posterior_mean_threashold, objective=objective,
                         member_map=member_map, dtype=dtype)
        self.temperature = temperature

    def do_generate_action(self, state, z_actions, eps, z_final, trace=None):
        """z_actions [I, N, H, A], eps [I, H, P*N, O], z_final [A] -> (action, best_score, iterations_run)."""
        dt = self.dt
        lb, ub, mu, sigma = so.sampling_params(self.action_space)
        a_dim = self.action_space.shape[0]
        lb = np.broadcast_to(np.asarray(lb, dtype=dt), (a_dim,))
        ub = np.broadcast_to(np.asarray(ub, dtype=dt), (a_dim,))
        mu = np.broadcast_to(np.asarray(mu, dtype=dt), (self.horizon, a_dim)).copy()
        sigma = np.broadcast_to(np.asarray(sigma, dtype=dt), (self.horizon, a_dim)).copy()
        best = np.zeros((a_dim,), dtype=dt)
        best_score = dt.type(-np.inf)
        state = np.asarray(state, dtype=dt)
        member_of_row = self.member_of_row()
        for it in range(self.iterations):
            acts = np.minimum(np.maximum(z_actions[it].astype(dt) * sigma + mu, lb), ub)
            acts_b = np.tile(acts, (self.particles, 1, 1))
            s0 = np.broadcast_to(state, (acts_b.shape[0], state.shape[0]))
            traj = self.model.unfold_sequences(s0, acts_b, eps[it], member_of_row)
            scores, ret, cost = self.compute_scores(traj, acts_b)
            top = best_candidate(scores)
            if top is not None and scores[top] > best_score:
                best = acts[top, 0].copy()
                best_score = scores[top]
            mu = mppi_update(mu, scores, acts, self.temperature, self.smoothing, dt)
            if trace is not None:
                trace.append(dict(actions=acts, ret=ret, cost=cost, scores=scores, mu=mu.copy(), best=best.copy(),
                                  best_score=best_score))
        action = mu[0] + np.asarray(z_final, dtype=dt) * dt.type(self.noise_stddev)
        return action, best_score, self.iterations
