"""Swish (tf.nn.swish, z * sigmoid(z)) forms of the CPU oracles, for the swish tests and tools/swish_bench.py.

The oracles in oracle/ restate the reference's ReLU model; these subclasses change only the hidden activation and,
for training, its derivative: swish(z) = z * (1 / (1 + exp(-z))) in the array's dtype, in the order the fp32 kernels
use, and swish'(z) = sigmoid(z) * (1 + z * (1 - sigmoid(z))). Everything else (heads, NLL, Adam, scoring, CEM) is the
oracles' own code.
"""
import numpy as np
import torch.nn.functional as F

from oracle import simba_oracle as so
from oracle import torch_ref as tr
from oracle import train_oracle as T


def sigmoid(z):
    one = z.dtype.type(1.0)
    with np.errstate(over='ignore'):                  # exp(-z) = inf for very negative z: sigmoid 0
        return one / (one + np.exp(-z))


def swish(z):
    return z * sigmoid(z)


def swish_grad(z):
    s = sigmoid(z)
    one = z.dtype.type(1.0)
    return s * (one + z * (one - s))


class MlpEnsemble(so.MlpEnsemble):
    """simba_oracle.MlpEnsemble with swish hidden layers."""

    def mlp(self, e, x):
        w = self.members[e]
        for l in range((len(w) - 4) // 2):
            x = swish(x @ w[2 * l] + w[2 * l + 1])
        mu = x @ w[-4] + w[-3]
        var = so.tf_softplus(x @ w[-2] + w[-1]) + self.dt.type(1e-4)
        return mu, var


class GaussianMlp(tr.GaussianMlp):
    """torch_ref.GaussianMlp with swish hidden layers."""

    def __call__(self, x):
        for w, b in self.hidden:
            x = F.silu(F.linear(x, w, b))
        return F.linear(x, *self.mu), tr.tf_softplus(F.linear(x, *self.var)) + 1e-4


class TorchEnsemble(tr.Ensemble):
    def __init__(self, members):
        self.members = [GaussianMlp(m) for m in members]


class MemberNet(T.MemberNet):
    """train_oracle.MemberNet with swish hidden layers: the backward pass multiplies by swish'(z) (and the dropout
    multiplier) where ReLU uses h > 0."""

    def forward(self, x, keep=None):
        L = self.n_layers
        hs, zs = [np.asarray(x, dtype=self.dtype)], []
        for l in range(L):
            z = hs[-1] @ self.arrays[2 * l] + self.arrays[2 * l + 1]
            h = swish(z)
            if keep is not None:
                h = h * keep[l].astype(self.dtype)
            zs.append(z)
            hs.append(h)
        mu = hs[-1] @ self.arrays[2 * L] + self.arrays[2 * L + 1]
        raw = hs[-1] @ self.arrays[2 * L + 2] + self.arrays[2 * L + 3]
        var = so.tf_softplus(raw) + self.dtype.type(1e-4)
        return mu, var, (hs, raw, zs)

    def loss_and_grads(self, x, y, loss_scale=1.0, keep=None):
        dt = self.dtype.type
        L = self.n_layers
        mu, var, (hs, raw, zs) = self.forward(x, keep)
        y = np.asarray(y, dtype=self.dtype)
        loss = T.negative_log_likelihood(y, mu, var) * dt(loss_scale)
        c = dt(loss_scale) / dt(mu.size)
        diff = mu - y
        d_mu = c * diff / var
        d_var = dt(0.5) * c * (dt(1.0) / var - np.square(diff) / np.square(var))
        d_raw = d_var * (dt(1.0) / (dt(1.0) + np.exp(-raw)))
        grads = [None] * len(self.arrays)
        h = hs[L]
        grads[2 * L] = h.T @ d_mu
        grads[2 * L + 1] = d_mu.sum(axis=0)
        grads[2 * L + 2] = h.T @ d_raw
        grads[2 * L + 3] = d_raw.sum(axis=0)
        d_h = d_mu @ self.arrays[2 * L].T + d_raw @ self.arrays[2 * L + 2].T
        for l in range(L - 1, -1, -1):
            g = swish_grad(zs[l])
            d_z = d_h * (keep[l].astype(self.dtype) * g if keep is not None else g)
            grads[2 * l] = hs[l].T @ d_z
            grads[2 * l + 1] = d_z.sum(axis=0)
            if l > 0:
                d_h = d_z @ self.arrays[2 * l].T
        return loss, grads


class EnsembleTrainer(T.EnsembleTrainer):
    """train_oracle.EnsembleTrainer over swish members."""

    def __init__(self, members, dtype=np.float32, **kw):
        super().__init__(members, dtype=dtype, **kw)
        self.nets = [MemberNet(n.arrays, dtype) for n in self.nets]


def planner(c, objective='penalty', **kw):
    """tests.helpers.oracle_planner with the swish ensemble in its transition model."""
    from tests import helpers
    pl = helpers.oracle_planner(c, objective, **kw)
    pl.model.model = MlpEnsemble(c['weights'], dtype=pl.model.model.dt)
    return pl
