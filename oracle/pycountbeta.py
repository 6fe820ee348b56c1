"""oracle/pycountbeta.py — TEST INFRASTRUCTURE, not product code.

FP64 restatement of the Metropolis-Hastings step for the Dirichlet concentration beta of a count view under the
Dirichlet-multinomial model (mvg_set_count_beta_prior), written with scipy.special.gammaln and independent of the
device's lnΓ difference:

  L(beta) = sum over live dishes k of  sum_{w : c_kw > 0} [lnΓ(beta + c_kw) - lnΓ(beta)]  -  [lnΓ(W beta + C_k) - lnΓ(W beta)]
  log beta' = log beta + step z
  log A = L(beta') - L(beta) + shape (log beta' - log beta) - rate (beta' - beta),   accept when log u < log A

and the posterior of beta at a fixed partition, p(beta) ∝ exp(L(beta)) Gamma(beta; shape, rate), by quadrature over a
grid in log beta.
"""
from __future__ import annotations

import math

import numpy as np
from scipy.special import gammaln


def dish_counts(cd, dish_of, n_vk):
    """The word counts of the live dishes of one count view from the device's per-slot table ``cd`` [vocab][cap] (the
    counts of the dish each slot serves), ``dish_of`` [cap] and ``n_vk`` [cap]: (counts [K][vocab], totals [K]), read at
    the lowest table slot of every dish with customers."""
    cd = np.asarray(cd)
    cols, ks = [], []
    for k in range(len(n_vk)):
        if n_vk[k] <= 0:
            continue
        slots = np.nonzero(np.asarray(dish_of) == k)[0]
        if len(slots):
            cols.append(int(slots[0]))
            ks.append(k)
    counts = cd[:, cols].T.astype(np.int64)
    return counts, counts.sum(axis=1)


class CountBetaTarget:
    """L(beta) of one count view at a fixed partition, from the dish word counts [K][vocab] (or any array of the
    nonzero cells) and the dish token totals [K].  Cells are grouped by value: lnΓ is evaluated once per distinct count."""

    def __init__(self, counts, totals, vocab):
        c = np.asarray(counts, np.int64).ravel()
        self.cval, self.cmul = np.unique(c[c > 0], return_counts=True)
        self.tval, self.tmul = np.unique(np.asarray(totals, np.int64), return_counts=True)
        self.vocab = int(vocab)

    def L(self, beta):
        """L at one beta or at an array of betas."""
        b = np.asarray(beta, np.float64)[..., None]
        wb = self.vocab * b
        cells = (gammaln(b + self.cval) - gammaln(b)) @ self.cmul.astype(np.float64)
        dens = (gammaln(wb + self.tval) - gammaln(wb)) @ self.tmul.astype(np.float64)
        out = cells - dens
        return float(out) if np.ndim(beta) == 0 else out


def propose(beta, z, step):
    return math.exp(math.log(beta) + step * z)


def log_accept(target, beta, beta_prop, shape, rate):
    return (target.L(beta_prop) - target.L(beta) + shape * (math.log(beta_prop) - math.log(beta))
            - rate * (beta_prop - beta))


def mh_step(target, beta, z, u, shape, rate, step):
    """One step given the proposal normal z and the acceptance uniform u: (next beta, log A, accepted)."""
    bp = propose(beta, z, step)
    la = log_accept(target, beta, bp, shape, rate)
    acc = math.log(u) < la
    return (bp if acc else beta), la, acc


def mh_chain(target, beta0, n_steps, shape, rate, step, seed):
    """n_steps steps from beta0 with numpy's normals and uniforms: the sampled betas [n_steps]."""
    rng = np.random.default_rng(seed)
    z = rng.standard_normal(n_steps)
    u = rng.random(n_steps)
    out = np.empty(n_steps)
    b = float(beta0)
    for i in range(n_steps):
        b = mh_step(target, b, z[i], u[i], shape, rate, step)[0]
        out[i] = b
    return out


def posterior_quadrature(target, shape, rate, n=8001):
    """Posterior of beta at the fixed partition on a grid in x = log beta, density ∝ exp(L(e^x) + shape x - rate e^x)
    (the Gamma prior with the Jacobian of x): {"mean_log_beta", "sd_log_beta", "mean_beta"}.  A coarse pass finds
    where the density lives, a fine one integrates it."""
    def logp(x):
        b = np.exp(x)
        return target.L(b) + shape * x - rate * b
    x = np.linspace(-20.0, 12.0, 4001)
    lp = logp(x)
    live = x[lp > lp.max() - 60.0]
    x = np.linspace(live.min() - 0.5, live.max() + 0.5, n)
    lp = logp(x)
    w = np.exp(lp - lp.max())
    w /= w.sum()
    m = float(w @ x)
    return {"mean_log_beta": m, "sd_log_beta": float(math.sqrt(w @ (x - m) ** 2)), "mean_beta": float(w @ np.exp(x))}


def batch_means_se(x, n_batches=50):
    """Standard error of the mean of a correlated series by batch means."""
    x = np.asarray(x, np.float64)
    b = len(x) // n_batches
    means = x[: b * n_batches].reshape(n_batches, b).mean(axis=1)
    return float(means.std(ddof=1) / math.sqrt(n_batches))
