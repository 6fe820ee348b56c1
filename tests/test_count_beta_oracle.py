"""The FP64 restatement of the count-view beta step (oracle/pycountbeta.py) on the CPU: its L(beta) is the collapsed
Dirichlet-multinomial marginal of the partition, and the Metropolis-Hastings chain it defines samples the posterior of
beta at a fixed partition (the quadrature mean, which a missing Jacobian term would miss by far)."""
import math

import numpy as np
import pytest
from scipy.special import gammaln

from conftest import make_count_view
import pycountbeta as pcb
import pydirmult


def _counts_of(cv, z, k_true):
    W = cv["vocab"]
    c = np.zeros((k_true, W), np.int64)
    for i in range(len(cv["rowptr"]) - 1):
        j0, j1 = cv["rowptr"][i], cv["rowptr"][i + 1]
        np.add.at(c[z[i]], cv["col"][j0:j1], cv["val"][j0:j1].astype(np.int64))
    return c


def _closed_form(c, W, beta):
    """sum over dishes of lnΓ(W beta) - lnΓ(W beta + C_k) + sum_w lnΓ(beta + c_kw) - lnΓ(beta), every word included."""
    tot = 0.0
    for row in c:
        tot += float(np.sum(gammaln(beta + row) - gammaln(beta))) - (gammaln(W * beta + row.sum()) - gammaln(W * beta))
    return tot


@pytest.mark.parametrize("beta", [0.5, 0.05, 3.0])
def test_restated_marginal_is_the_closed_form_and_the_oracle_marginal(oracle, beta):
    n, k_true, cap, W = 300, 5, 32, 60
    rng = np.random.default_rng(3)
    z = rng.integers(0, k_true, n)
    cv = make_count_view(n, W, z, k_true, seed=4, mean_len=20, concentration=0.05)
    c = _counts_of(cv, z, k_true)
    live = c.sum(axis=1) > 0
    t = pcb.CountBetaTarget(c[live], c[live].sum(axis=1), W)
    want = _closed_form(c[live], W, beta)
    assert abs(t.L(beta) - want) <= 1e-12 * abs(want)
    # the oracle's marginal at the handle's beta (dish k = table k)
    dish = np.full((1, cap), -1, np.int32)
    dish[0, :k_true] = np.arange(k_true)
    o = pydirmult.DirmultState([cv], cap, seed=5, count_beta=beta)
    o.set_assignment(z.astype(np.int32), dish)
    got = o.log_marginal_counts(0)
    assert abs(t.L(beta) - got) <= 1e-12 * abs(got)
    # the device's reading of the tables: the lowest table slot of each live dish
    cd = np.zeros((W, cap), np.int64)
    cd[:, :k_true] = c.T
    counts, totals = pcb.dish_counts(cd, dish[0], np.bincount(z, minlength=cap))
    assert pcb.CountBetaTarget(counts, totals, W).L(beta) == t.L(beta)


def test_one_word_vocabulary_has_no_likelihood():
    t = pcb.CountBetaTarget([[7], [30], [1]], [7, 30, 1], 1)
    for beta in (1e-4, 0.3, 1.0, 17.0, 1e4):
        assert abs(t.L(beta)) <= 1e-12 * (1.0 + abs(gammaln(beta + 30.0)))
    # ... so the step targets the prior alone: its quadrature mean is the Gamma's
    q = pcb.posterior_quadrature(t, 2.0, 3.0)
    assert abs(q["mean_beta"] - 2.0 / 3.0) < 1e-6


def test_mh_step_decision_and_proposal():
    t = pcb.CountBetaTarget([[3, 0, 1], [0, 5, 2]], [4, 7], 3)
    beta, z, s = 0.4, -0.7, 0.3
    bp = pcb.propose(beta, z, s)
    assert bp == math.exp(math.log(0.4) + 0.3 * -0.7)
    la = t.L(bp) - t.L(beta) + 2.0 * (math.log(bp) - math.log(beta)) - 1.5 * (bp - beta)
    assert pcb.log_accept(t, beta, bp, 2.0, 1.5) == la
    nxt, la2, acc = pcb.mh_step(t, beta, z, math.exp(la) * 0.999, 2.0, 1.5, s)
    assert acc and nxt == bp and la2 == la
    nxt, _, acc = pcb.mh_step(t, beta, z, min(1.0, math.exp(la) * 1.001), 2.0, 1.5, s)
    assert (not acc) and nxt == beta


def test_restated_chain_samples_the_quadrature_posterior():
    """Planted partition of make_count_view data with concentration 0.05; 20 000 steps from beta = 0.5.  The chain's
    mean of log beta is within 3 batch-means standard errors of the quadrature mean.  The data are few enough that the
    prior matters: without the Jacobian term (shape - 1 in place of shape) the target moves by about the posterior
    variance of log beta, far beyond that."""
    n, k_true, W = 60, 4, 100
    rng = np.random.default_rng(11)
    z = rng.integers(0, k_true, n)
    cv = make_count_view(n, W, z, k_true, seed=12, mean_len=30, concentration=0.05)
    c = _counts_of(cv, z, k_true)
    t = pcb.CountBetaTarget(c, c.sum(axis=1), W)
    shape, rate = 1.0, 1.0
    q = pcb.posterior_quadrature(t, shape, rate)
    assert q["mean_beta"] < 0.25                   # towards the data's concentration, away from the start
    chain = pcb.mh_chain(t, 0.5, 20000, shape, rate, 0.3, seed=13)
    lb = np.log(chain[2000:])
    se = pcb.batch_means_se(lb)
    assert abs(lb.mean() - q["mean_log_beta"]) < 3 * se + 1e-3, (lb.mean(), q, se)
    assert abs(lb.std() - q["sd_log_beta"]) < 0.25 * q["sd_log_beta"]
    # the chain without the Jacobian term samples another distribution, which the same check rejects
    no_jac = pcb.CountBetaTarget(c, c.sum(axis=1), W)
    q_wrong = pcb.posterior_quadrature(no_jac, shape - 1.0 + 1e-9, rate)
    assert abs(q_wrong["mean_log_beta"] - q["mean_log_beta"]) > 3 * se
