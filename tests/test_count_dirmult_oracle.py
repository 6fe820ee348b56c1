"""The Dirichlet-multinomial count likelihood (MVG_COUNT_DIRMULT) on the CPU: the FP64 restatement is the predictive
ratio of the closed-form marginal, the lnΓ-difference form the device uses for births and tables agrees with an exact
sum of logs, and the FP32 mirror of the device's stage A plus the common stage B agrees with the FP64 row log-weights."""
import math

import numpy as np
import pytest
from scipy.special import gammaln

from conftest import make_count_view
import pydirmult

LN2 = math.log(2.0)


def logm(rows, cv, beta):
    """Closed-form collapsed marginal of the rows of one dish (no multinomial coefficients)."""
    W = cv["vocab"]
    c = np.zeros(W)
    for i in rows:
        j0, j1 = cv["rowptr"][i], cv["rowptr"][i + 1]
        np.add.at(c, cv["col"][j0:j1], cv["val"][j0:j1])
    return float(np.sum(gammaln(beta + c) - gammaln(beta)) - (gammaln(W * beta + c.sum()) - gammaln(W * beta)))


def _bursty_view(n, vocab, z, k, seed, long_row=None):
    cv = make_count_view(n, vocab, z, k, seed=seed, mean_len=25, concentration=0.02)
    if long_row is not None:                      # one long, repetitive document
        rng = np.random.default_rng(seed + 100)
        r = rng.multinomial(long_row, rng.dirichlet(np.full(vocab, 0.05)))
        nz = np.nonzero(r)[0]
        rows = [(cv["col"][cv["rowptr"][i]:cv["rowptr"][i + 1]], cv["val"][cv["rowptr"][i]:cv["rowptr"][i + 1]]) for i in range(n)]
        rows[0] = (nz.astype(np.int32), r[nz].astype(np.float32))
        cv["rowptr"] = np.concatenate([[0], np.cumsum([len(c) for c, _ in rows])]).astype(np.int32)
        cv["col"] = np.concatenate([c for c, _ in rows]).astype(np.int32)
        cv["val"] = np.concatenate([v for _, v in rows]).astype(np.float32)
    return cv


def _state(oracle, views, cap, tab, dish, beta=0.5):
    o = pydirmult.DirmultState(views, cap, seed=5, count_beta=beta)
    o.set_assignment(tab, dish)
    return o


@pytest.mark.parametrize("beta", [0.5, 0.05])
def test_fp64_formula_is_the_predictive_ratio_of_the_marginal(oracle, beta):
    n, k_true, cap = 80, 4, 32
    rng = np.random.default_rng(1)
    z = rng.integers(0, k_true, n)
    cv = _bursty_view(n, 40, z, k_true, seed=2)
    assert cv["val"].max() >= 5                   # repeated words: where the plug-in and the exact form differ
    tab = z.astype(np.int32)                      # dish k = table k
    dish = np.full((1, cap), -1, np.int32)
    dish[0, :k_true] = np.arange(k_true)
    o = _state(oracle, [cv], cap, tab, dish, beta)
    members = [list(np.nonzero(z == k)[0]) for k in range(k_true)]
    for i in range(0, n, 3):
        own = int(z[i])
        for k in range(k_true):
            S = members[k]
            if k == own:                          # leave-one-out: the predictive under S \ {x}
                rest = [r for r in S if r != i]
                want = logm(S, cv, beta) - logm(rest, cv, beta)
                got = o.counts_log_f_vk(0, k, i, loo=True)
            else:
                want = logm(S + [i], cv, beta) - logm(S, cv, beta)
                got = o.counts_log_f_vk(0, k, i)
            assert abs(got - want) <= 1e-12 * max(1.0, abs(want)), (i, k, got, want)
        want = logm([i], cv, beta)
        assert abs(o.counts_log_f_new(0, i) - want) <= 1e-12 * max(1.0, abs(want)), i
    total = sum(logm(S, cv, beta) for S in members)
    assert abs(o.log_marginal_counts(0) - total) <= 1e-12 * abs(total)


def _lgamma_diff(a, x, loop=16):
    """Python statement of csrc/mv_device.cuh:lgamma_diff (the device's births, denominators and marginal)."""
    if x <= loop:
        return sum(math.log(a + j) for j in range(x))
    s = 0.0
    while a < loop:
        s += math.log(a)
        a += 1.0
        x -= 1
    b = a + x

    def tail(zz):
        r = 1.0 / zz
        r2 = r * r
        return r * (1.0 / 12 - r2 * (1.0 / 360 - r2 * (1.0 / 1260 - r2 * (1.0 / 1680))))
    return s + (a - 0.5) * math.log1p(x / a) + x * (math.log(b) - 1.0) + (tail(b) - tail(a))


def test_lgamma_difference_form_agrees_with_the_sum_of_logs():
    """lnΓ(a + x) - lnΓ(a) without cancellation: within 1e-14 relative (4e-16 measured) of the exactly summed logs over the range of
    pseudo-counts, dish totals and row lengths the sampler meets."""
    worst = 0.0
    for a in (0.05, 0.5, 3.7, 16.0, 17.5, 445 * 0.5, 6504.5, 2.5e5, 3.0e6):
        for x in (17, 18, 40, 100, 1000, 5000):
            exact = math.fsum(math.log(a + j) for j in range(x))
            worst = max(worst, abs(_lgamma_diff(a, x) - exact) / abs(exact))
    assert worst < 1e-14, worst


def _device_tables(o, v, cv, P, beta):
    """What k_counts_tables builds for view v: l2c / cnt_d per (word, table slot) and den per (row length, slot)."""
    cap, W = o.cap, cv["vocab"]
    nmax = int(max(cv["val"][cv["rowptr"][i]:cv["rowptr"][i + 1]].sum() for i in range(o.n)))
    l2c = np.zeros((W, cap), np.float32)
    cd = np.zeros((W, cap), np.int32)
    den = np.zeros((nmax + 1, cap), np.float32)
    for t in range(cap):
        k = P["dish"][v][t]
        if k < 0:
            continue
        cd[:, t] = o.cd[v][k]
        l2c[:, t] = np.log2(beta + o.cd[v][k].astype(np.float64)).astype(np.float32)
        base = W * beta + float(o.ctot[v][k])
        den[1:, t] = np.cumsum(np.log2(base + np.arange(nmax, dtype=np.float64))).astype(np.float32)
    return l2c, cd, den


def test_fp32_mirror_of_stage_a_agrees_with_fp64(oracle):
    """mvod_stageA_counts_f32 on the device's tables + mvo_stageB_f32_mixed: log-weights within 2e-5 of the FP64
    restatement (the bound of the plug-in count test), for two count views, dishes with several tables, a 1 500-token row."""
    n, k_true, cap, beta = 300, 5, 32, 0.5
    rng = np.random.default_rng(7)
    z = rng.integers(0, k_true, n)
    views = [_bursty_view(n, 120, z, k_true, seed=3, long_row=1500), _bursty_view(n, 60, (z + 1) % k_true, k_true, seed=4)]
    tab = (z + k_true * (rng.random(n) < 0.3)).astype(np.int32)      # dish k at tables k and k + k_true
    dish = np.full((2, cap), -1, np.int32)
    dish[:, :2 * k_true] = np.arange(2 * k_true) % k_true
    o = _state(oracle, views, cap, tab, dish, beta)
    P = o.make_params()
    assert np.all(P["AN"] == 1.0) and np.all(P["CN"] == 0.0)
    ps = oracle.params_struct(P)
    kind = np.ones(2, np.int32)
    tabs = [_device_tables(o, v, views[v], P, beta) for v in range(2)]
    L = oracle.lib()
    worst = 0.0
    for i in range(n):
        t0 = tab[i]
        acc = np.empty((2, cap), np.float32)
        loo = np.empty(2, np.float32)
        q = np.empty(2, np.float32)
        for v, cv in enumerate(views):
            j0, j1 = cv["rowptr"][i], cv["rowptr"][i + 1]
            k0 = P["dish"][v][t0]
            c1 = np.float32(cv["vocab"] * beta + float(o.ctot[v][k0]))
            acc[v], loo[v] = pydirmult.stageA_counts_dm_f32(cv["col"][j0:j1], cv["val"][j0:j1], *tabs[v], t0, beta, c1)
            q[v] = np.float32(-o.counts_log_f_new(v, i) / LN2)
        u = L.mvo_uf(5, 0, 0, 0, 0, i)
        _, lw32 = oracle.stageB_f32_mixed(ps, kind, acc, q, loo, t0, u, want_lw=True)
        lw64 = o.row_logweights(i) / LN2
        ok = np.isfinite(lw64)
        assert np.all(lw32[~ok] < -1e29)
        worst = max(worst, float(np.max(np.abs(lw32[ok] - lw64[ok]) / np.maximum(1.0, np.abs(lw64[ok])))))
    assert worst < 2e-5, worst
