"""GPU tests of the count-view beta step (mvg_set_count_beta_prior), against the FP64 restatement oracle/pycountbeta.py:

  * step parity sweep by sweep: log A within 1e-8, the same decision wherever |log u - log A| > 1e-6, the next beta
    within 2 ulp (z, u regenerated on the host from Philox domain 7);
  * after an acceptance: log2(beta + c) cells, the denominator table, -log2 f_new and C1 at the new beta within 1 FP32
    ulp, and stage A and the draws of the next sweep bit-exact against the FP32 mirror;
  * a one-word vocabulary (L = 0): the samples follow the Gamma prior; a planted partition: the posterior mean of beta;
  * graph replay, checkpoints, blocked sweeps with incremental counts, do_hyper = 0, the C ABI's rules and mvg_run's trace.
"""
import math
import os

import numpy as np
import pytest
from scipy import special, stats

from conftest import make_count_view
import pycountbeta as pcb
import pydirmult

pytestmark = pytest.mark.gpu
LN2 = math.log(2.0)


def _sampler(views, cap, seed, debug=False, prior=(1.0, 1.0, 0.3), beta0=None, engine=0):
    import mvc_b200
    n = len(views[0]["rowptr"]) - 1 if isinstance(views[0], dict) else len(views[0])
    dims = [0 if isinstance(v, dict) else np.asarray(v).reshape(n, -1).shape[1] for v in views]
    s = mvc_b200.Sampler(n, dims, cap=cap, seed=seed, engine=engine, debug_export=debug)
    for v, x in enumerate(views):
        if isinstance(x, dict):
            s.upload_view_csr(v, x["rowptr"], x["col"], x["val"], x["vocab"])
        else:
            s.upload_view(v, x)
    s.set_count_likelihood("dirmult")
    if beta0 is not None:
        s.set_count_beta(beta0)
    if prior is not None:
        s.set_count_beta_prior(*prior)
    return s


def _layout(name):
    rng = np.random.default_rng(4)
    k_true = 5
    if name == "dense+counts@32":
        n, cap = 600, 32
        z = rng.integers(0, k_true, n)
        mu = rng.normal(0, 2, (k_true, 4))
        views = [(mu[z] + rng.normal(0, 1, (n, 4))).astype(np.float32),
                 make_count_view(n, 200, z, k_true, seed=1, mean_len=25, concentration=0.02)]
    elif name == "counts+counts@64":
        n, cap = 600, 64
        z = rng.integers(0, k_true, n)
        views = [make_count_view(n, 200, z, k_true, seed=1, mean_len=25, concentration=0.02),
                 make_count_view(n, 64, (z + 1) % k_true, k_true, seed=2, mean_len=8, concentration=0.05)]
    else:                                                        # C4's view mix, small: 4 dense + 4 CSR at cap 256
        n, cap = 300, 256
        z = rng.integers(0, k_true, n)
        views = []
        for v in range(4):
            mu = rng.normal(0, 2, (k_true, 64))
            views.append((mu[z] + rng.normal(0, 1, (n, 64))).astype(np.float32))
            views.append(make_count_view(n, 300 + 50 * v, z, k_true, seed=10 + v, mean_len=20, concentration=0.03))
    return views, n, cap


def _ulps32(a, b):
    a, b = np.asarray(a, np.float32), np.asarray(b, np.float32)
    return np.abs(a.view(np.int32).astype(np.int64) - b.view(np.int32).astype(np.int64))


def _newdish_q(cv, beta):
    """-log2 f_new of every row at beta, FP64 by gammaln."""
    rp, val, W = cv["rowptr"], cv["val"].astype(np.float64), cv["vocab"]
    per = special.gammaln(beta + val) - special.gammaln(beta)
    cs = np.concatenate([[0.0], np.cumsum(per)])
    ns = np.concatenate([[0.0], np.cumsum(val)])
    lf = cs[rp[1:]] - cs[rp[:-1]]
    n = ns[rp[1:]] - ns[rp[:-1]]
    lf -= special.gammaln(W * beta + n) - special.gammaln(W * beta)
    return -lf / LN2


@pytest.mark.parametrize("layout", ["dense+counts@32", "counts+counts@64", "c4-mix@256"])
def test_step_parity_sweep_by_sweep(oracle, layout):
    import mvc_b200
    views, n, cap = _layout(layout)
    V, seed, shape, rate, step = len(views), 17, 1.0, 1.0, 0.05
    kind = np.array([1 if isinstance(v, dict) else 0 for v in views], np.int32)
    s = _sampler(views, cap, seed, debug=True, prior=(shape, rate, step))
    s.init_state_reference()
    Lb = mvc_b200.lib()
    Lo = oracle.lib()
    n_acc = n_rej = checked_after = 0
    beta = s.get_count_beta()
    assert np.all(beta[kind == 1] == np.float64(np.float32(0.5))) and np.all(beta[kind == 0] == 0.0)
    after_accept = False
    for _ in range(30):
        pre, P = s.get_state(), s.get_params()
        if after_accept:
            tabs = {v: s.get_count_tables(v) + (s.get_count_den(v)[0],) for v in range(V) if kind[v]}
        s.sweep(1, do_hyper=True)
        post = s.get_state()
        nb = s.get_count_beta()
        la_dev, acc_dev = s.get_count_beta_step()
        if after_accept:                                         # stage A and draws of the sweep after an acceptance
            acc, xx, raw = s.get_debug_rows()
            loo = s.get_debug_loo()
            ps = oracle.params_struct(P)
            for v in range(V):                                   # -log2 f_new as the draw read it, at the new beta
                if kind[v]:
                    assert _ulps32(xx[:, v], np.float32(_newdish_q(views[v], beta[v]))).max() <= 1, v
            for i in range(0, n, 3):
                t0 = pre["table_of"][i]
                for v in range(V):
                    if kind[v]:
                        cv = views[v]
                        j0, j1 = cv["rowptr"][i], cv["rowptr"][i + 1]
                        l2c, cd, _, den = tabs[v]
                        a, l = pydirmult.stageA_counts_dm_f32(cv["col"][j0:j1], cv["val"][j0:j1], l2c, cd, den, t0,
                                                           beta[v], P["C1"][v][t0])
                        assert np.array_equal(a, acc[i, v]) and l == loo[i, v], (i, v)
                    else:
                        a, qq = oracle.stageA_f32(views[v][i], P["m"][v])
                        assert np.array_equal(a, acc[i, v]) and qq == xx[i, v], (i, v)
                u = Lo.mvo_uf(seed, 0, 0, 0, pre["sweep"], i)
                ch = oracle.stageB_f32_mixed(ps, kind, acc[i], xx[i], loo[i], t0, u)
                ch = ch[0] if isinstance(ch, tuple) else ch
                assert ch == raw[i], (i, ch, raw[i])
            checked_after += 1
        after_accept = False
        for v in range(V):
            if not kind[v]:
                assert nb[v] == 0.0
                continue
            cv = views[v]
            _, cd, _ = s.get_count_tables(v)
            counts, totals = pcb.dish_counts(cd, post["dish_of"][v], post["n_vk"][v])
            t = pcb.CountBetaTarget(counts, totals, cv["vocab"])
            z = Lb.mvg_philox_normal(seed, 0, 7, v, pre["sweep"], 0)
            u = Lb.mvg_philox_uniform_f64(seed, 0, 7, v, pre["sweep"], 1)
            bp = pcb.propose(beta[v], z, step)
            la = pcb.log_accept(t, beta[v], bp, shape, rate)
            assert abs(la_dev[v] - la) <= 1e-8, (v, la_dev[v], la)
            if abs(math.log(u) - la) > 1e-6:
                assert bool(acc_dev[v]) == (math.log(u) < la), (v, la, math.log(u))
            if acc_dev[v]:
                n_acc += 1
                after_accept = True
                # (the device's exp and log are within 1 ulp each, the host's correctly rounded)
                assert abs(nb[v] - bp) <= 2 * np.spacing(bp), (v, nb[v], bp)
                # everything the next draw reads that depends on beta, at the new beta
                l2c, cd2, _ = s.get_count_tables(v)
                den, nmax = s.get_count_den(v)
                Pn = s.get_params()
                W = cv["vocab"]
                for tt in range(cap):
                    k = post["dish_of"][v][tt]
                    if k < 0:
                        continue
                    assert _ulps32(l2c[:, tt], np.float32(np.log2(nb[v] + cd2[:, tt]))).max() <= 1
                    C = float(post["sum_y2"][v][k])
                    assert Pn["C1"][v][tt] == np.float32(W * nb[v] + C)
                    a = W * nb[v] + C
                    den64 = (special.gammaln(a + np.arange(nmax + 1)) - special.gammaln(a)) / LN2
                    assert _ulps32(den[:, tt], np.float32(den64)).max() <= 1, (v, tt)
            else:
                n_rej += 1
                assert nb[v] == beta[v]
        beta = nb
    print(f"\n[count beta {layout}] {n_acc} accepted, {n_rej} rejected, {checked_after} sweeps after an acceptance checked")
    assert n_acc >= 5 and n_rej >= 5 and checked_after >= 1
    s.close()


def _prior_handle(seed, a, b, step, n=2000):
    rng = np.random.default_rng(seed)
    z = rng.integers(0, 3, n)
    lens = rng.poisson(20, n)
    cv = {"rowptr": np.concatenate([[0], np.cumsum(lens > 0)]).astype(np.int32),
          "col": np.zeros(int((lens > 0).sum()), np.int32), "val": lens[lens > 0].astype(np.float32), "vocab": 1}
    x = (rng.normal(0, 3, (3, 2))[z] + rng.normal(0, 1, (n, 2))).astype(np.float32)
    return _sampler([cv, x], 32, seed, prior=(a, b, step))


def test_one_word_vocabulary_samples_the_prior():
    a, b = 3.0, 2.0
    s = _prior_handle(5, a, b, 1.0)
    s.init_state_reference()
    tr = s.run(4000, 200, 1)
    lb = np.log(tr["count_beta"][:, 0])
    assert np.all(tr["count_beta"][:, 1] == 0.0)
    se = pcb.batch_means_se(lb)
    want_m, want_v = special.digamma(a) - math.log(b), special.polygamma(1, a)
    se_v = pcb.batch_means_se((lb - lb.mean()) ** 2)
    print(f"\n[count beta prior] mean log beta {lb.mean():.4f} (want {want_m:.4f}, se {se:.4f}), "
          f"var {lb.var():.4f} (want {want_v:.4f}, se {se_v:.4f})")
    assert abs(lb.mean() - want_m) < 4 * se
    assert abs(lb.var() - want_v) < 4 * se_v
    ks = stats.kstest(tr["count_beta"][::20, 0], stats.gamma(a, scale=1.0 / b).cdf)
    print(f"[count beta prior] KS p = {ks.pvalue:.4f} on {len(tr['count_beta'][::20])} thinned samples")
    assert ks.pvalue > 1e-3
    s.close()


def test_planted_partition_posterior_mean():
    n, W, k_true, shape, rate = 20000, 2000, 10, 1.0, 1.0
    rng = np.random.default_rng(21)
    z = rng.integers(0, k_true, n)
    cv = make_count_view(n, W, z, k_true, seed=22, mean_len=30, concentration=0.05)
    s = _sampler([cv], 64, 23, prior=(shape, rate, 0.3), beta0=0.5)
    dish = np.full((1, 64), -1, np.int32)
    dish[0, :k_true] = np.arange(k_true)
    s.set_state(z.astype(np.int32), dish, [1.0], [0.5], [1.0], 1.0, 0.6)
    tr = s.run(400, 150, 1)
    m = float(tr["count_beta"][:, 0].mean())
    c = np.zeros((k_true, W), np.int64)
    for i in range(n):
        j0, j1 = cv["rowptr"][i], cv["rowptr"][i + 1]
        np.add.at(c[z[i]], cv["col"][j0:j1], cv["val"][j0:j1].astype(np.int64))
    q = pcb.posterior_quadrature(pcb.CountBetaTarget(c, c.sum(axis=1), W), shape, rate)
    print(f"\n[count beta planted] chain mean {m:.5f}, quadrature mean at the planted partition {q['mean_beta']:.5f}")
    assert abs(m - q["mean_beta"]) <= 0.10 * q["mean_beta"]
    s.close()


def _det_views():
    rng = np.random.default_rng(6)
    n, k_true = 800, 4
    z = rng.integers(0, k_true, n)
    mu = rng.normal(0, 2, (k_true, 3))
    return [make_count_view(n, 150, z, k_true, seed=31, mean_len=25, concentration=0.03),
            (mu[z] + rng.normal(0, 1, (n, 3))).astype(np.float32)]


def _same(a, b, betas):
    for k in ("table_of", "n_t", "dish_of", "n_vk", "alpha_v", "sigma_v", "tau_v"):
        np.testing.assert_array_equal(a[k], b[k], err_msg=k)
    np.testing.assert_array_equal(betas[0], betas[1])


def test_graph_replay_checkpoint_blocked_and_no_hyper(tmp_path):
    views = _det_views()
    # graph replay (sweep(n) on a plain handle) against direct launches (a debug handle captures no graph)
    a = _sampler(views, 64, 8)
    a.init_state_reference()
    a.sweep(25, do_hyper=True)
    b = _sampler(views, 64, 8, debug=True)
    b.init_state_reference()
    for _ in range(25):
        b.sweep(1, do_hyper=True)
    ba, bb = a.get_count_beta(), b.get_count_beta()
    assert ba[0] != np.float64(np.float32(0.5))                 # the step moved beta
    _same(a.get_state(), b.get_state(), (ba, bb))
    b.close()
    # checkpoint: save after 15 more sweeps' worth, resume in a fresh handle and continue bit-identically
    ck = str(tmp_path / "beta.ckpt")
    a.save_checkpoint(ck)
    a.sweep(10, do_hyper=True)
    c = _sampler(views, 64, 8)
    c.load_checkpoint(ck)
    np.testing.assert_array_equal(c.get_count_beta(), ba)
    c.sweep(10, do_hyper=True)
    _same(a.get_state(), c.get_state(), (a.get_count_beta(), c.get_count_beta()))
    c.close()
    # do_hyper = 0 never moves beta
    before = a.get_count_beta()
    a.sweep(5, do_hyper=False)
    np.testing.assert_array_equal(a.get_count_beta(), before)
    a.close()

    def blocked():
        s = _sampler(views, 64, 9)
        s.set_sweep_blocks(4)
        s.set_stats_mode(True, 8)
        s.init_state_reference()
        s.sweep(20, do_hyper=True)
        out = s.get_state(), s.get_count_beta()
        s.close()
        return out
    (s1, b1), (s2, b2) = blocked(), blocked()
    _same(s1, s2, (b1, b2))
    assert b1[0] != np.float64(np.float32(0.5))


def test_api_rules_and_run_trace(tmp_path):
    import mvc_b200
    L = mvc_b200.lib()
    views = _det_views()
    n = len(views[1])
    # the prior's arguments and the handle's model
    s = _sampler(views, 32, 3, prior=None)
    for bad in ((0.0, 1.0, 0.3), (1.0, -1.0, 0.3), (1.0, 1.0, 0.0), (float("nan"), 1.0, 0.3), (1.0, float("inf"), 0.3)):
        assert L.mvg_set_count_beta_prior(s.h, *bad) == -1, bad
    s.close()
    p = mvc_b200.Sampler(n, [0, 3], cap=32, seed=3, engine=0)
    p.upload_view_csr(0, views[0]["rowptr"], views[0]["col"], views[0]["val"], views[0]["vocab"])
    p.upload_view(1, views[1])
    assert L.mvg_set_count_beta_prior(p.h, 1.0, 1.0, 0.3) == -4     # the plug-in likelihood: MVG_ESTATE
    p.close()
    d = mvc_b200.Sampler(n, [3], cap=32, seed=3, engine=0)
    d.upload_view(0, views[1])
    d.set_count_likelihood("dirmult")
    assert L.mvg_set_count_beta_prior(d.h, 1.0, 1.0, 0.3) == -4     # no count view: MVG_ESTATE
    d.init_state_reference()
    np.testing.assert_array_equal(d.get_count_beta(), [0.0])
    ck = tmp_path / "dense.ckpt"
    d.save_checkpoint(str(ck))                                      # a dense-only file has no beta block
    assert os.path.getsize(ck) == 8 + 8 * 8 + 4 * n + 4 * 32 + 8 * (3 + 2)
    d.close()
    s = _sampler(views, 32, 3, prior=None)
    s.init_state_reference()
    assert L.mvg_hyper_step_parts(s.h, 8) == -4                     # MVG_HYPER_COUNT_BETA without a prior
    assert L.mvg_set_count_beta_prior(s.h, 1.0, 1.0, 0.3) == -4     # after the first state call
    s.close()
    # mvg_run's trace is what get_count_beta reads after every kept sweep
    a = _sampler(views, 32, 3)
    a.init_state_reference()
    tr = a.run(30, 10, 2)
    b = _sampler(views, 32, 3)
    b.init_state_reference()
    want = []
    for it in range(30):
        b.sweep(1, do_hyper=True)
        if it >= 10 and (it - 10) % 2 == 0:
            want.append(b.get_count_beta())
    np.testing.assert_array_equal(tr["count_beta"], np.array(want))
    assert len(np.unique(tr["count_beta"][:, 0])) > 1
    # a hyper step alone moves beta at the same sweep index; MVG_HYPER_COUNT_BETA restricts it to beta
    st = b.get_state()
    for _ in range(6):
        b._ck(L.mvg_hyper_step_parts(b.h, 8))
    after = b.get_state()
    np.testing.assert_array_equal(after["tau_v"], st["tau_v"])
    np.testing.assert_array_equal(after["alpha_v"], st["alpha_v"])
    assert after["sweep"] == st["sweep"]
    # a count-view file holds beta; without the block it loads and keeps the handle's beta
    ck = tmp_path / "counts.ckpt"
    b.save_checkpoint(str(ck))
    raw = ck.read_bytes()
    beta_file = np.frombuffer(raw[-8 * 2:], np.float64)
    np.testing.assert_array_equal(beta_file, b.get_count_beta())
    old = tmp_path / "old.ckpt"
    old.write_bytes(raw[:-8 * 2])
    c = _sampler(views, 32, 3, beta0=0.7)
    c.load_checkpoint(str(old))
    np.testing.assert_array_equal(c.get_count_beta(), [np.float64(np.float32(0.7)), 0.0])
    c.close()
    a.close()
    b.close()
