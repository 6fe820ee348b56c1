"""GPU tests of the Dirichlet-multinomial count likelihood (MVG_COUNT_DIRMULT), against the CPU oracle:

  * dish word counts exact; the log2(beta + c) cells and the denominator table within 2e-6 of FP64;
  * stage A (k_counts_loglik_dm) and its leave-one-out value bit-exact against oracle/mv_oracle_dm.c:mvod_stageA_counts_f32
    fed the device's tables; raw draws bit-exact against mvo_stageB_f32_mixed; log-weights within 2e-5 of FP64;
  * births, deaths and counts exact against the oracle's Dirichlet-multinomial reseat, birth dish weights within 1e-8,
    hyperparameters within 1e-9; mvg_log_likelihood / saved_loglik within 1e-9 of the oracle's collapsed marginal;
  * the setter's rules, blocked sweeps with incremental counts, checkpoints, and a planted partition.
"""
import math

import numpy as np
import pytest

from conftest import make_count_view
import pydirmult

pytestmark = pytest.mark.gpu
LN2 = math.log(2.0)


def _with_long_row(cv, tokens, seed):
    """Row 0 replaced by one long, repetitive document of `tokens` tokens."""
    rng = np.random.default_rng(seed)
    W = cv["vocab"]
    r = rng.multinomial(tokens, rng.dirichlet(np.full(W, 0.05)))
    nz = np.nonzero(r)[0]
    rp = cv["rowptr"]
    col = np.concatenate([nz, cv["col"][rp[1]:]]).astype(np.int32)
    val = np.concatenate([r[nz], cv["val"][rp[1]:]]).astype(np.float32)
    rowptr = np.concatenate([[0], rp[1:] - rp[1] + len(nz)]).astype(np.int32)
    return {"rowptr": rowptr, "col": col, "val": val, "vocab": W}


def _bursty(n, vocab, z, k, seed, mean_len=25, long_row=None):
    cv = make_count_view(n, vocab, z, k, seed=seed, mean_len=mean_len, concentration=0.02)
    return _with_long_row(cv, long_row, seed + 1000) if long_row else cv


def _sampler(views, cap, seed, debug=True, model="dirmult"):
    import mvc_b200
    n = len(views[0]["rowptr"]) - 1 if isinstance(views[0], dict) else len(views[0])
    dims = [0 if isinstance(v, dict) else np.asarray(v).reshape(n, -1).shape[1] for v in views]
    s = mvc_b200.Sampler(n, dims, cap=cap, seed=seed, engine=0, debug_export=debug)
    for v, x in enumerate(views):
        if isinstance(x, dict):
            s.upload_view_csr(v, x["rowptr"], x["col"], x["val"], x["vocab"])
        else:
            s.upload_view(v, x)
    if model != "plugin":
        s.set_count_likelihood(model)
    return s


def _layout(layout):
    rng = np.random.default_rng(3)
    n, cap, k_true, sweeps = 600, 32, 5, 5
    if layout == "c4-mix":
        n, cap, sweeps = 260, 64, 3
    z = rng.integers(0, k_true, n)
    if layout == "dense+counts":
        mu = rng.normal(0, 2, (k_true, 4))
        views = [(mu[z] + rng.normal(0, 1, (n, 4))).astype(np.float32), _bursty(n, 200, z, k_true, seed=1, long_row=1200)]
    elif layout == "c4-mix":                                          # BASELINE configs[3]'s view mix: 4 dense + 4 CSR
        views = []
        for v in range(4):
            mu = rng.normal(0, 2, (k_true, 64))
            views.append((mu[z] + rng.normal(0, 1, (n, 64))).astype(np.float32))
            views.append(_bursty(n, 300 + 50 * v, z, k_true, seed=10 + v, mean_len=20, long_row=1100 if v == 0 else None))
    else:                                                             # counts+counts at cap 32, or at cap 256
        views = [_bursty(n, 200, z, k_true, seed=1, long_row=1200), _bursty(n, 64, (z + 1) % k_true, k_true, seed=2, mean_len=8)]
        if layout == "counts+counts@256":
            cap, sweeps = 256, 3
    return views, z, n, cap, sweeps


def _start(s, layout, n, V, cap):
    if layout != "counts+counts@256":
        s.init_state_reference()
        return
    rng = np.random.default_rng(9)                                    # 140 tables over 70 dishes: slots in every mask word
    tab = rng.integers(0, 140, n).astype(np.int32)
    dish = np.full((V, cap), -1, np.int32)
    dish[:, :140] = np.arange(140) // 2
    s.set_state(tab, dish, [1.0] * V, [0.5] * V, [1.0] * V, 1.0, 0.6)


@pytest.mark.parametrize("layout", ["dense+counts", "counts+counts", "c4-mix", "counts+counts@256"])
def test_dirmult_sweeps_match_the_oracle(oracle, layout):
    views, z, n, cap, sweeps = _layout(layout)
    V, seed = len(views), 91
    kind = np.array([1 if isinstance(v, dict) else 0 for v in views], np.int32)
    s = _sampler(views, cap, seed)
    _start(s, layout, n, V, cap)
    L = oracle.lib()
    births = 0
    for _ in range(sweeps):
        pre, P = s.get_state(), s.get_params()
        o = pydirmult.DirmultState(views, cap, seed=seed)
        o.alpha_v[:] = pre["alpha_v"]; o.sigma_v[:] = pre["sigma_v"]; o.tau_v[:] = pre["tau_v"]
        o.alpha_g, o.sigma_g, o.sweep = pre["alpha_g"], pre["sigma_g"], pre["sweep"]
        o.set_assignment(pre["table_of"], pre["dish_of"])
        for k in ("n_t", "n_vk", "l_vk"):
            np.testing.assert_array_equal(pre[k], getattr(o, k), err_msg=k)
        tabs = {}
        for v in range(V):
            if not kind[v]:
                np.testing.assert_allclose(pre["S1"][v], o.S1[v], rtol=1e-5, atol=1e-4)
                o.S1[v][:] = pre["S1"][v]
                continue
            l2c, cd, _ = s.get_count_tables(v)
            den, nmax = s.get_count_den(v)
            W = views[v]["vocab"]
            csum = np.concatenate([[0.0], np.cumsum(views[v]["val"], dtype=np.float64)])
            assert nmax == int((csum[views[v]["rowptr"][1:]] - csum[views[v]["rowptr"][:-1]]).max())
            tabs[v] = (l2c, cd, den)
            for t in range(cap):
                k = pre["dish_of"][v][t]
                if k < 0:
                    np.testing.assert_array_equal(cd[:, t], 0)
                    np.testing.assert_array_equal(den[:, t], 0.0)
                    continue
                np.testing.assert_array_equal(cd[:, t], o.cd[v][k], err_msg=f"dish counts view {v} table {t}")
                np.testing.assert_allclose(l2c[:, t], np.log2(o.count_beta + o.cd[v][k]), rtol=2e-6, atol=1e-6)
                den64 = np.concatenate([[0.0], np.cumsum(np.log2(W * o.count_beta + o.ctot[v][k] + np.arange(nmax, dtype=np.float64)))])
                np.testing.assert_allclose(den[:, t], den64, rtol=2e-6, atol=1e-6)
            np.testing.assert_array_equal(pre["sum_y2"][v], o.S2[v])
        o.S2[:] = pre["sum_y2"]
        Q = o.make_params()
        for k in ("dish", "lone", "single"):
            np.testing.assert_array_equal(P[k], Q[k], err_msg=k)
        for k in ("A", "C", "W", "W1", "AN", "CN", "WN", "LD", "LM", "LM1", "LMN"):
            a, b = P[k].astype(np.float64), Q[k].astype(np.float64)
            masked = b < -1e29
            np.testing.assert_array_equal(a[masked] < -1e29, True, err_msg=k)
            np.testing.assert_allclose(a[~masked], b[~masked], rtol=2e-5, atol=1e-6, err_msg=k)
        s.sweep(1, do_hyper=True)
        acc, xx, raw = s.get_debug_rows()
        loo = s.get_debug_loo()
        ps = oracle.params_struct(P)
        worst = 0.0
        for i in range(n):
            t0 = pre["table_of"][i]
            for v in range(V):
                if kind[v]:                                          # stage A of a count row: bit-exact
                    cv = views[v]
                    j0, j1 = cv["rowptr"][i], cv["rowptr"][i + 1]
                    a, l = pydirmult.stageA_counts_dm_f32(cv["col"][j0:j1], cv["val"][j0:j1], *tabs[v], t0, o.count_beta,
                                                       P["C1"][v][t0])
                    assert np.array_equal(a, acc[i, v]), (i, v)
                    assert l == loo[i, v], (i, v, l, loo[i, v])
                    q64 = -o.counts_log_f_new(v, i) / LN2                # what the new-dish term read: -log2 f_new
                    assert abs(float(xx[i, v]) - q64) <= 1e-6 * max(1.0, abs(q64)), (i, v, xx[i, v], q64)
                else:
                    a, qq = oracle.stageA_f32(views[v][i], P["m"][v])
                    assert np.array_equal(a, acc[i, v]) and qq == xx[i, v], (i, v)
            u = L.mvo_uf(seed, 0, 0, 0, pre["sweep"], i)
            ch, lw32 = oracle.stageB_f32_mixed(ps, kind, acc[i], xx[i], loo[i], t0, u, want_lw=True)
            assert ch == raw[i], (i, ch, raw[i])                      # integer draw: bit-exact
            if i % 5 == 0 or i == 0:                                 # log-weights against the FP64 restatement
                lw64 = o.row_logweights(i) / LN2
                ok = np.isfinite(lw64)
                assert np.all(lw32[~ok] < -1e29)
                worst = max(worst, float(np.max(np.abs(lw32[ok] - lw64[ok]) / np.maximum(1.0, np.abs(lw64[ok])))))
        assert worst < 2e-5, worst
        ns, rows, w = o.reseat(raw, want_births=True)
        births += ns
        post = s.get_state()
        for k in ("table_of", "n_t", "dish_of", "n_vk", "l_vk"):
            np.testing.assert_array_equal(post[k], getattr(o, k), err_msg=k)
        dns, drows, dw = s.get_debug_births()
        assert dns == ns and list(drows) == list(rows)
        if ns:
            np.testing.assert_allclose(dw, w, rtol=1e-8, atol=1e-12)
        for v in range(V):
            if not kind[v]:
                o.S1[v][:] = post["S1"][v]
        o.S2[:] = post["sum_y2"]
        o.hyper_step(use_lgamma=True)
        np.testing.assert_allclose(post["alpha_v"], o.alpha_v, rtol=1e-9)
        np.testing.assert_allclose(post["sigma_v"], o.sigma_v, rtol=1e-9)
        np.testing.assert_allclose(post["tau_v"], o.tau_v, rtol=1e-9)
        np.testing.assert_allclose([post["alpha_g"], post["sigma_g"]], [o.alpha_g, o.sigma_g], rtol=1e-9)
        _, per_view = s.log_likelihood()                            # collapsed marginal of the new partition
        for v in range(V):
            if kind[v]:
                want = o.log_marginal_counts(v)
                assert abs(per_view[v] - want) <= 1e-9 * abs(want), (v, per_view[v], want)
    assert births > 0
    s.close()


def test_saved_loglik_is_the_collapsed_marginal(oracle):
    """mvg_run's saved_loglik of a count-only chain under the Dirichlet-multinomial model: the oracle's marginal."""
    rng = np.random.default_rng(5)
    n, cap, k_true = 500, 32, 4
    z = rng.integers(0, k_true, n)
    views = [_bursty(n, 150, z, k_true, seed=21, long_row=1500), _bursty(n, 80, z, k_true, seed=22)]
    s = _sampler(views, cap, seed=4, debug=False)
    s.init_state_reference()
    tr = s.run(8, 5, 1)
    assert len(tr["loglik"]) == 3
    st = s.get_state()
    o = pydirmult.DirmultState(views, cap, seed=4)
    o.set_assignment(st["table_of"], st["dish_of"])
    want = o.log_marginal_counts(0) + o.log_marginal_counts(1)
    assert abs(tr["loglik"][-1] - want) <= 1e-9 * abs(want), (tr["loglik"][-1], want)
    tot, _ = s.log_likelihood()
    assert abs(tot - want) <= 1e-9 * abs(want)
    s.close()


def test_setter_rules():
    import mvc_b200
    rng = np.random.default_rng(1)
    n = 64
    cv = make_count_view(n, 30, rng.integers(0, 2, n), 2, seed=1)
    s = _sampler([cv], 32, seed=1, debug=False, model="plugin")
    L = mvc_b200.lib()
    assert L.mvg_set_count_likelihood(s.h, 7) == -1                   # unknown model: MVG_EINVAL
    assert L.mvg_set_count_likelihood(s.h, -1) == -1
    with pytest.raises(mvc_b200.MvgError):
        s.set_count_likelihood("exact")
    s.set_count_likelihood("dirmult")
    s.set_count_likelihood("plugin")                                  # may change until the first state call
    s.init_state_reference()
    with pytest.raises(mvc_b200.MvgError) as e:
        s.get_count_den(0)                                            # the plug-in model has no denominator table
    assert e.value.code == -4
    assert L.mvg_set_count_likelihood(s.h, 1) == -4                   # MVG_ESTATE after the first state call
    s.close()
    bad = dict(cv, val=cv["val"] + 0.5)                               # non-integer counts: refused at upload
    s = mvc_b200.Sampler(n, [0], cap=32, seed=1, engine=0)
    s.set_count_likelihood("dirmult")
    with pytest.raises(mvc_b200.MvgError) as e:
        s.upload_view_csr(0, bad["rowptr"], bad["col"], bad["val"], bad["vocab"])
    assert e.value.code == -1
    s.close()


def test_blocked_incremental_sweeps_and_checkpoints_are_deterministic(tmp_path):
    """Blocked sweeps with incremental word counts: two handles agree exactly, customers and tokens are conserved, and a
    checkpoint resumes the chain bit-identically."""
    rng = np.random.default_rng(6)
    n, cap, k_true = 800, 64, 4
    z = rng.integers(0, k_true, n)
    mu = rng.normal(0, 2, (k_true, 3))
    views = [_bursty(n, 150, z, k_true, seed=31, long_row=1300), (mu[z] + rng.normal(0, 1, (n, 3))).astype(np.float32)]

    def chain(sweeps, ckpt=None, resume=None):
        s = _sampler(views, cap, seed=8, debug=False)
        s.set_sweep_blocks(4)
        s.set_stats_mode(True, 8)
        if resume is not None:
            s.load_checkpoint(resume)
        else:
            s.init_state_reference()
        s.sweep(sweeps, do_hyper=True)
        if ckpt is not None:
            s.save_checkpoint(ckpt)
        st = s.get_state()
        _, _, ct = s.get_count_tables(0)
        s.close()
        return st, ct

    a, ct = chain(30)
    b, _ = chain(30)
    for k in ("table_of", "n_t", "dish_of", "n_vk", "alpha_v", "sigma_v"):
        np.testing.assert_array_equal(a[k], b[k], err_msg=k)
    assert int(a["n_t"].sum()) == n and (a["n_vk"].sum(1) == n).all()
    assert int(ct.sum()) == int(views[0]["val"].sum())
    ck = tmp_path / "dm.ckpt"
    chain(20, ckpt=ck)
    c, _ = chain(10, resume=ck)
    for k in ("table_of", "n_t", "dish_of", "n_vk", "alpha_v", "sigma_v"):
        np.testing.assert_array_equal(a[k], c[k], err_msg=k)


# Measured on an NVIDIA B200 (1000 W power limit): ARI 0.996 in both views, 4 tables live after 150 sweeps.
ARI_PLANTED = 0.95


def test_count_only_planted_partition_is_recovered():
    """Two count views carry the whole signal: from an over-split start the Dirichlet-multinomial chain finds the
    planted clusters."""
    rng = np.random.default_rng(12)
    n, cap, k_true = 2000, 32, 4
    z = rng.integers(0, k_true, n)
    views = [make_count_view(n, 300, z, k_true, seed=4, mean_len=40, concentration=0.05),
             make_count_view(n, 120, z, k_true, seed=5, mean_len=20, concentration=0.05)]
    s = _sampler(views, cap, seed=7, debug=False)
    tab = rng.integers(0, cap // 2, n).astype(np.int32)
    dish = np.full((2, cap), -1, np.int32)
    dish[:, :cap // 2] = np.arange(cap // 2)
    s.set_state(tab, dish, [1.0] * 2, [0.5] * 2, [1.0] * 2, 1.0, 0.6)
    s.sweep(150, do_hyper=True)
    st = s.get_state()
    assert st["n_t"].sum() == n
    aris = [s.adjusted_rand_index(v, z)[0] for v in range(2)]
    print(f"\n[dirmult planted] ARI per view {aris}, tables live {int((st['n_t'] > 0).sum())}")
    assert min(aris) > ARI_PLANTED, aris
    s.close()


def test_real_reuters_collection_in_dirmult_mode(oracle):
    """BASELINE configs[1] under the Dirichlet-multinomial model: 25 sweeps from an over-split start, then the CPU
    restatement from the device's state: counts exact, the next sweep's draws agree except on CDF edges."""
    import mvc_b200
    from mvc_b200 import reuters
    cached = reuters.load_cached()
    if cached is None:
        pytest.skip("data_cache/reuters21578_csr.npz not present (python -m mvc_b200.reuters writes it where the .sgm files are)")
    views, ids = cached
    n, cap, seed = len(ids), 64, 1999
    rng = np.random.default_rng(seed)
    tab = rng.integers(0, cap // 2, n).astype(np.int32)
    dish = np.full((3, cap), -1, np.int32)
    dish[:, :cap // 2] = np.arange(cap // 2)
    s = mvc_b200.Sampler(n, [0, 0, 0], cap=cap, seed=seed, engine=1, debug_export=True)
    for v, x in enumerate(views):
        s.upload_view_csr(v, x["rowptr"], x["col"], x["val"], x["vocab"])
    s.set_count_likelihood("dirmult")
    s.set_state(tab, dish, [1.0] * 3, [0.5] * 3, [1.0] * 3, 1.0, 0.6)
    s.sweep(25, do_hyper=True)
    pre = s.get_state()
    assert int(pre["n_t"].sum()) == n
    o = pydirmult.DirmultState(views, cap, seed=seed)
    o.alpha_v[:] = pre["alpha_v"]; o.sigma_v[:] = pre["sigma_v"]; o.tau_v[:] = pre["tau_v"]
    o.alpha_g, o.sigma_g, o.sweep = pre["alpha_g"], pre["sigma_g"], pre["sweep"]
    o.set_assignment(pre["table_of"], pre["dish_of"])
    for k in ("n_t", "n_vk", "l_vk"):
        np.testing.assert_array_equal(pre[k], getattr(o, k), err_msg=k)
    for v in range(3):
        _, cd, _ = s.get_count_tables(v)
        for t in np.nonzero(pre["n_t"] > 0)[0]:
            np.testing.assert_array_equal(cd[:, t], o.cd[v][pre["dish_of"][v][t]])
    s.sweep(1, do_hyper=True)
    _, _, raw = s.get_debug_rows()
    agree = float((o.draw_rows(threads=8) == raw).mean())
    assert agree > 0.995, agree
    print(f"\n[reuters dirmult] draw agreement with the FP64 restatement {agree:.5f}")
    s.close()
