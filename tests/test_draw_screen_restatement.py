"""The FP64 restatement of draw screening (oracle/pyscreen.py) against known values and against the CPU restatement of
the bound in test_draw_screen_bound.py.  The GPU test test_gpu_draw_screen_oracle.py checks the device against it."""
import numpy as np
import pytest

import pyscreen as ps
from test_draw_screen_bound import T, _coefficients, _err, _params, _perturb


def _bits(x):
    return np.asarray(x, np.float32).view(np.uint32)


def test_tf32_round_known_values_ties_and_carries():
    f = np.float32
    cases = [
        (1.0, 1.0),
        (-2.5, -2.5),
        (0.0, 0.0),
        (1.0 + 2.0 ** -10, 1.0 + 2.0 ** -10),                   # representable: unchanged
        (1.0 + 2.0 ** -11, 1.0 + 2.0 ** -10),                   # exact tie: away from zero (ties-to-even gives 1)
        (-(1.0 + 2.0 ** -11), -(1.0 + 2.0 ** -10)),
        (1.0 + 2.0 ** -11 - 2.0 ** -23, 1.0),                   # just below the tie: down
        (1.0 + 3 * 2.0 ** -11, 1.0 + 2.0 ** -9),                # tie above an odd mantissa: away
        (1.0 + 5 * 2.0 ** -11, 1.0 + 3 * 2.0 ** -10),           # tie above an even mantissa: away (ties-to-even: down)
        (2.0 - 2.0 ** -11, 2.0),                                # the tie carries into the exponent
        (-(2.0 - 2.0 ** -23), -2.0),
        (f(np.nextafter(f(4.0), f(0))), 4.0),
    ]
    for x, want in cases:
        got = ps.tf32_round(np.array([x], np.float32))[0]
        assert _bits(got) == _bits(want), (x, float(got), want)
    # the low 13 bits are clear for every input
    rng = np.random.default_rng(0)
    x = (rng.standard_normal(10000) * 10.0 ** rng.uniform(-6, 6, 10000)).astype(np.float32)
    assert not np.any(_bits(ps.tf32_round(x)) & np.uint32(0x1FFF))


def test_tf32_split_is_nearly_exact():
    rng = np.random.default_rng(1)
    b = (rng.standard_normal(200000) * 10.0 ** rng.uniform(-4, 4, 200000)).astype(np.float32)
    b[:4] = [2.0 - 2.0 ** -11, -(2.0 - 2.0 ** -23), 1.0 + 2.0 ** -11, 0.0]
    hi, lo = ps.tf32_split(b)
    assert not np.any((_bits(hi) | _bits(lo)) & np.uint32(0x1FFF))
    # hi is the nearest TF32 value, so |b - hi| <= 2^-11 |b|; lo rounds the remainder to 11 bits again
    r = np.abs(b.astype(np.float64) - hi.astype(np.float64))
    assert np.all(r <= 2.0 ** -11 * np.abs(b.astype(np.float64)))
    err = np.abs(b.astype(np.float64) - hi.astype(np.float64) - lo.astype(np.float64))
    assert np.all(err <= 2.0 ** -22 * np.abs(b.astype(np.float64))), float(np.max(err / np.maximum(np.abs(b), 1e-30)))


def _as_block(p):
    """A parameter dict of test_draw_screen_bound in the get_params() layout, plus its scaled means."""
    V = p["A"].shape[0]
    P = {k: np.asarray(p[k], np.float32) for k in ("A", "A1", "C", "C1", "LM", "LM1")}
    P.update(dish=np.tile(np.arange(T, dtype=np.int32), (V, 1)), lone=np.ones((V, T), np.int32),
             LMN=np.full(2, -1e30, np.float32))
    return P, np.asarray(p["b"], np.float32).astype(np.float64)


@pytest.mark.parametrize("V", [1, 2, 3])
@pytest.mark.parametrize("kind", ["random", "along_row", "jump"])
def test_coefficients_and_error_equal_the_bound_restatement(V, kind):
    rng = np.random.default_rng(100 + V)
    for _ in range(20):
        p = {k: np.asarray(a, np.float32) for k, a in _params(rng, V).items()}
        t0 = int(rng.integers(0, T))
        x = [rng.normal(0, 2.0, 64).astype(np.float32) + p["b"][v, t0] * 0.5 for v in range(V)]
        q = _perturb(rng, p, kind, x, t0)
        P, b = _as_block(q)
        R, rb = _as_block(p)
        c0, cA, cB = _coefficients(q, p)
        k0, kA, kB = ps.coefficients(P, b, R, rb)
        e0, eA, eB = ps.coefficients(P, b, refresh=True)
        # the skip coefficients are twice the drift plus the evaluation error of the sweep's parameters
        np.testing.assert_allclose(k0 - e0, 2 * c0, rtol=1e-9, atol=1e-12)
        np.testing.assert_allclose(kA[:V] - eA[:V], 2 * cA, rtol=1e-9, atol=1e-15)
        np.testing.assert_allclose(kB[:V] - eB[:V], 2 * cB * ps.NORM_UP, rtol=1e-9, atol=1e-12)
        assert not np.any(kA[V:]) and not np.any(kB[V:]) and not np.any(eA[V:]) and not np.any(eB[V:])
        # the refresh coefficients evaluated at the row are its error budget (the |x| term rounded up by 1 + 2^-12)
        e = ps.err_row(P, b, [xv[None, :] for xv in x])[0]
        np.testing.assert_allclose(e, _err(q, x), rtol=1e-12)
        xx = np.array([np.dot(xv.astype(np.float64), xv.astype(np.float64)) for xv in x])
        at_row = e0 + sum(eA[v] * xx[v] + eB[v] * np.sqrt(xx[v]) / ps.NORM_UP for v in range(V))
        np.testing.assert_allclose(at_row, e, rtol=1e-12)


def test_coefficients_leave_out_masked_terms_and_guard_zero_slopes():
    rng = np.random.default_rng(5)
    p = {k: np.asarray(a, np.float32) for k, a in _params(rng, 2).items()}
    P, b = _as_block(p)
    base = ps.coefficients(P, b, refresh=True)
    M = {k: v.copy() for k, v in P.items()}
    M["C1"][1, 7] = -1e30                     # a table of one customer: C1 and LM1 masked
    M["LM1"][7] = -1e30
    k0, kA, kB = ps.coefficients(M, b, refresh=True)
    assert np.isfinite(k0) and k0 <= base[0] * (1 + 1e-12)
    k0s, _, _ = ps.coefficients(M, b, M, b)   # against itself: no drift, and the masked entries add nothing
    assert k0s == k0
    Z = {k: v.copy() for k, v in P.items()}
    Z["A"][0, 3] = 0.0                        # R = A1 / A is taken as 0 where A == 0
    assert ps.ratio(Z)[0, 3] == 0.0 and np.isfinite(ps.coefficients(Z, b, P, b)[2]).all()
    # R enters as max(1, R): all ratios below one leave the dot-product budget at max |b|
    S = {k: v.copy() for k, v in P.items()}
    S["A1"] = (S["A"] * np.float32(0.5)).astype(np.float32)
    _, _, kB1 = ps.coefficients(S, b, refresh=True)
    nb = np.sqrt((b ** 2).sum(axis=2)).max(axis=1)
    np.testing.assert_allclose(kB1[:2], ps.EPS_DOT * nb * ps.NORM_UP, rtol=1e-14)


def test_row_bound_never_rounds_below_fp64():
    rng = np.random.default_rng(9)
    for V in (1, 2, 3):
        for _ in range(50):
            k = np.zeros(7, np.float32)
            k[0] = rng.uniform(0, 50)
            k[1:1 + V] = 10.0 ** rng.uniform(-8, 0, V)
            k[4:4 + V] = 10.0 ** rng.uniform(-4, 2, V)
            xx = (10.0 ** rng.uniform(-3, 5, (4000, V))).astype(np.float32)
            q = ps.row_bound(k, xx)
            q64 = ps.row_bound64(k, xx)
            assert q.dtype == np.float32 and np.all(q.astype(np.float64) >= q64)
            assert np.all(q.astype(np.float64) <= q64 * (1 + 2.0 ** -20) + 1e-30)
    # device_k rounds upward too
    k = ps.device_k(1.0 / 3.0, np.array([0.1, 0.2, 0.0]), np.array([1e-7, 0.0, 0.0]))
    assert k.dtype == np.float32 and np.all(k.astype(np.float64) >= np.array([1 / 3, 0.1, 0.2, 0, 1e-7, 0, 0]))


def test_gaps_and_mode_prediction_on_a_small_block():
    rng = np.random.default_rng(3)
    V, N = 2, 500
    p = {k: np.asarray(a, np.float32) for k, a in _params(rng, V).items()}
    P, b = _as_block(p)
    X = [rng.normal(0, 2.0, (N, 64)).astype(np.float32) for _ in range(V)]
    Tt = rng.integers(0, T, N)
    lw = ps.log_weights64(X, P, b, Tt)
    g = ps.gaps64(X, P, b, Tt)
    for i in range(0, N, 37):                 # one row at a time, straight from the definitions
        xs = [x[i].astype(np.float64) for x in X]
        t0 = Tt[i]
        oth = [float(P["LM"][t]) + sum(float(P["C"][v, t]) - float(P["A"][v, t]) * (xs[v] @ xs[v]) + xs[v] @ b[v, t]
                                       for v in range(V)) for t in range(T) if t != t0]
        R = np.float32(P["A1"][:, t0] / P["A"][:, t0])
        own = float(P["LM1"][t0]) + sum(float(P["C1"][v, t0]) - float(P["A1"][v, t0]) * (xs[v] @ xs[v])
                                        + float(R[v]) * (xs[v] @ b[v, t0]) for v in range(V))
        assert lw[i, t0] == pytest.approx(own, rel=1e-13)
        assert g[i] == pytest.approx(own - max(oth), rel=1e-10, abs=1e-9)
    ref = {k: v.copy() for k, v in P.items()}
    assert ps.predict_mode(P, 10, 0, 0, ref) == ps.MODE_REFRESH
    assert ps.predict_mode(P, 10, 1, 0, ref) == ps.MODE_SKIP
    assert ps.predict_mode(P, 64, 1, 0, ref) == ps.MODE_REFRESH
    assert ps.predict_mode(P, 5, 1, 2 ** 32 - 3, ref) == ps.MODE_SKIP          # the sweep counter wraps
    assert ps.predict_mode(P, 10, 1, 0, ref, blocks=2) == ps.MODE_OFF
    for key, idx, val, want in (("dish", (0, 5), -1, ps.MODE_OFF), ("lone", (1, 2), 0, ps.MODE_OFF),
                                ("LMN", (0,), 3.0, ps.MODE_OFF), ("C1", (0, 9), -1e30, ps.MODE_REFRESH),
                                ("LM1", (9,), -1e30, ps.MODE_REFRESH), ("dish", (0, 5), 6, ps.MODE_REFRESH)):
        Q = {k: v.copy() for k, v in P.items()}
        Q[key][idx] = val
        assert ps.predict_mode(Q, 10, 1, 0, ref) == want, key
