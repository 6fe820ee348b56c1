"""The bound behind draw screening (DESIGN.md §4.1.1), restated on the CPU.

k_draw_screen bounds the change of a row's gap g = lw_t0 - max_{t != t0} lw_t between two parameter blocks by
Q = 2 [c0 + sum_v (cA_v |x_v|^2 + cB_v |x_v|)] and the FP32 evaluation error of each side by
e = 2^-14 (max |LM| + sum_v max |C|) + sum_v (2^-14 max A |x_v|^2 + (2^-8 + 2^-14) max(1, R) max |b| |x_v|).
Here the log-weights are evaluated in FP64 (exact restatement) and in FP32 in the kernel's order of operations, for random
and adversarial perturbations (means moved along the row, one table's mass or offset jumped), and the change of the FP32
gap must stay within Q + e(before) + e(after).
"""
import numpy as np
import pytest

T = 64


def _params(rng, V):
    p = {"LM": rng.uniform(8, 14, T), "LM1": None, "A": rng.uniform(0.2, 0.9, (V, T)), "C": rng.uniform(-200, -20, (V, T)),
         "b": rng.normal(0, 2.0, (V, T, 64))}
    p["LM1"] = p["LM"] - rng.uniform(1e-5, 1e-3, T)
    p["A1"] = p["A"] * (1 + rng.uniform(1e-5, 1e-3, (V, T)))
    p["C1"] = p["C"] + rng.uniform(-1e-3, 1e-3, (V, T))
    return p


def _f32(p):
    return {k: np.asarray(v, np.float32) for k, v in p.items()}


def _ratio(p):
    return (p["A1"].astype(np.float32) / p["A"].astype(np.float32)).astype(np.float32)


def _lw64(p, x, t0):
    """Exact log-weights of one row from the FP32 parameter values."""
    q = {k: v.astype(np.float64) for k, v in p.items()}
    V = len(x)
    xx = np.array([np.dot(xv.astype(np.float64), xv.astype(np.float64)) for xv in x])
    dots = np.stack([q["b"][v] @ x[v].astype(np.float64) for v in range(V)])      # [V, T]
    lw = q["LM"] + sum(q["C"][v] - q["A"][v] * xx[v] + dots[v] for v in range(V))
    R = _ratio(p).astype(np.float64)
    lw[t0] = q["LM1"][t0] + sum(q["C1"][v, t0] - q["A1"][v, t0] * xx[v] + R[v, t0] * dots[v, t0] for v in range(V))
    return lw


def _lw32(p, x, t0):
    """The same in FP32, in the order k_draw_tc evaluates it (base, A (-|x|^2), dot products, leave-one-out)."""
    f = np.float32
    V = len(x)
    xx = [f(np.sum(xv.astype(np.float32) ** 2, dtype=np.float32)) for xv in x]
    dots = [(p["b"][v].astype(np.float64) @ x[v].astype(np.float64)).astype(np.float32) for v in range(V)]
    base = p["LM"].astype(np.float32)
    for v in range(V):
        base = (base + p["C"][v]).astype(np.float32)
    lw = base
    for v in range(V):
        lw = (lw + p["A"][v] * f(-xx[v])).astype(np.float32)
    for v in range(V):
        lw = (lw + dots[v]).astype(np.float32)
    R = _ratio(p)
    dsum = f(0)
    for v in range(V):
        own = dots[v][t0]
        plain = f(own + f(p["A"][v, t0] * f(-xx[v]) + p["C"][v, t0]))
        loo = f(R[v, t0] * own + f(p["A1"][v, t0] * f(-xx[v]) + p["C1"][v, t0]))
        dsum = f(dsum + f(loo - plain))
    lw = lw.copy()
    lw[t0] = f(lw[t0] + f(dsum + f(p["LM1"][t0] - p["LM"][t0])))
    return lw


def _gap(lw, t0):
    return lw[t0] - np.max(np.delete(lw, t0))


def _coefficients(p, q):
    """Drift coefficients (c0, cA_v, cB_v) between two parameter blocks, as k_draw_screen computes them."""
    P, Q = ({k: v.astype(np.float64) for k, v in r.items()} for r in (p, q))
    c0 = max(np.max(np.abs(P["LM"] - Q["LM"])), np.max(np.abs(P["LM1"] - Q["LM1"])))
    c0 += sum(max(np.max(np.abs(P["C"][v] - Q["C"][v])), np.max(np.abs(P["C1"][v] - Q["C1"][v]))) for v in range(len(P["A"])))
    cA = np.maximum(np.max(np.abs(P["A"] - Q["A"]), axis=1), np.max(np.abs(P["A1"] - Q["A1"]), axis=1))
    Rp, Rq = _ratio(p).astype(np.float64), _ratio(q).astype(np.float64)
    db = np.linalg.norm(P["b"] - Q["b"], axis=2)
    dRb = np.linalg.norm(Rp[..., None] * P["b"] - Rq[..., None] * Q["b"], axis=2)
    cB = np.maximum(np.max(db, axis=1), np.max(dRb, axis=1))
    return c0, cA, cB


def _err(p, x):
    P = {k: v.astype(np.float64) for k, v in p.items()}
    V = len(x)
    nx = [np.linalg.norm(xv.astype(np.float64)) for xv in x]
    mag = max(np.max(np.abs(P["LM"])), np.max(np.abs(P["LM1"])))
    mag += sum(max(np.max(np.abs(P["C"][v])), np.max(np.abs(P["C1"][v]))) for v in range(V))
    e = 2.0 ** -14 * mag
    R = _ratio(p).astype(np.float64)
    for v in range(V):
        e += 2.0 ** -14 * max(np.max(P["A"][v]), np.max(P["A1"][v])) * nx[v] ** 2
        e += (2.0 ** -8 + 2.0 ** -14) * max(1.0, np.max(R[v])) * np.max(np.linalg.norm(P["b"][v], axis=1)) * nx[v]
    return e


def _perturb(rng, p, kind, x, t0):
    q = {k: v.copy() for k, v in p.items()}
    s = 10.0 ** rng.uniform(-6, -2)
    if kind == "random":
        for k in ("LM", "A", "C", "b"):
            q[k] = q[k] * (1 + s * rng.standard_normal(q[k].shape))
        q["LM1"] = q["LM"] - (p["LM"] - p["LM1"])
        q["A1"] = q["A"] * (p["A1"] / p["A"])
        q["C1"] = q["C"] + (p["C1"] - p["C"])
    elif kind == "along_row":          # every mean moves along the row itself: Cauchy-Schwarz is tight
        for v in range(len(x)):
            u = x[v] / np.linalg.norm(x[v])
            q["b"][v] = q["b"][v] + s * 50 * u[None, :] * np.sign(rng.standard_normal((T, 1)))
    else:                              # the best other table jumps: its mass and offset
        lw = _lw64(p, x, t0)
        lw[t0] = -np.inf
        t = int(np.argmax(lw))
        q["LM"][t] += s * 100
        q["C"][0, t] += s * 100
    return _f32(q)


@pytest.mark.parametrize("V", [1, 3])
@pytest.mark.parametrize("kind", ["random", "along_row", "jump"])
def test_gap_change_stays_within_the_bound(V, kind):
    rng = np.random.default_rng(11 + V)
    worst = 0.0
    for trial in range(40):
        p = _f32(_params(rng, V))
        t0 = int(rng.integers(0, T))
        x = [rng.normal(0, 2.0, 64).astype(np.float32) + p["b"][v, t0] * 0.5 for v in range(V)]
        q = _perturb(rng, p, kind, x, t0)
        c0, cA, cB = _coefficients(p, q)
        nx = [np.linalg.norm(xv.astype(np.float64)) for xv in x]
        xx = [nv ** 2 for nv in nx]
        drift = 2.0 * (c0 + sum(cA[v] * xx[v] + cB[v] * nx[v] for v in range(V)))
        # exact: the gap moves by at most the drift term
        d64 = abs(_gap(_lw64(q, x, t0), t0) - _gap(_lw64(p, x, t0), t0))
        assert d64 <= drift * (1 + 1e-12), (trial, d64, drift)
        # FP32 as the kernel evaluates it: within the drift plus the error term of each side
        d32 = abs(float(_gap(_lw32(q, x, t0), t0)) - float(_gap(_lw32(p, x, t0), t0)))
        bound = drift + _err(p, x) + _err(q, x)
        assert d32 <= bound, (trial, d32, bound)
        worst = max(worst, d32 / bound)
    assert worst > 0.0
