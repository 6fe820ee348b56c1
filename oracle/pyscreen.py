"""oracle/pyscreen.py — TEST INFRASTRUCTURE, not product code.

The FP64 restatement of draw screening (DESIGN.md §4.1.1, csrc/mv_draw_screen.cu): the TF32 split of the scaled means,
the coefficients of the row bound
Q = k0 + sum_v (kA_v |x_v|^2 + kB_v |x_v|), its FP32 evaluation per row, the verdict of a sweep (off / refresh / skip),
and each row's exact lead over the best other table.  Parameter blocks are dicts in the layout of Sampler.get_params():
A, C, A1, C1, dish, lone [V, cap], LM, LM1 [cap], LMN [2]; scaled means b are arrays [V, cap, D].

Only tests import this module; it needs numpy alone.
"""
from __future__ import annotations

import numpy as np

MODE_OFF, MODE_REFRESH, MODE_SKIP = 0, 1, 2      # kScreenOff, kScreenRefresh, kScreenSkip
PERIOD = 64                                      # kScreenPeriod
THRESHOLD = 31.0                                 # the dominant-option shortcut of k_draw_tc, in log2 units
EPS_ROUND = 2.0 ** -14                           # FP32 evaluation: ~30 roundings of the largest magnitudes
EPS_DOT = 2.0 ** -8 + 2.0 ** -14                 # 3-pass TF32 dot products, times max(1, R)
NORM_UP = 1.0 + 2.0 ** -12                       # |x| from the stored FMA sum of squares
SLACK = 1.0 + 2.0 ** -30                         # the FP64 arithmetic of the kernel


def masked(x):
    """A masked FP32 weight (-1e30: empty table without the customer, free slot)."""
    return ~(np.asarray(x, np.float32) > np.float32(-1.0e29))


def tf32_round(x):
    """cvt.rna.tf32.f32: round to 10 mantissa bits, nearest, ties away from zero; the result is an FP32 value."""
    bits = np.ascontiguousarray(x, np.float32).view(np.uint32)
    return ((bits + np.uint32(0x1000)) & np.uint32(0xFFFFE000)).view(np.float32)


def tf32_split(b):
    """(hi, lo) as k_finalize writes mean_hi / mean_lo from b = float32(2 A m): hi = tf32(b), lo = tf32(b - hi)."""
    b = np.ascontiguousarray(b, np.float32)
    hi = tf32_round(b)
    lo = tf32_round((b - hi).astype(np.float32))
    return hi, lo


def scaled_b(P):
    """b = float32(2 A m) per view and table slot, [V, cap, D] (pyoracle.scaled_means for every view)."""
    return np.stack([(2.0 * np.asarray(P["A"][v], np.float64)[:, None] * np.asarray(P["m"][v], np.float64)).astype(np.float32)
                     for v in range(len(P["m"]))])


def ratio(P):
    """R = A1 / A as the kernels stage it: one FP32 division, 0 where A == 0."""
    A = np.asarray(P["A"], np.float32)
    A1 = np.asarray(P["A1"], np.float32)
    with np.errstate(divide="ignore", invalid="ignore"):
        r = (A1 / A).astype(np.float32)
    return np.where(A != 0.0, r, np.float32(0.0))


def _f64(a):
    return np.asarray(a, np.float32).astype(np.float64)


def coefficients(P, b, ref=None, ref_b=None, refresh=False):
    """(k0, kA[3], kB[3]) of the row bound in FP64, before the kernel rounds them up to FP32.

    b, ref_b: [V, cap, D] scaled means in FP64 (mean_hi + mean_lo of the sweep and of the reference).  In a refresh the
    reference is the sweep itself: the drift terms are zero and only the evaluation error remains.  C1 and LM1 are left
    out where they are masked (a table of one customer)."""
    A, A1, C, C1 = (_f64(P[k]) for k in ("A", "A1", "C", "C1"))
    LM, LM1 = _f64(P["LM"]), _f64(P["LM1"])
    V = A.shape[0]
    b = np.asarray(b, np.float64)
    m1 = masked(P["C1"])
    l1 = masked(P["LM1"])
    R = ratio(P).astype(np.float64)
    nb = np.sqrt(np.sum(b * b, axis=2)).max(axis=1)                              # [V] max_t |b_vt|
    maxR = np.maximum(1.0, R.max(axis=1))
    magC = np.maximum(np.abs(C).max(axis=1), np.where(m1, 0.0, np.abs(C1)).max(axis=1))
    maxA = np.maximum(np.abs(A), np.abs(A1)).max(axis=1)
    magLM = max(np.abs(LM).max(), np.where(l1, 0.0, np.abs(LM1)).max())
    dC, dA, ndb, dLM = np.zeros(V), np.zeros(V), np.zeros(V), 0.0
    if not refresh:
        rA, rA1, rC, rC1 = (_f64(ref[k]) for k in ("A", "A1", "C", "C1"))
        rb = np.asarray(ref_b, np.float64)
        Rr = ratio(ref).astype(np.float64)
        dC = np.maximum(np.abs(C - rC).max(axis=1), np.where(m1, 0.0, np.abs(C1 - rC1)).max(axis=1))
        dA = np.maximum(np.abs(A - rA), np.abs(A1 - rA1)).max(axis=1)
        sd = np.sqrt(np.sum((b - rb) ** 2, axis=2))
        sr = np.sqrt(np.sum((R[..., None] * b - Rr[..., None] * rb) ** 2, axis=2))
        ndb = np.maximum(sd, sr).max(axis=1)
        dLM = max(np.abs(LM - _f64(ref["LM"])).max(), np.where(l1, 0.0, np.abs(LM1 - _f64(ref["LM1"]))).max())
    kA, kB = np.zeros(3), np.zeros(3)
    kA[:V] = 2.0 * dA + EPS_ROUND * maxA
    kB[:V] = (2.0 * ndb + EPS_DOT * maxR * nb) * NORM_UP
    k0 = 2.0 * (dLM + dC.sum()) + EPS_ROUND * (magLM + magC.sum())
    return float(k0), kA, kB


def device_k(k0, kA, kB):
    """The coefficients as k_draw_screen stores them: times (1 + 2^-30), rounded up to FP32, [k0, kA[3], kB[3]]."""
    return _round_up(np.concatenate([[k0], kA, kB]) * SLACK)


def _round_up(x):
    """FP64 -> the smallest FP32 value >= x."""
    x = np.asarray(x, np.float64)
    f = x.astype(np.float32)
    return np.where(f.astype(np.float64) < x, np.nextafter(f, np.float32(np.inf)), f).astype(np.float32)


def rownorms(x):
    """|x|^2 of every row as the device stores it at upload (k_rownorms: sequential FP32 FMA over the columns)."""
    x = np.asarray(x, np.float32).astype(np.float64)
    q = np.zeros(x.shape[0], np.float32)
    for d in range(x.shape[1]):
        q = (x[:, d] * x[:, d] + q.astype(np.float64)).astype(np.float32)
    return q


def row_bound(k, xx):
    """screen_row_bound of mv_ctx.h on the host: q = k0, then for every view q = fma_ru(kA_v, xx_v, q) and
    q = fma_ru(kB_v, sqrt_ru(xx_v), q).  k: [7] FP32, xx: [N, V] FP32 squared norms.  Every step rounds upward, so the
    result is never below the exact value of k0 + sum_v (kA_v xx_v + kB_v sqrt(xx_v))."""
    k = np.asarray(k, np.float32).astype(np.float64)
    xx = np.asarray(xx, np.float32)
    q = np.full(xx.shape[0], k[0], np.float64)
    for v in range(xx.shape[1]):
        x = xx[:, v].astype(np.float64)
        q = _round_up(k[1 + v] * x + q).astype(np.float64)
        q = _round_up(k[4 + v] * _round_up(np.sqrt(x)).astype(np.float64) + q).astype(np.float64)
    return q.astype(np.float32)


def row_bound64(k, xx):
    """The same in FP64 without rounding (what row_bound may never fall below)."""
    k = np.asarray(k, np.float64)
    xx = np.asarray(xx, np.float64)
    return k[0] + sum(k[1 + v] * xx[:, v] + k[4 + v] * np.sqrt(xx[:, v]) for v in range(xx.shape[1]))


def log_weights64(X, P, b, T):
    """Exact log2 weights [N, cap] of every row, from the FP32 parameter values: LM + sum_v (C - A |x|^2 + x.b) for the
    other tables, LM1 + sum_v (C1 - A1 |x|^2 + R x.b) for the row's own table T.  X: per view [N, D] FP32."""
    A, A1, C, C1 = (_f64(P[k]) for k in ("A", "A1", "C", "C1"))
    R = ratio(P).astype(np.float64)
    T = np.asarray(T, np.int64)
    rows = np.arange(len(T))
    lw = np.repeat(_f64(P["LM"])[None, :], len(T), axis=0)
    own = _f64(P["LM1"])[T].copy()
    for v, x in enumerate(X):
        x = np.asarray(x, np.float32).astype(np.float64)
        xx = np.einsum("nd,nd->n", x, x)
        dot = x @ np.asarray(b[v], np.float64).T
        lw += C[v][None, :] - A[v][None, :] * xx[:, None] + dot
        own += C1[v, T] - A1[v, T] * xx + R[v, T] * dot[rows, T]
    lw[rows, T] = own
    return lw


def gaps64(X, P, b, T):
    """Each row's lead (log2) of its own table T over the best other table, exact from the FP32 parameter values."""
    lw = log_weights64(X, P, b, T)
    rows = np.arange(len(T))
    own = lw[rows, T].copy()
    lw[rows, T] = -np.inf
    return own - lw.max(axis=1)


def err_row(P, b, X):
    """Per-row budget of one FP32 evaluation of the gap (DESIGN.md §4.1.1): 2^-14 of the magnitudes of LM, C and
    A |x|^2, and (2^-8 + 2^-14) max(1, R) max_t |b_vt| |x_v| for the dot products; |x| exact."""
    A, A1, C, C1 = (_f64(P[k]) for k in ("A", "A1", "C", "C1"))
    b = np.asarray(b, np.float64)
    m1 = masked(P["C1"])
    l1 = masked(P["LM1"])
    LM, LM1 = _f64(P["LM"]), _f64(P["LM1"])
    mag = max(np.abs(LM).max(), np.where(l1, 0.0, np.abs(LM1)).max())
    mag += sum(max(np.abs(C[v]).max(), np.where(m1[v], 0.0, np.abs(C1[v])).max()) for v in range(A.shape[0]))
    R = ratio(P).astype(np.float64)
    e = np.full(np.asarray(X[0]).shape[0], EPS_ROUND * mag)
    for v, x in enumerate(X):
        x = np.asarray(x, np.float32).astype(np.float64)
        xx = np.einsum("nd,nd->n", x, x)
        e += EPS_ROUND * max(np.abs(A[v]).max(), np.abs(A1[v]).max()) * xx
        e += EPS_DOT * max(1.0, R[v].max()) * np.sqrt(np.sum(b[v] ** 2, axis=1)).max() * np.sqrt(xx)
    return e


def predict_mode(P, sweep, valid, ref_sweep, ref, blocks=1):
    """The verdict k_draw_screen reaches for the draw of `sweep` with parameter block P: off when a table slot is free
    (a new-table option), a dish is shared or free in a view, or the sweep runs in blocked passes; refresh when no
    reference stands, the reference is PERIOD sweeps old, or a dish, a lone flag or the masking of C1, LM or LM1 differs
    from it; skip otherwise."""
    if blocks != 1 or not masked(P["LMN"]).all() or (np.asarray(P["dish"]) < 0).any() or not np.asarray(P["lone"]).all():
        return MODE_OFF
    if not valid or ((int(sweep) - int(ref_sweep)) & 0xFFFFFFFF) >= PERIOD:
        return MODE_REFRESH
    if not (np.array_equal(P["dish"], ref["dish"]) and np.array_equal(P["lone"], ref["lone"])
            and np.array_equal(masked(P["C1"]), masked(ref["C1"])) and np.array_equal(masked(P["LM"]), masked(ref["LM"]))
            and np.array_equal(masked(P["LM1"]), masked(ref["LM1"]))):
        return MODE_REFRESH
    return MODE_SKIP
