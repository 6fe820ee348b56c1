"""The tile test of draw screening (csrc/mv_draw_screen.cuh, DESIGN.md §4.1.1): a tile of 128 rows whose least margin,
less the row bound at the tile's largest squared norms, exceeds the threshold must have every row pass the per-row
test.  Both tests are restated on the host with the device's FP32 roundings: the row bound rounded upward step by
step (oracle/pyscreen.row_bound), the subtraction rounded downward.  The summaries are formed as the device forms them:
a NaN norm enters the tile maximum as +inf and a NaN margin enters the minimum as -inf."""
import numpy as np

import pyscreen as ps

TILE = 128


def _fsub_rd(a, b):
    """FP32 a - b rounded toward -inf (__fsub_rd); a, b FP32."""
    d = np.asarray(a, np.float32).astype(np.float64) - np.asarray(b, np.float32).astype(np.float64)
    with np.errstate(invalid="ignore", over="ignore"):
        f = d.astype(np.float32)
        return np.where(f.astype(np.float64) > d, np.nextafter(f, np.float32(-np.inf)), f).astype(np.float32)


def _row_pass(k, xx, margin):
    with np.errstate(invalid="ignore", over="ignore"):
        return _fsub_rd(margin, ps.row_bound(k, xx)) > ps.THRESHOLD


def _tile_pass(k, xx, margin):
    """Tile verdicts from the summaries: [n_tiles]."""
    t = xx.shape[0] // TILE
    x = np.where(np.isnan(xx), np.float32(np.inf), xx).reshape(t, TILE, -1).max(axis=1).astype(np.float32)
    m = np.where(np.isnan(margin), np.float32(-np.inf), margin).reshape(t, TILE).min(axis=1).astype(np.float32)
    return _row_pass(k, x, m)


def _coeffs(rng, V):
    k = np.zeros(7, np.float32)
    k[0] = rng.choice([0.0, rng.uniform(0, 4), 10.0 ** rng.uniform(-6, 1)])
    for v in range(V):
        k[1 + v] = rng.choice([0.0, 10.0 ** rng.uniform(-7, -1)])
        k[4 + v] = rng.choice([0.0, 10.0 ** rng.uniform(-6, 0)])
    return k


def _check(k, xx, margin):
    tile = _tile_pass(k, xx, margin)
    rows = _row_pass(k, xx, margin).reshape(-1, TILE)
    bad = np.nonzero(tile & ~rows.all(axis=1))[0]
    assert len(bad) == 0, f"tiles {bad[:8]} pass the tile test with a failing row"
    return tile, rows


def test_tile_test_implies_every_row_random():
    rng = np.random.default_rng(7)
    n_tile_pass = n_row_only = 0
    for trial in range(200):
        V = int(rng.integers(1, 4))
        k = _coeffs(rng, V)
        n_tiles = 16
        scale = 10.0 ** rng.uniform(-2, 4)
        xx = (rng.gamma(rng.uniform(0.5, 8), 1.0, (n_tiles * TILE, V)) * scale).astype(np.float32)
        q = ps.row_bound(k, xx).astype(np.float64)
        # margins spread around the threshold plus each row's bound, so that rows and tiles fall on both sides
        margin = (ps.THRESHOLD + q + rng.normal(0, 10.0 ** rng.uniform(-3, 1), q.shape) + rng.uniform(0, 3)).astype(np.float32)
        tile, rows = _check(k, xx, margin)
        n_tile_pass += int(tile.sum())
        n_row_only += int((~tile & rows.all(axis=1)).sum())
    # adequacy: both verdicts occur, and the tile test is at times weaker than the rows (the per-row fallback matters)
    assert n_tile_pass > 200 and n_row_only > 50, (n_tile_pass, n_row_only)


def test_tile_test_implies_every_row_adversarial():
    rng = np.random.default_rng(11)
    for trial in range(300):
        V = int(rng.integers(1, 4))
        k = _coeffs(rng, V)
        xx = np.full((TILE, V), np.float32(rng.uniform(0, 500)), np.float32)
        # one row carries the largest norms, another the least margin; neighbours one ulp apart
        j_big, j_low = rng.integers(0, TILE, 2)
        xx[j_big] = np.nextafter(xx[j_big], np.float32(np.inf))
        xx[rng.integers(0, TILE)] = np.nextafter(xx[0], np.float32(0))
        q = ps.row_bound(k, xx)
        margin = (q.astype(np.float64) + ps.THRESHOLD).astype(np.float32)
        margin = np.nextafter(margin, np.float32(np.inf)) if trial % 2 else margin   # exactly at / one ulp above
        margin[j_low] = np.nextafter(margin[j_low], np.float32(-np.inf))
        if trial % 3 == 0:
            margin[:] = np.float32(rng.uniform(31, 40))
        _check(k, xx, margin)


def test_tile_summaries_of_masked_and_nan_rows_fail():
    k = np.array([0.5, 1e-3, 1e-3, 0, 1e-2, 1e-2, 0], np.float32)
    xx = np.full((4 * TILE, 2), 10.0, np.float32)
    margin = np.full(4 * TILE, 1000.0, np.float32)
    margin[TILE + 5] = np.float32(-1.0e30)       # masked: the row records no margin
    xx[2 * TILE + 9, 1] = np.nan
    margin[3 * TILE + 77] = np.nan
    tile, rows = _check(k, xx, margin)
    assert tile.tolist() == [True, False, False, False]
    assert rows.all(axis=1).tolist() == [True, False, False, False]
