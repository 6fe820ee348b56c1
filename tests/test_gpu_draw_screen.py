"""Draw screening (tensor-core engine, DESIGN.md §4.1.1) leaves the chain exactly as it is.

Every case runs the same chain twice, screening on and off, and requires identical table_of, n_t, dish_of, n_vk, l_vk,
S1, S2 and hyperparameters after at least 300 sweeps.  The separated-cluster cases also require that screening does
something: after warm-up more than 90 % of the rows skip the draw.
"""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu
CAP = 64


def _data(n, n_views, k_true, spread=2.0, seed=7):
    rng = np.random.default_rng(seed)
    z = rng.integers(0, k_true, n).astype(np.int32)
    views = []
    for _ in range(n_views):
        mu = rng.normal(0.0, spread, (CAP, 64)).astype(np.float32)
        views.append(mu[z] + rng.standard_normal((n, 64), dtype=np.float32))
    dish = np.tile(np.arange(CAP, dtype=np.int32), (n_views, 1))
    dish[:, k_true:] = -1
    return views, z, dish


def _sampler(views, screen, incremental=True):
    import mvc_b200
    s = mvc_b200.Sampler(len(views[0]), [64] * len(views), cap=CAP, seed=1999, engine=mvc_b200.ENGINE_TCGEN05)
    for v, x in enumerate(views):
        s.upload_view(v, x)
    if incremental:
        s.set_stats_mode(True, 64)
    s.set_draw_screen(screen)
    return s


def _set(s, tab, dish, V):
    s.set_state(tab, dish, [1.0] * V, [0.5] * V, [1.0] * V, 1.0, 0.6)


def _assert_same(a, b):
    sa, sb = a.get_state(), b.get_state()
    for k in ("table_of", "n_t", "dish_of", "n_vk", "l_vk", "sum_y", "sum_y2", "alpha_v", "sigma_v", "tau_v",
              "alpha_g", "sigma_g", "sweep"):
        np.testing.assert_array_equal(np.asarray(sa[k]), np.asarray(sb[k]), err_msg=k)


def _screened_fraction(s, n, sweeps=12):
    """Median over single sweeps of the fraction of rows the most recent draw screened (a refresh sweep screens none)."""
    f = []
    for _ in range(sweeps):
        s.sweep(1, True)
        f.append(s.draw_screen_stats()["rows_screened"] / n)
    return float(np.median(f))


def _pair(views, tab, dish, **kw):
    on, off = _sampler(views, True, **kw), _sampler(views, False, **kw)
    for s in (on, off):
        _set(s, tab, dish, len(views))
    return on, off


@pytest.mark.parametrize("n_views", [1, 2, 3])
def test_separated_clusters_identical_and_mostly_screened(n_views):
    n = 200_000
    views, z, dish = _data(n, n_views, CAP)
    on, off = _pair(views, z, dish)
    for s in (on, off):
        s.sweep(300, True)
    _assert_same(on, off)
    assert on.draw_screen_stats()["enabled"] and not off.draw_screen_stats()["enabled"]
    frac = _screened_fraction(on, n)
    _screened_fraction(off, n)
    assert frac > 0.9, frac
    _assert_same(on, off)
    on.close(); off.close()


@pytest.mark.parametrize("case", ["overlapping", "free_slots", "shared_dishes"])
def test_other_regimes_identical(case):
    n = 200_000
    if case == "overlapping":
        views, z, dish = _data(n, 3, CAP, spread=0.35)
    elif case == "free_slots":                          # births and deaths: the sweep has a new-table option
        views, z, dish = _data(n, 3, CAP - 4)
    else:                                               # tables 0 and 1 share a dish in view 0
        views, z, dish = _data(n, 3, CAP)
        dish[0, 1] = 0
    on, off = _pair(views, z, dish)
    for s in (on, off):
        s.sweep(300, True)
    _assert_same(on, off)
    on.close(); off.close()


def test_blocked_sweeps_set_state_and_checkpoint_resume(tmp_path):
    n = 200_000
    views, z, dish = _data(n, 3, CAP)
    on, off = _pair(views, z, dish)
    for s in (on, off):
        s.sweep(100, True)
        s.set_sweep_blocks(3)                           # blocked passes evaluate every row and drop the reference
        s.sweep(5, True)
        s.set_sweep_blocks(1)
        s.sweep(100, True)
    _assert_same(on, off)
    # set_state mid-chain: a different seating (some rows moved) replaces the one the margins were recorded at
    st = on.get_state()
    tab = st["table_of"].copy()
    rng = np.random.default_rng(3)
    idx = rng.choice(n, 5000, replace=False)
    tab[idx] = rng.integers(0, CAP, len(idx))
    for s in (on, off):
        s.set_state(tab, st["dish_of"], st["alpha_v"], st["sigma_v"], st["tau_v"], st["alpha_g"], st["sigma_g"], st["sweep"])
        s.sweep(100, True)
    _assert_same(on, off)
    # checkpoint resume mid-chain, into a fresh handle with screening on
    path = tmp_path / "chain.ckpt"
    on.save_checkpoint(path)
    resumed = _sampler(views, True)
    resumed.load_checkpoint(path)
    for s in (resumed, off):
        s.sweep(100, True)
    _assert_same(resumed, off)
    resumed.close(); on.close(); off.close()


def test_switch_and_stats_on_the_cuda_core_engine():
    import mvc_b200
    views, z, dish = _data(4096, 2, CAP)
    s = mvc_b200.Sampler(4096, [64, 64], cap=CAP, seed=1, engine=mvc_b200.ENGINE_SIMT)
    for v, x in enumerate(views):
        s.upload_view(v, x)
    _set(s, z, dish, 2)
    s.sweep(3, True)
    assert s.draw_screen_stats() == {"enabled": False, "rows_screened": 0, "tiles_evaluated": 0}
    s.close()
