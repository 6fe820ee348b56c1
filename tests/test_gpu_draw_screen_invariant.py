"""A tile that draw screening settles is written nothing by k_draw_tc (DESIGN.md §4.1.1): its rows must already hold
choice == table_cur, and its birth and moved words must already be zero.  Checked after every sweep of screened chains,
through the read-only inspector Sampler.get_draw_rows, for every tile the screen record says was skipped: on separated
data, on parameters that drift every sweep, and across the calls that discard, replace or interrupt the chain."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu
CAP = 64
D = 64


@pytest.fixture(scope="module")
def mvc():
    import mvc_b200
    return mvc_b200


def _sampler(mvc, views):
    s = mvc.Sampler(len(views[0]), [D] * len(views), cap=CAP, seed=2024, engine=mvc.ENGINE_TCGEN05)
    for v, x in enumerate(views):
        s.upload_view(v, x)
    s.set_draw_screen(True)
    return s


def _set(s, tab, dish, hyp=None):
    V = s.V
    if hyp is None:
        s.set_state(tab, dish, [1.0] * V, [0.5] * V, [1.0] * V, 1.0, 0.6)
    else:
        s.set_state(tab, dish, hyp["alpha_v"], hyp["sigma_v"], hyp["tau_v"], hyp["alpha_g"], hyp["sigma_g"], hyp["sweep"])


def _dish(V):
    return np.tile(np.arange(CAP, dtype=np.int32), (V, 1))


def _separated(rng, n, V, spread=2.0):
    z = np.concatenate([np.arange(CAP), rng.integers(0, CAP, n - CAP)]).astype(np.int32)
    mu = [rng.normal(0.0, spread, (CAP, D)) for _ in range(V)]
    X = [(mu[v][z] + rng.standard_normal((n, D))).astype(np.float32) for v in range(V)]
    return mu, z, X


class Inspect:
    """After each call, the most recent draw's skipped tiles are checked against the buffers it left behind."""

    def __init__(self, s):
        self.s = s
        self.n = s.n_rows
        self.n_tiles = (self.n + 127) // 128
        self.skip_draws = 0
        self.tiles_checked = 0

    def check(self):
        r = self.s.get_draw_screen_record()
        if r["mode"] != 2:
            return
        skipped = np.ones(self.n_tiles, bool)
        skipped[r["tiles"][:r["n_eval"]]] = False
        d = self.s.get_draw_rows()
        rows = np.nonzero(np.repeat(skipped, 128)[:self.n])[0]
        bad = rows[d["choice"][rows] != d["table_cur"][rows]]
        assert len(bad) == 0, f"sweep {r['sweep']}: {len(bad)} rows of skipped tiles with choice != table_cur, first {bad[:8]}"
        words = np.nonzero(np.repeat(skipped, 4)[:len(d["movedmask"])])[0]
        assert not d["birthmask"][words].any(), f"sweep {r['sweep']}: birth bits in skipped tiles"
        assert not d["movedmask"][words].any(), f"sweep {r['sweep']}: moved bits in skipped tiles"
        self.skip_draws += 1
        self.tiles_checked += int(skipped.sum())

    def sweep(self, k=1):
        for _ in range(k):
            self.s.sweep(1, True)
            self.check()

    def profile(self):
        self.s.profile_sweep(True)
        self.check()


def test_separated(mvc):
    rng = np.random.default_rng(5)
    _, z, X = _separated(rng, 40000, 3)
    s = _sampler(mvc, X)
    s.set_stats_mode(True, 64)
    _set(s, z, _dish(3))
    w = Inspect(s)
    w.sweep(140)
    assert w.skip_draws > 100 and w.tiles_checked > 100 * 200, (w.skip_draws, w.tiles_checked)
    s.close()


def test_drifting_parameters(mvc):
    # 3 % of the rows sit midway between two tables and flip every sweep, so the parameters move every sweep and the
    # tiles of those rows are evaluated (and their moved words set) again and again
    rng = np.random.default_rng(23)
    n, V = 24000, 2
    mu, z, X = _separated(rng, n, V)
    k = int(0.03 * n)
    a = z[:k]
    b = (a + 1 + rng.integers(0, CAP - 1, k)) % CAP
    for v in range(V):
        X[v][:k] = (0.5 * (mu[v][a] + mu[v][b]) + 0.3 * rng.standard_normal((k, D))).astype(np.float32)
    s = _sampler(mvc, X)
    _set(s, z, _dish(V))
    w = Inspect(s)
    w.sweep(140)
    moved = int(np.sum(s.get_state()["table_of"][:k] != z[:k]))
    assert moved > k // 5, moved
    assert w.skip_draws > 100, w.skip_draws
    s.close()


def test_events(mvc, tmp_path):
    rng = np.random.default_rng(47)
    n, V = 20000, 2
    _, z, X = _separated(rng, n, V)
    s = _sampler(mvc, X)
    _set(s, z, _dish(V))
    w = Inspect(s)

    def hyp_of(st):
        return {k: st[k] for k in ("alpha_v", "sigma_v", "tau_v", "alpha_g", "sigma_g", "sweep")}

    w.sweep(70)                                         # past a period refresh
    s.hyper_step(); w.check()
    w.profile()
    w.sweep(3)
    s.hyper_step(); w.sweep(3)
    w.profile()
    s.set_sweep_blocks(2); w.sweep(2)                   # blocked passes: no screening
    s.set_sweep_blocks(1); w.profile(); w.sweep(3)
    st = s.get_state()                                  # set_state mid-chain with some rows moved
    tab = st["table_of"].copy()
    idx = rng.choice(n, 500, replace=False)
    tab[idx] = rng.integers(0, CAP, len(idx))
    _set(s, tab, st["dish_of"], hyp_of(st)); w.profile(); w.sweep(3)
    path = tmp_path / "chain.ckpt"                      # checkpoint resume into the same handle
    s.save_checkpoint(path)
    w.sweep(2)
    s.load_checkpoint(path); w.profile(); w.sweep(3)
    st = s.get_state()                                  # one slot left free: births, no screening until it fills
    tab = st["table_of"].copy()
    tab[tab == CAP - 1] = 0
    dish = st["dish_of"].copy()
    dish[:, CAP - 1] = -1
    _set(s, tab, dish, hyp_of(st)); w.profile(); w.sweep(6)
    _set(s, z, _dish(V), hyp_of(s.get_state())); w.profile(); w.sweep(3)
    s.set_draw_screen(False); w.sweep(2)                # switched off and on: the reference is dropped
    s.set_draw_screen(True); w.profile(); w.sweep(5)
    assert w.skip_draws > 20, w.skip_draws
    s.close()
