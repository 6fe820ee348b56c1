"""Draw screening (DESIGN.md §4.1.1) checked draw by draw against its FP64 restatement (oracle/pyscreen.py).

test_gpu_draw_screen.py compares chains with screening on and off.  That comparison cannot see a bound that is too small
by a few log2 units: once a row leads by more than ~24-30 its FP32 draw is its own table for every uniform, so a screened
row that should not have been is caught only with a probability of about 2^-gap.  Here every draw is inspected instead
(Sampler.get_draw_screen_record) and compared with what the design says it must be:

* the mode (off / refresh / skip), the reference copy (bit for bit) and the bound coefficients k0, kA_v, kB_v;
* the tile list: a tile is evaluated exactly when one of its rows has margin_prev - Q(row) <= 31;
* every screened row leads in FP64 by more than 31 less one evaluation error, keeps its table and its margin;
* every recorded margin lies within one evaluation error of (FP64 gap - Q), and margins are recorded where they must be.

Regimes: rows placed just above the threshold (edge), parameters that move every sweep (drift), the MUFU engine (fast),
and the calls that discard or replace a draw in flight (events).  The adequacy numbers each regime must reach were set
from a B200 run; the measured values stand next to them.
"""
import numpy as np
import pytest

import pyscreen as ps

pytestmark = pytest.mark.gpu
CAP = 64
D = 64


@pytest.fixture(scope="module")
def mvc():
    import mvc_b200
    return mvc_b200


def _sampler(mvc, views, screen=True, engine=None, incremental=False):
    s = mvc.Sampler(len(views[0]), [D] * len(views), cap=CAP, seed=2024,
                    engine=mvc.ENGINE_TCGEN05 if engine is None else engine)
    for v, x in enumerate(views):
        s.upload_view(v, x)
    if incremental:
        s.set_stats_mode(True, 64)
    s.set_draw_screen(screen)
    return s


def _dish(V):
    return np.tile(np.arange(CAP, dtype=np.int32), (V, 1))


def _set(s, tab, dish, hyp=None):
    V = s.V
    if hyp is None:
        s.set_state(tab, dish, [1.0] * V, [0.5] * V, [1.0] * V, 1.0, 0.6)
    else:
        s.set_state(tab, dish, hyp["alpha_v"], hyp["sigma_v"], hyp["tau_v"], hyp["alpha_g"], hyp["sigma_g"], hyp.get("sweep", 0))


class Watch:
    """Follows one chain op by op and checks every draw it can pair with its inputs.

    After a replayed sweep the most recent draw is the NEXT sweep's, issued at the end of the graph with the parameters
    get_params() shows now; after a direct launch (the first sweep, blocked passes, profile_sweep) it is the draw of the
    sweep just finished, with the parameters from before the call.  A replayed sweep without a draw in flight first
    launches its own draw directly; that one is not observed, only predicted (its mode, and the reference it leaves)."""

    def __init__(self, s, views):
        self.s, self.X = s, [np.ascontiguousarray(x, np.float32) for x in views]
        self.N, self.V = s.n_rows, s.V
        self.n_tiles = (self.N + 127) // 128
        self.xx = np.stack([ps.rownorms(x) for x in self.X], axis=1)
        self.tile_rows = np.minimum(128, self.N - 128 * np.arange(self.n_tiles))
        self.valid, self.ref_sweep, self.ref, self.ref_b = 0, 0, None, None
        self.margin = None                   # margins after the last draw, when known
        self.pending = False                 # a draw of the next sweep is in flight (graph replay)
        self.last = None                     # (sweep, rows that must keep their table, T) of the last observed draw
        self.blocks, self.screen = 1, True
        self.log = []                        # one entry per observed draw
        self._snap()

    # ---- inputs ---------------------------------------------------------------------------------------------------
    def _snap(self):
        P = self.s.get_params()
        b = ps.scaled_b(P)
        hi, lo = ps.tf32_split(b)
        st = self.s.get_state()
        self.cur = {"P": P, "b": b, "hi": hi, "lo": lo, "T": st["table_of"], "sweep": st["sweep"], "state": st}

    def _record(self):
        r = self.s.get_draw_screen_record()
        r["hi"], r["lo"] = (r["ref_b"][i].reshape(self.V, CAP, D) for i in (0, 1))
        return r

    # ---- ops --------------------------------------------------------------------------------------------------------
    def sweep(self, n=1):
        for _ in range(n):
            pre = self.cur
            self.s.sweep(1, True)
            self._snap()
            self._check_applied(pre)
            if not self.screen:
                self.pending = False
                continue
            rec = self._record()
            if rec["sweep"] == self.cur["sweep"]:            # graph replay: the next sweep's draw is in flight
                if not self.pending:
                    self._unobserved(pre)
                self._check(self.cur, rec)
                self.pending = True
            else:                                            # launched directly: this sweep's draw
                assert rec["sweep"] == pre["sweep"] == self.cur["sweep"] - 1, (rec["sweep"], pre["sweep"])
                self._check(pre, rec)
                self._check_applied(pre)
                self.pending = False

    def profile(self):
        """mvg_profile_sweep: the draw in flight (if any) is run again under events, directly."""
        pre = self.cur
        self.s.profile_sweep(True)
        self._snap()
        rec = self._record()
        assert rec["sweep"] == pre["sweep"] == self.cur["sweep"] - 1
        self.last = None                                     # a pending draw of this sweep is replaced by the rerun
        self._check(pre, rec)
        self._check_applied(pre)
        self.pending = False

    def hyper(self):
        self.s.hyper_step()
        self._drop()
        self._snap()

    def blocks_(self, n):
        self.s.set_sweep_blocks(n)
        self.blocks = n
        self._drop()
        self._snap()

    def screen_(self, on):
        self.s.set_draw_screen(on)
        self.screen = on
        self._drop(invalidate=True)
        self._snap()

    def set_state(self, tab, dish, hyp):
        _set(self.s, tab, dish, hyp)
        self._drop(invalidate=True)
        self._snap()

    def load(self, path):
        self.s.load_checkpoint(path)
        self._drop(invalidate=True)
        self._snap()

    def _drop(self, invalidate=False):
        self.pending = False
        self.last = None
        if invalidate:
            self.valid = 0
            self.margin = None

    # ---- checks -----------------------------------------------------------------------------------------------------
    def _check_applied(self, pre):
        """The rows the last observed draw fixed at their table sit there once its sweep has been applied."""
        if self.last is None or self.last[0] != pre["sweep"] or self.cur["sweep"] != pre["sweep"] + 1:
            return
        _, stay, T = self.last
        bad = np.nonzero(self.cur["T"][stay] != T[stay])[0]
        assert len(bad) == 0, f"sweep {pre['sweep']}: {len(bad)} screened or recorded rows changed table"
        self.last = None

    def _unobserved(self, inp):
        mode = ps.predict_mode(inp["P"], inp["sweep"], self.valid, self.ref_sweep, self.ref, self.blocks)
        self.log.append({"sweep": inp["sweep"], "mode": mode, "seen": False})
        self._advance(inp, mode)
        self.margin = None

    def _advance(self, inp, mode):
        if mode == ps.MODE_OFF:
            self.valid = 0
        elif mode == ps.MODE_REFRESH:
            self.valid, self.ref_sweep = 1, inp["sweep"]
            self.ref, self.ref_b = inp["P"], inp["hi"].astype(np.float64) + inp["lo"].astype(np.float64)
            self.ref_hi, self.ref_lo = inp["hi"], inp["lo"]

    def _check(self, inp, rec):
        P, T, s = inp["P"], inp["T"], inp["sweep"]
        V, N = self.V, self.N
        want = ps.predict_mode(P, s, self.valid, self.ref_sweep, self.ref, self.blocks)
        assert rec["mode"] == want, f"sweep {s}: device mode {rec['mode']}, predicted {want}"
        stats = self.s.draw_screen_stats()
        entry = {"sweep": s, "mode": want, "seen": True}
        self.log.append(entry)
        if want == ps.MODE_OFF:
            assert rec["valid"] == 0
            assert stats["rows_screened"] == 0 and stats["tiles_evaluated"] == self.n_tiles
            if self.margin is not None:                      # nothing is recorded
                assert np.array_equal(rec["margin"].view(np.uint32), self.margin.view(np.uint32))
            self._advance(inp, want)
            return
        b64 = inp["hi"].astype(np.float64) + inp["lo"].astype(np.float64)
        refresh = want == ps.MODE_REFRESH
        if refresh:
            assert rec["valid"] == 1 and rec["ref_sweep"] == s, (rec["valid"], rec["ref_sweep"], s)
            for k in ("dish", "A", "C", "A1", "C1", "lone", "LM", "LM1"):
                assert np.array_equal(np.asarray(rec["ref"][k]).view(np.uint32), np.asarray(P[k]).view(np.uint32)), k
            assert np.array_equal(rec["hi"].view(np.uint32), inp["hi"].view(np.uint32)), "reference mean_hi"
            assert np.array_equal(rec["lo"].view(np.uint32), inp["lo"].view(np.uint32)), "reference mean_lo"
            k0, kA, kB = ps.coefficients(P, b64, refresh=True)
        else:
            assert rec["valid"] == 1 and rec["ref_sweep"] == self.ref_sweep
            for k in ("dish", "A", "C", "A1", "C1", "lone", "LM", "LM1"):
                assert np.array_equal(np.asarray(rec["ref"][k]).view(np.uint32), np.asarray(self.ref[k]).view(np.uint32)), k
            assert np.array_equal(rec["hi"].view(np.uint32), self.ref_hi.view(np.uint32))
            assert np.array_equal(rec["lo"].view(np.uint32), self.ref_lo.view(np.uint32))
            k0, kA, kB = ps.coefficients(P, b64, self.ref, self.ref_b)
        host = np.concatenate([[k0], kA, kB])
        dev = rec["k"].astype(np.float64)
        live = np.array([True] + [v < V for v in range(3)] * 2)
        assert np.all(dev[~live] == 0.0), dev
        lo_ok = dev[live] >= host[live] * (1 - 2.0 ** -40)
        hi_ok = dev[live] <= host[live] * (1 + 2.0 ** -20)
        assert lo_ok.all() and hi_ok.all(), f"sweep {s}: k device {dev} host {host}"
        entry.update(k=dev.copy())

        Q = ps.row_bound(rec["k"], self.xx).astype(np.float64)
        g64 = ps.gaps64(self.X, P, inp["b"], T)
        e = ps.err_row(P, inp["b"], self.X)
        tile_of = np.arange(N) // 128
        if refresh:
            evaluated = np.ones(self.n_tiles, bool)
            assert stats["rows_screened"] == 0 and stats["tiles_evaluated"] == self.n_tiles
        else:
            n_eval = rec["n_eval"]
            lst = rec["tiles"][:n_eval]
            assert 0 <= n_eval <= self.n_tiles
            assert np.all((lst >= 0) & (lst < self.n_tiles)), "tile index out of range"
            assert len(np.unique(lst)) == n_eval, "tile listed twice"
            evaluated = np.zeros(self.n_tiles, bool)
            evaluated[lst] = True
            assert stats["tiles_evaluated"] == n_eval
            assert stats["rows_screened"] == int(self.tile_rows[~evaluated].sum())
            # the list: a tile is evaluated exactly when one of its rows fails margin_prev - Q > 31
            base = self.margin if self.margin is not None else rec["margin"]
            slack = base.astype(np.float64) - Q
            amb = np.abs(slack - ps.THRESHOLD) <= 1e-5 * ps.THRESHOLD
            fail = (slack <= ps.THRESHOLD) & ~amb
            passing = (slack > ps.THRESHOLD) & ~amb
            t_fail = np.bincount(tile_of, weights=fail.astype(float), minlength=self.n_tiles) > 0
            t_pass = np.bincount(tile_of, weights=passing.astype(float), minlength=self.n_tiles) == self.tile_rows
            assert not np.any(~evaluated & t_fail), f"sweep {s}: screened tiles with a failing row: {np.nonzero(~evaluated & t_fail)[0][:8]}"
            if self.margin is not None:
                assert not np.any(evaluated & t_pass), f"sweep {s}: evaluated tiles that pass: {np.nonzero(evaluated & t_pass)[0][:8]}"
            screened = ~evaluated[tile_of]
            # the core check: a screened row leads in FP64 by more than the threshold less one evaluation error
            bad = np.nonzero(screened & ~(g64 > ps.THRESHOLD - e))[0]
            assert len(bad) == 0, f"sweep {s}: screened rows {bad[:8]} lead by {g64[bad[:8]]} (error budget {e[bad[:8]]})"
            if self.margin is not None:
                assert np.array_equal(rec["margin"][screened].view(np.uint32), self.margin[screened].view(np.uint32))
            entry.update(tiles_screened=int((~evaluated).sum()), n_tiles=self.n_tiles,
                         min_slack=float(np.min(g64[screened] - ps.THRESHOLD)) if screened.any() else None)
        # the margins the draw recorded for the rows it evaluated
        ev = evaluated[tile_of]
        m = rec["margin"].astype(np.float64)
        fin = ev & (m > -1e29)
        ulp = 2.0 * np.spacing(np.abs(g64 - Q).astype(np.float32)).astype(np.float64)
        lo_b, hi_b = g64 - Q - e - ulp, g64 - Q + e
        bad = np.nonzero(fin & ~((m >= lo_b) & (m <= hi_b)))[0]
        assert len(bad) == 0, f"sweep {s}: margins {m[bad[:6]]} outside [{lo_b[bad[:6]]}, {hi_b[bad[:6]]}]"
        own_lm1 = ~ps.masked(np.asarray(P["LM1"])[T])
        must = ev & (g64 > ps.THRESHOLD + e) & own_lm1
        bad = np.nonzero(must & ~fin)[0]
        assert len(bad) == 0, f"sweep {s}: rows {bad[:8]} lead by {g64[bad[:8]]} but recorded no margin"
        bad = np.nonzero(ev & (g64 < ps.THRESHOLD - e) & fin)[0]
        assert len(bad) == 0, f"sweep {s}: rows {bad[:8]} lead by only {g64[bad[:8]]} but recorded a margin"
        stay = fin | ~ev
        self.last = (s, stay, T)
        self._advance(inp, want)
        self.margin = rec["margin"].copy()


def _assert_same(a, b):
    sa, sb = a.get_state(), b.get_state()
    for k in ("table_of", "n_t", "dish_of", "n_vk", "l_vk", "sum_y", "sum_y2", "alpha_v", "sigma_v", "tau_v",
              "alpha_g", "sigma_g", "sweep"):
        np.testing.assert_array_equal(np.asarray(sa[k]), np.asarray(sb[k]), err_msg=k)


def _modes(w):
    return [e["mode"] for e in w.log]


def _period_refreshes(w):
    return sum(1 for e in w.log if e["mode"] == ps.MODE_REFRESH and e["sweep"] >= ps.PERIOD)


# ---- data ---------------------------------------------------------------------------------------------------------------
def _separated(rng, n, V, spread=2.0, scale=None):
    z = np.concatenate([np.arange(CAP), rng.integers(0, CAP, n - CAP)]).astype(np.int32)
    mu = [rng.normal(0.0, spread, (CAP, D)) for _ in range(V)]
    X = [(mu[v][z] + rng.standard_normal((n, D))) for v in range(V)]
    if scale:
        for v, f in scale.items():
            mu[v] = mu[v] * f
            X[v] = X[v] * f
    return mu, z, X


def _hypers_after(mvc, X, z, sweeps=30):
    s = _sampler(mvc, [x.astype(np.float32) for x in X])
    _set(s, z, _dish(len(X)))
    s.sweep(sweeps, True)
    st = s.get_state()
    s.close()
    return {k: st[k] for k in ("alpha_v", "sigma_v", "tau_v", "alpha_g", "sigma_g")}


def _edge_data(mvc, n=38401, V=3, n_edge=128 * 90, seed=11):
    """Separated clusters, plus n_edge rows on the line from their own centre towards a neighbouring one, placed so that
    their FP64 lead at the start is spread over [31, 60] and sorted by it: the edge rows fill whole tiles, and tiles of
    rows just above what screening can prove sit next to tiles just below."""
    rng = np.random.default_rng(seed)
    mu, z, X = _separated(rng, n, V)
    hyp = _hypers_after(mvc, X, z)
    edge = np.arange(128, 128 + n_edge)                    # whole tiles from tile 1 on
    nb = np.array([(int(z[i]) + 1 + int(rng.integers(0, CAP - 1))) % CAP for i in edge])
    target = np.sort(rng.uniform(33.0, 58.0, n_edge))
    base = [X[v][edge] - mu[v][z[edge]] for v in range(V)]   # the row's noise
    lam = np.full(n_edge, 0.3)
    s = _sampler(mvc, [x.astype(np.float32) for x in X])
    grid = np.linspace(0.0, 1.0, 81)                       # at lambda = 1 the row sits at the neighbour's centre
    for _ in range(3):
        for v in range(V):
            X[v][edge] = mu[v][z[edge]] + base[v] + lam[:, None] * (mu[v][nb] - mu[v][z[edge]])
            s.upload_view(v, X[v].astype(np.float32))
        _set(s, z, _dish(V), hyp)
        P = s.get_params()
        b = ps.scaled_b(P)
        g = np.empty((len(grid), n_edge))
        for j, l in enumerate(grid):
            Xl = [(mu[v][z[edge]] + base[v] + l * (mu[v][nb] - mu[v][z[edge]])).astype(np.float32) for v in range(V)]
            g[j] = ps.gaps64(Xl, P, b, z[edge])
        # the lead falls along the line: interpolate where it first drops below the target
        j = np.argmax(g < target[None, :], axis=0)
        j = np.maximum(j, 1)
        r = np.arange(n_edge)
        g0, g1 = g[j - 1, r], g[j, r]
        lam = grid[j - 1] + (grid[j] - grid[j - 1]) * np.clip((g0 - target) / np.maximum(g0 - g1, 1e-12), 0.0, 1.0)
    s.close()
    for v in range(V):
        X[v][edge] = mu[v][z[edge]] + base[v] + lam[:, None] * (mu[v][nb] - mu[v][z[edge]])
    return [x.astype(np.float32) for x in X], z, hyp, edge


def _run_pair(mvc, views, z, hyp, sweeps, engine=None, incremental=False):
    """The inspected chain (screening on) and the same chain with screening off, sweep by sweep."""
    on = _sampler(mvc, views, True, engine, incremental)
    off = _sampler(mvc, views, False, engine, incremental)
    _set(on, z, _dish(len(views)), hyp)
    _set(off, z, _dish(len(views)), hyp)
    w = Watch(on, views)
    w.sweep(sweeps)
    for _ in range(sweeps):
        off.sweep(1, True)
    return w, on, off


# ---- regimes ------------------------------------------------------------------------------------------------------------
def test_edge_rows_just_above_the_threshold(mvc):
    views, z, hyp, edge = _edge_data(mvc)
    s0 = _sampler(mvc, views)
    _set(s0, z, _dish(3), hyp)
    P0 = s0.get_params()
    g0 = ps.gaps64(views, P0, ps.scaled_b(P0), z)[edge]
    s0.close()
    assert np.mean((g0 >= 31) & (g0 <= 60)) > 0.95, np.percentile(g0, [0, 5, 50, 95, 100])
    w, on, off = _run_pair(mvc, views, z, hyp, 140, incremental=True)
    _assert_same(on, off)
    assert _period_refreshes(w) >= 2, _modes(w)
    skips = [e for e in w.log if e["mode"] == ps.MODE_SKIP and e["seen"]]
    assert len(skips) > 100
    frac = np.median([e["tiles_screened"] / e["n_tiles"] for e in skips])
    slack = min(e["min_slack"] for e in skips if e["min_slack"] is not None)
    print(f"edge: median screened tile fraction {frac:.3f}, smallest g64 - 31 over screened rows {slack:.2f}")
    # measured on one B200 (1000 W): 0.744 of the tiles screened (median over skip draws), smallest slack 6.1
    assert frac > 0.6, frac
    assert slack < 10.0, slack
    on.close(); off.close()


def test_drift_parameters_move_every_sweep(mvc):
    rng = np.random.default_rng(23)
    n, V = 24000, 2
    mu, z, X = _separated(rng, n, V, scale={1: 6.0})
    hyp = _hypers_after(mvc, X, z)
    # 3 % of the rows sit midway between two tables (noise only across the line between them) and flip every sweep;
    # they fill the first tiles, so the others can be screened
    k = int(0.03 * n)
    a = z[:k].copy()
    bb = (a + 1 + rng.integers(0, CAP - 1, k)) % CAP
    for v in range(V):
        f = 6.0 if v == 1 else 1.0
        mid = 0.5 * (mu[v][a] + mu[v][bb])
        d = mu[v][bb] - mu[v][a]
        u = d / np.linalg.norm(d, axis=1, keepdims=True)
        noise = f * rng.standard_normal((k, D))
        noise -= np.sum(noise * u, axis=1, keepdims=True) * u
        X[v][:k] = mid + noise
    views = [x.astype(np.float32) for x in X]
    w, on, off = _run_pair(mvc, views, z, hyp, 140)
    _assert_same(on, off)
    assert _period_refreshes(w) >= 2, _modes(w)
    ref_k = np.median([e["k"] for e in w.log if e["mode"] == ps.MODE_REFRESH and e["seen"]], axis=0)
    skip_k = np.max([e["k"] for e in w.log if e["mode"] == ps.MODE_SKIP and e["seen"]], axis=0)
    moved = int(np.sum(on.get_state()["table_of"][:k] != z[:k]))
    print(f"drift: k at refresh {ref_k}, largest k in skip draws {skip_k}, flippers away from start {moved} of {k}")
    assert moved > k // 5
    # measured on one B200 (1000 W): k0 0.049 at refresh, up to 75 in skip draws (x1500); kB 0.108 -> 4.7 (x43) in view
    # 0 and 0.0147 -> 0.51 (x35) in the scaled view 1
    assert skip_k[0] > 100 * ref_k[0], (skip_k, ref_k)
    assert skip_k[4] > 10 * ref_k[4] and skip_k[5] > 10 * ref_k[5], (skip_k, ref_k)
    on.close(); off.close()


def test_fast_engine_one_view(mvc):
    rng = np.random.default_rng(31)
    mu, z, X = _separated(rng, 30000, 1)
    views = [x.astype(np.float32) for x in X]
    s = _sampler(mvc, views, engine=mvc.ENGINE_TCGEN05_FAST)
    _set(s, z, _dish(1))
    w = Watch(s, views)
    w.sweep(140)
    assert _period_refreshes(w) >= 2, _modes(w)
    assert sum(1 for e in w.log if e["mode"] == ps.MODE_SKIP and e["seen"]) > 100
    s.close()


def test_events_that_discard_or_replace_a_draw(mvc, tmp_path):
    rng = np.random.default_rng(47)
    n, V = 20000, 2
    mu, z, X = _separated(rng, n, V)
    views = [x.astype(np.float32) for x in X]
    s = _sampler(mvc, views)
    _set(s, z, _dish(V))
    w = Watch(s, views)

    def hyp_of(st):
        return {k: st[k] for k in ("alpha_v", "sigma_v", "tau_v", "alpha_g", "sigma_g", "sweep")}

    def last(mode):
        assert w.log[-1]["seen"] and w.log[-1]["mode"] == mode, w.log[-4:]

    w.sweep(3)
    # run up to a period refresh in flight, then throw it away: the rerun screens against the discarded reference
    for _ in range(80):
        w.sweep(1)
        if w.log[-1]["mode"] == ps.MODE_REFRESH and w.log[-1]["sweep"] >= ps.PERIOD:
            break
    last(ps.MODE_REFRESH)
    assert w.pending
    w.hyper()
    w.profile()
    last(ps.MODE_SKIP)
    w.sweep(3)
    w.hyper()                                           # the same, with the rerun launched by the next replay
    w.sweep(3)
    w.profile()                                         # a pending draw run again under events
    last(ps.MODE_SKIP)
    w.sweep(2)
    w.blocks_(2)                                        # blocked passes: no screening, no reference
    w.sweep(2)
    last(ps.MODE_OFF)
    w.blocks_(1)
    w.profile()
    last(ps.MODE_REFRESH)
    w.sweep(3)
    st = s.get_state()                                  # set_state mid-chain with some rows moved
    tab = st["table_of"].copy()
    idx = rng.choice(n, 500, replace=False)
    tab[idx] = rng.integers(0, CAP, len(idx))
    w.set_state(tab, st["dish_of"], hyp_of(st))
    w.profile()
    last(ps.MODE_REFRESH)
    w.sweep(3)
    path = tmp_path / "chain.ckpt"                      # checkpoint resume into the same handle
    s.save_checkpoint(path)
    w.sweep(2)
    w.load(path)
    w.profile()
    last(ps.MODE_REFRESH)
    w.sweep(3)
    st = s.get_state()                                  # one slot left free: no screening until it fills or is reset
    tab = st["table_of"].copy()
    tab[tab == CAP - 1] = 0
    dish = st["dish_of"].copy()
    dish[:, CAP - 1] = -1
    w.set_state(tab, dish, hyp_of(st))
    w.profile()
    last(ps.MODE_OFF)
    w.sweep(4)
    w.set_state(z, _dish(V), hyp_of(s.get_state()))
    w.profile()
    last(ps.MODE_REFRESH)
    w.sweep(3)
    w.screen_(False)                                    # switched off and on: the reference is dropped
    w.sweep(2)
    assert s.draw_screen_stats() == {"enabled": False, "rows_screened": 0, "tiles_evaluated": 0}
    w.screen_(True)
    w.profile()
    last(ps.MODE_REFRESH)
    w.sweep(3)
    seen = [e["mode"] for e in w.log if e["seen"]]
    print(f"events: {len(w.log)} draws ({len(seen)} inspected): off {seen.count(0)}, refresh {seen.count(1)}, skip {seen.count(2)}")
    assert seen.count(ps.MODE_SKIP) > 20              # measured: 103 of 113 draws inspected, 89 of them skip draws
    s.close()
