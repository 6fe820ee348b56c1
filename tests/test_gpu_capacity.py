"""Table capacities 128 and 256 (CUDA-core engine): creation rules, one-sweep parity against the CPU oracle on dense,
scalar and count views, posterior summaries with labels above slot 63, checkpoint resume, and the row-sharded chain.

The parity checks are those of tests/test_gpu_parity.py (_one_sweep_parity): parameter block against make_params, draws
bit-exact against mvo_stageB_f32 fed the device's dot products, births / dish weights against mvo_reseat, counts exact,
sums within 1e-5 of the FP64 rebuild, hyperparameters within 1e-9 of mvo_hyper_step.  The states are chosen to reach what
only the wide capacities have: more than 128 live dishes in a view (EPPF blocks 5-8), dishes served by tables in
different 64-slot mask words, free slots above 64, and all 256 slots live."""
import os
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest

ROOT = Path(__file__).resolve().parents[1]
if __name__ != "__main__":
    from conftest import make_count_view, make_mixture
    from test_gpu_parity import RTOL_STATS, _mk_mixed_sampler, _mk_sampler, _one_sweep_parity

pytestmark = pytest.mark.gpu
MVG_EUNSUPPORTED = -6


def _wide_state(n, V, cap, live, rng, singles=6):
    """Tables 0..live-1 occupied (the last `singles` by one customer each), the rest free.  View 0: dish t % 150 (more
    than 128 dishes, tables t and t + 150 share one across mask words); view 1: dish t // 2; further views: 7 t mod 200
    (mod cap when that is smaller)."""
    tab = rng.integers(0, live - singles, n).astype(np.int32)
    tab[:live] = np.arange(live)
    dish = np.full((V, cap), -1, np.int32)
    t = np.arange(live)
    for v in range(V):
        dish[v, :live] = (t % 150) if v == 0 else ((t // 2) if v == 1 else (7 * t) % min(200, cap))
    return tab, dish


def test_capacity_creation_rules():
    import mvc_b200
    for cap in (128, 256):
        s = mvc_b200.Sampler(300, [4, 4], cap=cap, seed=1)
        assert s.cap == cap
        s.close()
    for cap in (96, 512, 16):
        with pytest.raises(mvc_b200.MvgError) as e:
            mvc_b200.Sampler(300, [4, 4], cap=cap, seed=1)
        assert e.value.code == MVG_EUNSUPPORTED, cap
    # the tensor-core engine is built for cap 64: asked for explicitly at 128 it is refused at the first state call
    views, _ = make_mixture(300, [64], 4, seed=2)
    s = _mk_sampler(views, 128, seed=1, engine=mvc_b200.ENGINE_TCGEN05)
    with pytest.raises(mvc_b200.MvgError) as e:
        s.init_state_reference()
    assert e.value.code == MVG_EUNSUPPORTED
    s.close()


@pytest.mark.parametrize("dims,cap,n,live", [([64, 64, 64], 256, 4001, 230), ([8] * 5, 128, 1503, 110), ([1, 1], 256, 3001, 220)])
def test_wide_capacity_dense_parity(oracle, dims, cap, n, live):
    """engine AUTO: at cap > 64 it must be the CUDA-core engine, whose dot products are checked bit for bit."""
    views, _ = make_mixture(n, dims, 12, seed=21)
    s = _mk_sampler(views, cap, seed=77, engine=0)
    rng = np.random.default_rng(5)
    V = len(dims)
    tab, dish = _wide_state(n, V, cap, live, rng)
    s.set_state(tab, dish, np.full(V, 1.0), np.full(V, 0.5), np.full(V, 0.9), 1.0, 0.6, sweep=3)
    st = s.get_state()
    assert (st["l_vk"][0] > 0).sum() == min(150, live)
    births = 0
    for it in range(4):
        births += _one_sweep_parity(oracle, s, views, cap, 77, do_hyper=(it % 2 == 0))
    assert births > 0
    assert s.get_state()["n_t"].sum() == n
    s.close()


def test_wide_capacity_full_masks_new_table(oracle):
    """All 256 slots occupied: no birth may happen (capacity rule) and nothing is lost.  Tables may empty during a sweep,
    so the rule is checked on every sweep that starts with no free slot (the first one at least)."""
    n, cap = 256 * 5, 256
    views, _ = make_mixture(n, [4, 4], 32, seed=3)
    s = _mk_sampler(views, cap, seed=5)
    tab = (np.arange(n) % cap).astype(np.int32)
    dish = np.stack([np.arange(cap) % 200, np.arange(cap) // 2]).astype(np.int32)
    s.set_state(tab, dish, [1.0, 1.0], [0.5, 0.5], [1.0, 1.0], 5.0, 0.9)
    full_sweeps = 0
    for _ in range(3):
        full = bool((s.get_state()["n_t"] > 0).all())
        _one_sweep_parity(oracle, s, views, cap, 5, do_hyper=False)
        _, _, raw = s.get_debug_rows()
        if full:
            assert (raw >= 0).all()
            full_sweeps += 1
    assert full_sweeps >= 1
    assert s.get_state()["n_t"].sum() == n
    s.close()


def test_wide_capacity_count_views_parity(oracle):
    """The C4 view mix (4 dense D = 64 + 4 CSR) at cap 256: count tables, leave-one-out values, draws, births, counts."""
    n, cap, k_true, seed = 700, 256, 5, 91
    rng = np.random.default_rng(3)
    z = rng.integers(0, k_true, n)
    views = []
    for v in range(4):
        mu = rng.normal(0, 2, (k_true, 64))
        views.append((mu[z] + rng.normal(0, 1, (n, 64))).astype(np.float32))
        views.append(make_count_view(n, 300 + 50 * v, z, k_true, seed=10 + v, mean_len=20))
    V = len(views)
    kind = np.array([1 if isinstance(v, dict) else 0 for v in views], np.int32)
    s = _mk_mixed_sampler(views, cap, seed)
    tab, dish = _wide_state(n, V, cap, 210, rng)
    s.set_state(tab, dish, np.full(V, 1.0), np.full(V, 0.5), np.full(V, 1.0), 1.0, 0.6)
    L = oracle.lib()
    births = 0
    for it in range(3):
        pre, P = s.get_state(), s.get_params()
        o = oracle.OracleState(views, cap, seed=seed)
        o.alpha_v[:] = pre["alpha_v"]; o.sigma_v[:] = pre["sigma_v"]; o.tau_v[:] = pre["tau_v"]
        o.alpha_g, o.sigma_g, o.sweep = pre["alpha_g"], pre["sigma_g"], pre["sweep"]
        o.set_assignment(pre["table_of"], pre["dish_of"])
        for k in ("n_t", "n_vk", "l_vk"):
            np.testing.assert_array_equal(pre[k], getattr(o, k), err_msg=k)
        tabs = {}
        for v in range(V):
            if not kind[v]:
                np.testing.assert_allclose(pre["S1"][v], o.S1[v], rtol=RTOL_STATS, atol=1e-4)
                o.S1[v][:] = pre["S1"][v]
                continue
            l2t, cd, ct = s.get_count_tables(v)
            tabs[v] = (l2t, cd)
            W = views[v]["vocab"]
            for t in range(cap):                                     # dish counts as seen from every table slot: exact
                k = pre["dish_of"][v][t]
                want = o.cd[v][k] if k >= 0 else np.zeros(W, np.int64)
                np.testing.assert_array_equal(cd[:, t], want, err_msg=f"dish counts view {v} table {t}")
                if k >= 0:
                    ref = np.log2((o.count_beta + o.cd[v][k]) / (W * o.count_beta + o.ctot[v][k]))
                    np.testing.assert_allclose(l2t[:, t], ref, rtol=2e-6, atol=1e-6)
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
        for i in range(n):
            t0 = pre["table_of"][i]
            for v in range(V):
                if kind[v]:
                    cv = views[v]
                    j0, j1 = cv["rowptr"][i], cv["rowptr"][i + 1]
                    a, l, tot = oracle.stageA_counts_f32(cv["col"][j0:j1], cv["val"][j0:j1], tabs[v][0], tabs[v][1], t0,
                                                         o.count_beta, P["C1"][v][t0])
                    assert np.array_equal(a, acc[i, v]) and tot == xx[i, v], (i, v)
                    assert l == loo[i, v], (i, v, l, loo[i, v])
                else:
                    a, q = oracle.stageA_f32(views[v][i], P["m"][v])
                    assert np.array_equal(a, acc[i, v]) and q == xx[i, v], (i, v)
            u = L.mvo_uf(seed, 0, 0, 0, pre["sweep"], i)
            ch, _ = oracle.stageB_f32_mixed(ps, kind, acc[i], xx[i], loo[i], t0, u, want_lw=True)
            assert ch == raw[i], (i, ch, raw[i])
        ns, rows, w = o.reseat(raw, want_births=True)
        births += ns
        post = s.get_state()
        for k in ("table_of", "n_t", "dish_of", "n_vk", "l_vk"):
            np.testing.assert_array_equal(post[k], getattr(o, k), err_msg=k)
        dns, drows, dw = s.get_debug_births()
        assert dns == ns and list(drows) == list(rows)
        if ns:
            np.testing.assert_allclose(dw, w, rtol=1e-9, atol=1e-12)
        for v in range(V):
            if not kind[v]:
                o.S1[v][:] = post["S1"][v]
        o.S2[:] = post["sum_y2"]
        o.hyper_step(use_lgamma=True)
        np.testing.assert_allclose(post["alpha_v"], o.alpha_v, rtol=1e-9)
        np.testing.assert_allclose(post["sigma_v"], o.sigma_v, rtol=1e-9)
        np.testing.assert_allclose(post["tau_v"], o.tau_v, rtol=1e-9)
        np.testing.assert_allclose([post["alpha_g"], post["sigma_g"]], [o.alpha_g, o.sigma_g], rtol=1e-9)
    assert births > 0
    s.close()


def _ari(tab):
    """Adjusted Rand index from a contingency table (Hubert and Arabie)."""
    c2 = lambda x: x * (x - 1) / 2.0
    n = tab.sum()
    sij, sa, sb = c2(tab.astype(np.float64)).sum(), c2(tab.sum(1).astype(np.float64)).sum(), c2(tab.sum(0).astype(np.float64)).sum()
    exp = sa * sb / c2(float(n))
    return (sij - exp) / (0.5 * (sa + sb) - exp)


def test_wide_capacity_posterior_summaries():
    """Labels, ARI with a [256][n_classes] contingency table and co-clustering counts, with live labels in slots >= 64."""
    n, cap, V = 1800, 256, 2
    views, z = make_mixture(n, [3, 2], 6, seed=8)
    s = _mk_sampler(views, cap, seed=17, debug=False)
    rng = np.random.default_rng(2)
    tab = rng.integers(0, cap, n).astype(np.int32)
    tab[:cap] = np.arange(cap)
    dish = np.stack([np.arange(cap), (np.arange(cap) * 5) % cap]).astype(np.int32)
    s.set_state(tab, dish, np.full(V, 1.0), np.full(V, 0.5), np.full(V, 0.9), 1.0, 0.6)
    s.sweep(2, do_hyper=True)
    st = s.get_state()
    labels = s.cluster_labels()
    for v in range(V):
        np.testing.assert_array_equal(labels[v], st["dish_of"][v][st["table_of"]])
        assert labels[v].max() >= 64
        ari, ctab = s.adjusted_rand_index(v, z)
        assert ctab.shape == (cap, int(z.max()) + 1)
        ref = np.zeros_like(ctab)
        np.add.at(ref, (labels[v], z), 1)
        np.testing.assert_array_equal(ctab, ref)
        assert abs(ari - _ari(ref)) < 1e-12
    for view in (-1, 0):                                              # tables, then the dishes of view 0
        s.coclustering_begin(view)
        want = np.zeros((n, n), np.uint32)
        for _ in range(2):
            s.sweep(1, do_hyper=True)
            s.coclustering_accumulate()
            st = s.get_state()
            lab = st["table_of"] if view < 0 else st["dish_of"][0][st["table_of"]]
            assert lab.max() >= 64
            want += (lab[:, None] == lab[None, :]).astype(np.uint32)
        got, ns = s.coclustering_get()
        assert ns == 2
        np.testing.assert_array_equal(got, want)
    s.close()


def test_wide_capacity_checkpoint_resumes_bit_identically(tmp_path):
    n, dims, cap = 2100, [64, 64], 256
    views, _ = make_mixture(n, dims, 9, seed=8)
    rng = np.random.default_rng(4)
    tab, dish = _wide_state(n, 2, cap, 200, rng)
    hyp = ([1.0, 1.0], [0.5, 0.5], [0.9, 0.9], 1.0, 0.6)
    a = _mk_sampler(views, cap, seed=3, engine=0, debug=False)
    a.set_state(tab, dish, *hyp)
    a.sweep(3, do_hyper=True)
    ck = tmp_path / "chain.mvg"
    a.save_checkpoint(ck)
    a.sweep(4, do_hyper=True)
    ref = a.get_state()
    a.close()
    b = _mk_sampler(views, cap, seed=3, engine=0, debug=False)
    b.load_checkpoint(ck)
    b.sweep(4, do_hyper=True)
    got = b.get_state()
    b.close()
    for k in ("table_of", "n_t", "dish_of", "n_vk", "l_vk", "alpha_v", "sigma_v", "tau_v"):
        np.testing.assert_array_equal(got[k], ref[k], err_msg=k)
    assert got["sweep"] == ref["sweep"] == 7 and got["alpha_g"] == ref["alpha_g"]


@pytest.mark.parametrize("transport", ["nccl", "p2p"])
def test_wide_capacity_two_gpu_chain_matches_one_gpu(transport):
    """A world-2 row-sharded dense chain at cap 256 keeps the states of the one-GPU chain (this file, run under torchrun,
    is the per-rank program)."""
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr", "127.0.0.1",
           "--master-port", {"nccl": "29527", "p2p": "29528"}[transport], str(Path(__file__).resolve())]
    env = dict(os.environ, MVG_TEST_P2P="1" if transport == "p2p" else "0")
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=300, env=env)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-4000:]
    assert "SHARD_OK" in r.stdout, r.stdout[-2000:]


def _shard_main():
    import torch
    import torch.distributed as dist
    for p in (ROOT, ROOT / "multiview-clustering_b200", ROOT / "tests"):
        sys.path.insert(0, str(p))
    import mvc_b200
    from conftest import make_mixture
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    dist.init_process_group("gloo")
    torch.cuda.set_device(local)
    n, dims, cap, sweeps = 128 * 100 + 19, [64, 64], 256, 20
    views, _ = make_mixture(n, dims, 40, seed=17)
    tab, dish = _wide_state(n, 2, cap, 200, np.random.default_rng(3))
    hyp = ([1.0] * 2, [0.5] * 2, [1.0] * 2, 1.0, 0.6)
    lo, hi = rank * n // world, (rank + 1) * n // world
    s = mvc_b200.Sampler(hi - lo, dims, cap=cap, seed=77, device=local, engine=0, rank=rank, world=world,
                         row_offset=lo, n_rows_global=n)
    uid = [mvc_b200.Sampler.nccl_unique_id() if rank == 0 else None]
    dist.broadcast_object_list(uid, src=0)
    s.comm_init_rank(uid[0])
    for v in range(2):
        s.upload_view(v, views[v][lo:hi])
    if os.environ.get("MVG_TEST_P2P") == "1":
        handles = [None] * world
        dist.all_gather_object(handles, s.p2p_export())
        s.p2p_attach(handles)
    s.set_state(tab[lo:hi], dish, *hyp)
    kept = []
    for _ in range(sweeps):
        s.sweep(1, do_hyper=True)
        st = s.get_state()
        kept.append((st["table_of"], st["n_t"], st["dish_of"]))
    parts = [None] * world
    dist.all_gather_object(parts, (lo, kept))
    s.close()
    if rank == 0:
        parts.sort(key=lambda p: p[0])
        one = mvc_b200.Sampler(n, dims, cap=cap, seed=77, device=local, engine=0)
        for v in range(2):
            one.upload_view(v, views[v])
        one.set_state(tab, dish, *hyp)
        agree = []
        for i in range(sweeps):
            one.sweep(1, do_hyper=True)
            ref = one.get_state()
            got = np.concatenate([p[1][i][0] for p in parts])
            agree.append(float((ref["table_of"] == got).mean()))
            np.testing.assert_array_equal(np.bincount(got, minlength=cap), parts[0][1][i][1])
        one.close()
        assert agree[0] == 1.0, agree
        assert min(agree) > 0.999, agree            # FP32 partial sums are grouped per shard: a CDF-edge draw may flip
        print(f"SHARD_OK world={world} cap={cap} agreement={agree}")
    dist.barrier()
    dist.destroy_process_group()


if __name__ == "__main__":
    _shard_main()
