"""The count-view likelihoods side by side on one GPU: the plug-in multinomial (MVG_COUNT_PLUGIN) and the collapsed
Dirichlet-multinomial (MVG_COUNT_DIRMULT), on the same data, start and seed.

Workloads (CUDA-core engine):
  * C2-shaped: 21 578 rows, three count views of vocabularies 13 008 / 5 728 / 445 and ~1.16 M nonzeros in all, cap 64,
    over-split start (32 tables, one dish each).  The real Reuters-21578 collection when data_cache/ holds it, otherwise
    synthetic documents of that shape (seed 1999): heavy-tailed lengths, 20 topics, words from a topic band or uniform,
    counts 1 + Geometric(1/2).
  * C4-shaped count views at a reduced N (--c4-rows): four views of vocab 16 384, nnz/row ~ Poisson(48), counts
    1 + Geometric(1/2), cap 256, 96 planted clusters, over-split start (192 live tables).
Per workload and model: time per sweep over a timed window (CUDA events, mvg_last_sweep_ms), the per-phase split of
mvg_profile_sweep (median), the time of the stage-A kernel alone (torch.profiler, k_counts_loglik vs k_counts_loglik_dm),
the share of nonzeros with x > 1, and tables_live.  Prints one JSON object; --out writes it too.

    python profiles/count_dirmult_probe.py --out profiles/r03_count_dirmult.json
"""
import argparse
import json
import subprocess
import sys
from pathlib import Path

import numpy as np
import torch

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT / "multiview-clustering_b200"))
import mvc_b200  # noqa: E402

SEED = 1999


def device_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader,nounits",
                        "-i", "0"], capture_output=True, text=True).stdout.strip().split(", ")
    p = torch.cuda.get_device_properties(0)
    return {"name": q[0] if q and q[0] else p.name, "power_limit_w": float(q[1]), "max_sm_clock_mhz": float(q[2]),
            "sms": p.multi_processor_count}


def synthetic_view(rng, n, vocab, nnz_target, z, k_true):
    lens = np.maximum(1, rng.lognormal(0.0, 0.9, n))
    lens = np.maximum(1, np.round(lens * nnz_target / lens.sum())).astype(np.int64)
    lens = np.minimum(lens, vocab)
    rowptr = np.concatenate([[0], np.cumsum(lens)]).astype(np.int64)
    nnz = int(rowptr[-1])
    row = np.repeat(np.arange(n), lens)
    band = (z[row] * (vocab // k_true) + rng.integers(0, max(16, vocab // 8), nnz)) % vocab
    col = np.where(rng.random(nnz) < 0.6, band, rng.integers(0, vocab, nnz))
    # distinct words per row: sort (row, col) and drop repeats
    key = row * vocab + col
    key = np.unique(key)
    row, col = key // vocab, key % vocab
    rowptr = np.concatenate([[0], np.cumsum(np.bincount(row, minlength=n))]).astype(np.int32)
    val = rng.geometric(0.5, len(col)).astype(np.float32)
    return {"rowptr": rowptr, "col": col.astype(np.int32), "val": val, "vocab": int(vocab)}


def c2_views():
    try:
        from mvc_b200 import reuters
        cached = reuters.load_cached()
    except Exception:                       # noqa: BLE001 - the cache is optional
        cached = None
    if cached is not None:
        views, _ = cached
        return views, "Reuters-21578 (data_cache)"
    rng = np.random.default_rng(SEED)
    n, k_true = 21578, 20
    z = rng.integers(0, k_true, n)
    views = [synthetic_view(rng, n, 13008, 870_000, z, k_true), synthetic_view(rng, n, 5728, 230_000, z, k_true),
             synthetic_view(rng, n, 445, 60_000, z, k_true)]
    return views, "synthetic, Reuters-shaped (the collection was not cached)"


def c4_views(n):
    rng = np.random.default_rng(SEED)
    k_true, vocab = 96, 16384
    z = rng.integers(0, k_true, n)
    views = []
    for _ in range(4):
        lens = np.maximum(1, rng.poisson(48, n)).astype(np.int64)
        row = np.repeat(np.arange(n), lens)
        nnz = len(row)
        band = (z[row] * 160 + rng.integers(0, 512, nnz)) % vocab
        col = np.where(rng.random(nnz) < 0.5, band, rng.integers(0, vocab, nnz))
        key = np.unique(row * vocab + col)
        row, col = key // vocab, key % vocab
        rowptr = np.concatenate([[0], np.cumsum(np.bincount(row, minlength=n))]).astype(np.int32)
        views.append({"rowptr": rowptr, "col": col.astype(np.int32), "val": rng.geometric(0.5, len(col)).astype(np.float32),
                      "vocab": vocab})
    coin = rng.random(n) < 0.5
    return views, (z + k_true * coin).astype(np.int32)


def make_sampler(views, cap, tab, model):
    n = len(views[0]["rowptr"]) - 1
    s = mvc_b200.Sampler(n, [0] * len(views), cap=cap, seed=SEED, engine=mvc_b200.ENGINE_SIMT)
    for v, x in enumerate(views):
        s.upload_view_csr(v, x["rowptr"], x["col"], x["val"], x["vocab"])
    s.set_count_likelihood(model)
    V = len(views)
    dish = np.full((V, cap), -1, np.int32)
    live = int(tab.max()) + 1
    dish[:, :live] = np.arange(live)
    s.set_state(tab, dish, [1.0] * V, [0.5] * V, [1.0] * V, 1.0, 0.6)
    return s


def stage_a_ms(s, sweeps):
    """Mean device time per launch of the count stage-A kernel over `sweeps` sweeps (torch.profiler, its own run)."""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        s.sweep(sweeps, do_hyper=True)
        s.sync()
    tot, cnt = 0.0, 0
    for e in prof.key_averages():
        if "k_counts_loglik" in e.key:
            tot += e.device_time_total if hasattr(e, "device_time_total") else e.cuda_time_total
            cnt += e.count
    return (tot / 1e3 / cnt) if cnt else None


def measure(views, cap, tab, model, warmup, sweeps, reps):
    s = make_sampler(views, cap, tab, model)
    s.sweep(warmup, do_hyper=True)
    s.sync()
    s.sweep(sweeps, do_hyper=True)
    s.sync()
    ms = s.last_sweep_ms() / sweeps
    runs = [s.profile_sweep(do_hyper=True) for _ in range(reps)]
    split = {k: float(np.median([r[k] for r in runs])) for k in runs[0]}
    a_ms = stage_a_ms(s, 5)
    st = s.get_state(with_rows=False)
    s.close()
    return {"ms_per_sweep": ms, "per_phase_ms": split, "stage_a_ms": a_ms, "tables_live": int((st["n_t"] > 0).sum())}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--c4-rows", type=int, default=500_000)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--sweeps", type=int, default=30)
    ap.add_argument("--profile-reps", type=int, default=5)
    ap.add_argument("--out")
    a = ap.parse_args()
    res = {"device": device_info(), "warmup_sweeps": a.warmup, "timed_sweeps": a.sweeps,
           "sources": {"ms_per_sweep": "CUDA events on the library stream around the timed mvg_sweep call / sweeps",
                       "per_phase_ms": f"mvg_profile_sweep, median of {a.profile_reps} sweeps after the window; "
                                       "draw includes the count stage A",
                       "stage_a_ms": "torch.profiler CUDA activity, mean per launch of k_counts_loglik[_dm] over 5 sweeps"},
           "workloads": {}}
    c2, c2_src = c2_views()
    n2 = len(c2[0]["rowptr"]) - 1
    rng = np.random.default_rng(SEED)
    tab2 = rng.integers(0, 32, n2).astype(np.int32)
    c4, tab4 = c4_views(a.c4_rows)
    for name, views, cap, tab, src in (("C2", c2, 64, tab2, c2_src),
                                       ("C4_counts", c4, 256, tab4, f"synthetic, N = {a.c4_rows}, 4 count views")):
        vals = np.concatenate([v["val"] for v in views])
        w = {"data": src, "rows": len(views[0]["rowptr"]) - 1, "cap": cap,
             "vocab": [v["vocab"] for v in views], "nnz": [int(len(v["val"])) for v in views],
             "share_nnz_x_gt_1": float((vals > 1).mean()),
             "n_max_tokens": [int(max(np.diff(np.concatenate([[0.0], np.cumsum(v["val"], dtype=np.float64)])[v["rowptr"]])))
                              for v in views]}
        for model in ("plugin", "dirmult"):
            w[model] = measure(views, cap, tab, model, a.warmup, a.sweeps, a.profile_reps)
        if w["plugin"]["stage_a_ms"] and w["dirmult"]["stage_a_ms"]:
            w["stage_a_ratio_dirmult_over_plugin"] = w["dirmult"]["stage_a_ms"] / w["plugin"]["stage_a_ms"]
        w["sweep_ratio_dirmult_over_plugin"] = w["dirmult"]["ms_per_sweep"] / w["plugin"]["ms_per_sweep"]
        res["workloads"][name] = w
    print(json.dumps(res))
    if a.out:
        Path(a.out).parent.mkdir(parents=True, exist_ok=True)
        Path(a.out).write_text(json.dumps(res, indent=1) + "\n")


if __name__ == "__main__":
    main()
