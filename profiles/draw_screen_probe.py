"""Draw screening A/B on the C3 shape (DESIGN.md §4.1.1): N = 1M, three dense views of 64 dims, cap 64, one GPU,
incremental statistics, hyper step on — bench.py's data (its generator, seed 1999) and start.

For each data set — separated clusters (bench.py's default), overlapping clusters (planted means N(0, 0.35^2 I)) and 60
planted clusters (four free table slots: births, the new-table marginal) — two handles, screening on and off, run
--warmup sweeps, then --rounds timed windows of --sweeps sweeps each, alternating on / off (CUDA events of the
library's stream).  Recorded per window: ms per sweep and the draw kernel's in-kernel clock; then, over --sample single
sweeps of the screened chain, the fraction of rows screened, tiles evaluated and the bytes the draw actually moves:
evaluated rows x (768 B of features + 8 B) + screened rows x 28 B (table, margin, three norms, choice, mask bits).
Both chains are compared at the end (table_of, n_t): they must be identical.  Prints one JSON object; --out writes it.

    python profiles/draw_screen_probe.py --out profiles/r04_draw_screen.json
"""
import argparse
import json
import subprocess
import sys
from pathlib import Path

import numpy as np
import torch

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "multiview-clustering_b200"))
import bench  # noqa: E402  (data generator and start state of the benchmark)
import mvc_b200  # noqa: E402

N = 1_000_000
FULL_ROW_BYTES = 3 * 64 * 4 + 8
SCREENED_ROW_BYTES = 4 + 4 + 12 + 4 + 4


def device_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader,nounits",
                        "-i", "0"], capture_output=True, text=True).stdout.strip().split(", ")
    p = torch.cuda.get_device_properties(0)
    return {"name": q[0] if q and q[0] else p.name, "power_limit_w": float(q[1]), "max_sm_clock_mhz": float(q[2]),
            "sms": p.multi_processor_count}


def run_case(name, spread, k_true, a):
    mus = bench.planted_means(np.random.default_rng(bench.SEED), spread)
    views, z = bench.make_rows_numpy(0, N, mus, k_true=k_true)
    tab, dish, hyp = bench.initial_state(z, k_true)
    dev = [torch.from_numpy(v).cuda() for v in views]
    hs = {}
    for on in (True, False):
        s = mvc_b200.Sampler(N, bench.DIMS, cap=bench.CAP, seed=bench.SEED, engine=mvc_b200.ENGINE_TCGEN05)
        for v in range(3):
            s.attach_view_device(v, dev[v])
        s.set_stats_mode(True, 64)
        s.set_draw_screen(on)
        s.set_state(tab, dish, hyp["alpha_v"], hyp["sigma_v"], hyp["tau_v"], hyp["alpha_g"], hyp["sigma_g"])
        s.sweep(a.warmup, True)
        s.sync()
        hs[on] = s
    win = {True: [], False: []}
    for _ in range(a.rounds):
        for on in (True, False):
            s = hs[on]
            s.kernel_clock(0, reset=True)
            s.sweep(a.sweeps, True)
            s.sync()
            d_ms, d_n = s.kernel_clock(0)
            win[on].append({"ms_per_sweep": s.last_sweep_ms() / a.sweeps, "draw_kernel_ms": d_ms / d_n if d_n else None})
    frac, tiles = [], []
    for _ in range(a.sample):
        for on in (True, False):
            hs[on].sweep(1, True)
        st = hs[True].draw_screen_stats()
        frac.append(st["rows_screened"] / N)
        tiles.append(st["tiles_evaluated"])
    a_on, a_off = hs[True].get_state(), hs[False].get_state()
    same = bool(np.array_equal(a_on["table_of"], a_off["table_of"]) and np.array_equal(a_on["n_t"], a_off["n_t"]))
    for s in hs.values():
        s.close()
    f = float(np.mean(frac))
    med = {on: float(np.median([w["ms_per_sweep"] for w in win[on]])) for on in (True, False)}
    return {"data": name, "planted_clusters": k_true, "spread": spread,
            "ms_per_sweep_median": {"screen_on": med[True], "screen_off": med[False]}, "speedup": med[False] / med[True],
            "windows": {"screen_on": win[True], "screen_off": win[False]},
            "rows_screened_fraction_mean": f, "rows_screened_fraction_per_sweep": frac, "tiles_evaluated_per_sweep": tiles,
            "draw_bytes_per_sweep": {"screen_on": N * (1 - f) * FULL_ROW_BYTES + N * f * SCREENED_ROW_BYTES,
                                     "screen_off": N * FULL_ROW_BYTES},
            "chains_identical": same}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--warmup", type=int, default=50)
    ap.add_argument("--sweeps", type=int, default=200)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--sample", type=int, default=64, help="single sweeps over which the screened fraction is averaged")
    ap.add_argument("--out")
    a = ap.parse_args()
    rec = {"device": device_info(), "shape": "C3: N=1M, 3 dense views x 64 dims, cap 64, one GPU, incremental statistics, hyper step",
           "timing": "CUDA events of the library's stream over each window (graph replays); windows alternate on / off",
           "cases": [run_case("separated", 2.0, 64, a), run_case("overlapping", 0.35, 64, a), run_case("free_slots", 2.0, 60, a)]}
    print(json.dumps(rec, indent=1))
    if a.out:
        Path(a.out).parent.mkdir(parents=True, exist_ok=True)
        Path(a.out).write_text(json.dumps(rec, indent=1) + "\n")


if __name__ == "__main__":
    main()
