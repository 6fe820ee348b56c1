"""Cost of the count-view beta step (mvg_set_count_beta_prior) on one GPU, under MVG_COUNT_DIRMULT.

Workloads (CUDA-core engine; the data of profiles/count_dirmult_probe.py, same seed and over-split start):
  * C2-shaped: 21 578 rows, count views of vocabularies 13 008 / 5 728 / 445, cap 64;
  * C4-shaped count views at a reduced N (--c4-rows): four views of vocab 16 384, cap 256.
Per workload: time per sweep with the step off (no prior) and on (prior Gamma(1, 1), step 0.3) over a timed window
(CUDA events, mvg_last_sweep_ms); then, in a run of its own under torch.profiler, sweeps one at a time with the step on:
the device time of k_count_beta_step and of the refresh (the second k_counts_tables launch of the sweep and
k_counts_newdish), split by sweeps in which some view accepted and sweeps in which none did, and the acceptance rate.
Prints one JSON object; --out writes it too.

    python profiles/count_beta_probe.py --out profiles/r03_count_beta.json
"""
import argparse
import json
import sys
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT / "multiview-clustering_b200"))
sys.path.insert(0, str(ROOT / "profiles"))
import mvc_b200  # noqa: E402
from count_dirmult_probe import SEED, c2_views, c4_views, device_info  # noqa: E402

PRIOR = (1.0, 1.0, 0.3)


def make_sampler(views, cap, tab, prior):
    n = len(views[0]["rowptr"]) - 1
    s = mvc_b200.Sampler(n, [0] * len(views), cap=cap, seed=SEED, engine=mvc_b200.ENGINE_SIMT)
    for v, x in enumerate(views):
        s.upload_view_csr(v, x["rowptr"], x["col"], x["val"], x["vocab"])
    s.set_count_likelihood("dirmult")
    if prior:
        s.set_count_beta_prior(*PRIOR)
    V = len(views)
    dish = np.full((V, cap), -1, np.int32)
    live = int(tab.max()) + 1
    dish[:, :live] = np.arange(live)
    s.set_state(tab, dish, [1.0] * V, [0.5] * V, [1.0] * V, 1.0, 0.6)
    return s


def sweep_ms(views, cap, tab, prior, warmup, sweeps):
    s = make_sampler(views, cap, tab, prior)
    s.sweep(warmup, do_hyper=True)
    s.sync()
    s.sweep(sweeps, do_hyper=True)
    s.sync()
    ms = s.last_sweep_ms() / sweeps
    beta = s.get_count_beta().tolist()
    s.close()
    return ms, beta


def step_kernels(views, cap, tab, warmup, sweeps):
    """Device time per sweep of the step and of its refresh, by torch.profiler, accepted and rejected sweeps apart."""
    from torch.autograd import DeviceType
    from torch.profiler import ProfilerActivity, profile
    s = make_sampler(views, cap, tab, True)
    s.sweep(warmup, do_hyper=True)
    s.sync()
    accepted = []
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(sweeps):
            s.sweep(1, do_hyper=True)
            accepted.append(s.get_count_beta_step()[1])
    s.close()
    ev = sorted((e for e in prof.events() if e.device_type == DeviceType.CUDA),
                key=lambda e: e.time_range.start)

    def per_sweep(name, per, pick):
        us = [e.time_range.elapsed_us() for e in ev if name in e.name]
        assert len(us) == per * sweeps, (name, len(us), per * sweeps)
        return np.array(us[pick::per], np.float64)

    step = per_sweep("k_count_beta_step", 1, 0)
    refresh = per_sweep("k_counts_tables", 2, 1) + per_sweep("k_counts_newdish", 1, 0)
    acc = np.array([bool(a.any()) for a in accepted])
    cnt = np.array(accepted)                     # every view of these workloads is a count view

    def stats(x):
        return {"sweeps": int(len(x)), "median_ms": float(np.median(x)) / 1e3 if len(x) else None,
                "mean_ms": float(x.mean()) / 1e3 if len(x) else None}
    return {"step_kernel": stats(step),
            "step_plus_refresh_some_view_accepted": stats((step + refresh)[acc]),
            "step_plus_refresh_none_accepted": stats((step + refresh)[~acc]),
            "acceptance_rate_per_view_step": float(cnt.mean())}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--c4-rows", type=int, default=50_000)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--sweeps", type=int, default=30)
    ap.add_argument("--profiled-sweeps", type=int, default=40)
    ap.add_argument("--out")
    a = ap.parse_args()
    res = {"device": device_info(), "prior_shape_rate_step": PRIOR, "warmup_sweeps": a.warmup, "timed_sweeps": a.sweeps,
           "sources": {"ms_per_sweep": "CUDA events on the library stream around the timed mvg_sweep call / sweeps",
                       "kernels": f"torch.profiler CUDA activity over {a.profiled_sweeps} sweeps issued one at a time "
                                  "(a separate run); refresh = second k_counts_tables launch + k_counts_newdish"},
           "workloads": {}}
    c2, c2_src = c2_views()
    n2 = len(c2[0]["rowptr"]) - 1
    tab2 = np.random.default_rng(SEED).integers(0, 32, n2).astype(np.int32)
    c4, tab4 = c4_views(a.c4_rows)
    for name, views, cap, tab, src in (("C2", c2, 64, tab2, c2_src),
                                       ("C4_counts", c4, 256, tab4, f"synthetic, N = {a.c4_rows}, 4 count views")):
        w = {"data": src, "rows": len(views[0]["rowptr"]) - 1, "cap": cap, "vocab": [v["vocab"] for v in views]}
        w["ms_per_sweep_step_off"], _ = sweep_ms(views, cap, tab, False, a.warmup, a.sweeps)
        w["ms_per_sweep_step_on"], w["beta_after_window"] = sweep_ms(views, cap, tab, True, a.warmup, a.sweeps)
        w["kernels"] = step_kernels(views, cap, tab, a.warmup, a.profiled_sweeps)
        res["workloads"][name] = w
        print(name, json.dumps(w), flush=True)
    print(json.dumps(res))
    if a.out:
        Path(a.out).parent.mkdir(parents=True, exist_ok=True)
        Path(a.out).write_text(json.dumps(res, indent=1) + "\n")


if __name__ == "__main__":
    main()
