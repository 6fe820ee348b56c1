#!/usr/bin/env python
"""bench.py — Gibbs allocation sweeps of the multiview Pitman-Yor sampler on B200.

    python bench.py --gpus N --steps K --warmup W           (N > 1: launched under torchrun)
    python bench.py --impl reference --gpus N --steps K --warmup W

Workload (BASELINE.json configs[2], SURVEY.md §8d "C3"): synthetic 3-view Gaussian mixture,
N = 1M customers, D = 64 per view, cap K = 64 tables/dishes, FP32, seed 1999.  A "step" is ONE sweep
of the hot path: likelihood + draw for every customer, birth/death bookkeeping, sufficient-statistics
rebuild and the hyperparameter step.  metric = obs x view x K updates per second (whole job).
With N GPUs the customers are row-sharded and the per-table statistics are exchanged by one NCCL
all-gather per sweep.  Default scaling is "weak": every GPU holds one C3-sized shard (1M customers), so
the chain has N x 1M customers and `value` counts the updates of all ranks; `--scaling strong` keeps the
chain at 1M customers in total and splits it over the ranks instead.

The timed `value` has the data resident in HBM (inputs 768 MB >> 126 MB L2, so every sweep streams
from HBM; no extra L2 flush).  `e2e` is the same metric through the reference-facing call with HOST
buffers: upload of the views from pinned memory, state set, K sweeps, read-back of table_of.  K is --steps, as in
the timed `value`; at small K the upload and the state set dominate it (a caller's chain runs thousands of sweeps).

`--dump-outputs DIR` writes the chain state the timed sweeps leave behind (what mvg_get_state returns after the last
timed sweep) as DIR/<name>.npy, so that two builds can be compared output for output on identical seeded inputs.
Only the C3 workload (the default) dumps; c1, c2, c5 and --impl reference refuse the flag.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent
sys.dont_write_bytecode = True          # the tree may be read-only: nothing is written into it
for p in (ROOT, ROOT / "multiview-clustering_b200"):
    if str(p) not in sys.path:
        sys.path.insert(0, str(p))

N_ROWS = 1_000_000
DIMS = [64, 64, 64]
CAP = 64
SEED = 1999
NCU_TRAFFIC_BYTES = 792.1e6     # measured DRAM traffic of one k_draw_tc launch at N=1M (profiles/r02_ncu_draw.md; algorithmic: 776 MB + 12 MB of stored squared norms)
METRIC = "obs_x_view_x_K_updates_per_s"
UNIT = "updates/s"


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=1000)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--rows", type=int, default=N_ROWS, help="customers per GPU (weak) / in total (strong); default: the named config")
    ap.add_argument("--scaling", default="strong", choices=["weak", "strong"],
                    help="strong (default; north_star: N = 1M row-sharded over 1/2/4/8 GPUs): --rows customers split over the "
                         "GPUs, and the weak figure is measured beside it (`weak` sub-record); weak: --rows customers per GPU")
    ap.add_argument("--engine", type=int, default=0, help="0 auto, 1 CUDA-core, 2 tcgen05")
    ap.add_argument("--k-true", type=int, default=CAP, help="planted clusters (default 64 = every table slot in use; "
                    "fewer leaves free slots, so the new-table marginal is evaluated as well)")
    ap.add_argument("--workload", default="c3", choices=["c3", "c1", "c2", "c5"],
                    help="c3: the headline configuration (default).  c1: BASELINE configs[0], the reference's own case "
                         "(New_Simulation.R: N=500, two scalar views), reported in sweeps/s with --chains independent "
                         "chains per GPU; with --impl reference the UNMODIFIED reference sampler (oracle/_ref) is timed.  "
                         "c2: BASELINE configs[1]/[4], three sparse count views with the shapes of Reuters-21578 (synthetic "
                         "topics; the .sgm files do not travel to the GPU box), --chains chains per GPU.  "
                         "c5: BASELINE configs[4], --chains independent chains of the Reuters config per GPU; their pooled posterior "
                         "co-clustering matrix (a fixed subsample of the documents) is compared with CPU chains of the FP64 restatement")
    ap.add_argument("--synthetic-reuters", action="store_true", help="c2: synthetic topics even when the ingested collection is cached")
    ap.add_argument("--chains", type=int, default=8, help="c1: independent chains per GPU, one stream each")
    ap.add_argument("--exchange", default="auto", choices=["auto", "p2p", "nccl"],
                    help="N > 1: transport of the once-per-sweep packets: p2p = stores into the peers' memory over NVLink "
                         "(constant ~26 us per sweep; falls back to NCCL if the buffers cannot be mapped), nccl = "
                         "ncclAllGather (15 us at 2 GPUs, 39 us at 8); auto = p2p")
    ap.add_argument("--no-hyper", action="store_true")
    ap.add_argument("--role-profile", action="store_true", help="print the tcgen05 kernel's per-role wait cycles (debug)")
    ap.add_argument("--stats", default="incremental", choices=["incremental", "rebuild"],
                    help="how the sufficient statistics follow the assignments (include/mvg.h: mvg_set_stats_mode): incremental = only "
                         "the rows that moved are re-read (running FP64 sums, a full rebuild every 64 sweeps) — the reference's own "
                         "remove/add bookkeeping, batched; rebuild = every sweep re-reads all rows.  The other mode is measured beside "
                         "the headline (`stats_rebuild` sub-record)")
    ap.add_argument("--no-extra", action="store_true", help="skip the sub-records (rebuild mode, overlapping clusters)")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-weak", action="store_true", help="N > 1: skip the weak-scaling sub-record")
    ap.add_argument("--no-free-slots", action="store_true", help="N = 1: skip the run with free table slots")
    ap.add_argument("--no-checks", action="store_true", help="skip the sharded-vs-one-GPU replay and the CPU-mirror spot check")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--cpu-rows", type=int, default=0, help="rows of the CPU sample (0: sized for ~15 s)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="C3 only (the other workloads and --impl reference refuse it): "
                    "write the state after the last timed sweep as DIR/<name>.npy (table_of of every row, per-table counts "
                    "and sums, hyperparameters; float32/float64)")
    args = ap.parse_args()
    if args.dump_outputs and (args.workload != "c3" or args.impl != "b200"):
        ap.error("--dump-outputs applies to the C3 workload of --impl b200")
    return args


# ---------------------------------------------------------------------------------------------
# synthetic workload (SURVEY.md §8d C3): z ~ U{0..63}, mu_vk ~ N(0, 2^2 I), x = mu + N(0, I)
# ---------------------------------------------------------------------------------------------
def planted_means(rng, spread=2.0):
    return [rng.normal(0.0, spread, (CAP, d)).astype(np.float32) for d in DIMS]


def make_rows_numpy(lo, hi, mus, seed=SEED, k_true=CAP):
    """Rows [lo, hi) of the global data set, reproducible per 65536-row block (shard-invariant)."""
    B = 65536
    views = [np.empty((hi - lo, d), np.float32) for d in DIMS]
    z = np.empty(hi - lo, np.int32)
    b = lo // B
    while b * B < hi:
        rng = np.random.default_rng([seed, b])
        zb = rng.integers(0, CAP, B).astype(np.int32)
        if k_true < CAP:
            zb = zb % k_true
        nb = [rng.standard_normal((B, d), dtype=np.float32) for d in DIMS]
        s, e = max(lo, b * B), min(hi, (b + 1) * B)
        z[s - lo:e - lo] = zb[s - b * B:e - b * B]
        for v in range(len(DIMS)):
            views[v][s - lo:e - lo] = mus[v][zb[s - b * B:e - b * B]] + nb[v][s - b * B:e - b * B]
        b += 1
    return views, z


def initial_state(z, k_true=CAP):
    dish = np.tile(np.arange(CAP, dtype=np.int32), (len(DIMS), 1))      # dish_of[v][t] = t
    dish[:, k_true:] = -1                                               # unused table slots are free
    hyp = dict(alpha_v=[1.0] * len(DIMS), sigma_v=[0.5] * len(DIMS), tau_v=[1.0] * len(DIMS), alpha_g=1.0, sigma_g=0.6)
    return z.astype(np.int32), dish, hyp


# ---------------------------------------------------------------------------------------------
class ClockSampler(threading.Thread):
    """SM clock and throttle reasons sampled DURING the timed region: NVML (a query takes ~0.1 ms, so that even a
    20-sweep region of a few milliseconds gets samples), nvidia-smi as the fallback."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
    BITS = {"hw_slowdown": 0x8, "hw_thermal_slowdown": 0x40, "sw_thermal_slowdown": 0x20, "sw_power_cap": 0x4}

    def __init__(self, gpu_index):
        super().__init__(daemon=True)
        self.gpu, self.stop_flag = gpu_index, False
        self.sm, self.mx, self.reasons, self.power, self.mem = [], [], set(), [], []
        self.nvml = None
        try:
            import pynvml
            pynvml.nvmlInit()
            # NVML enumerates physical devices: honour CUDA_VISIBLE_DEVICES when it lists plain indices
            vis = os.environ.get("CUDA_VISIBLE_DEVICES", "")
            idx = gpu_index
            if vis and all(t.strip().isdigit() for t in vis.split(",")):
                idx = int(vis.split(",")[gpu_index])
            self.handle = pynvml.nvmlDeviceGetHandleByIndex(idx)
            self.mx.append(float(pynvml.nvmlDeviceGetMaxClockInfo(self.handle, pynvml.NVML_CLOCK_SM)))
            self.nvml = pynvml
            self.sample()                                       # the first query of a process can take tens of ms: not inside the region
            self.sm, self.power, self.reasons, self.mem = [], [], set(), []
        except Exception:                                       # noqa: BLE001
            self.nvml = None

    def sample(self):
        if self.nvml is not None:
            n = self.nvml
            self.sm.append(float(n.nvmlDeviceGetClockInfo(self.handle, n.NVML_CLOCK_SM)))
            try:
                self.mem.append(float(n.nvmlDeviceGetClockInfo(self.handle, n.NVML_CLOCK_MEM)))
            except Exception:                                   # noqa: BLE001
                pass
            try:
                r = int(n.nvmlDeviceGetCurrentClocksEventReasons(self.handle))
            except Exception:                                   # noqa: BLE001
                r = int(n.nvmlDeviceGetCurrentClocksThrottleReasons(self.handle))
            for name, bit in self.BITS.items():
                if r & bit:
                    self.reasons.add(name)
            try:
                self.power.append(n.nvmlDeviceGetPowerUsage(self.handle) / 1e3)
            except Exception:                                   # noqa: BLE001
                pass
            return
        out = subprocess.run(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-i", str(self.gpu)],
                             capture_output=True, text=True, timeout=5).stdout.strip()
        r = [x.strip() for x in out.split(",")]
        if len(r) > 8 and r[1].replace(".", "").isdigit():
            self.sm.append(float(r[1])); self.mx.append(float(r[2]))
            for name, val in zip(["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"], r[5:9]):
                if val.lower().startswith("active"):
                    self.reasons.add(name)

    def run(self):
        while not self.stop_flag:
            try:
                self.sample()
            except Exception:                                   # noqa: BLE001
                pass
            time.sleep(0.0005 if self.nvml is not None else 0.02)

    def summary(self):
        return {"sm_mhz": float(np.median(self.sm)) if self.sm else None, "sm_max_mhz": max(self.mx) if self.mx else None,
                "reasons": sorted(self.reasons), "samples": len(self.sm),
                "power_w_median": float(np.median(self.power)) if self.power else None,
                "sm_mhz_min": float(np.min(self.sm)) if self.sm else None,
                "mem_mhz": float(np.median(self.mem)) if self.mem else None,
                "source": "nvml" if self.nvml is not None else "nvidia-smi"}


def measured_peak():
    f = ROOT / "MEASURED_PEAKS.json"
    if f.exists():
        return float(json.loads(f.read_text())["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def cpu_port_throughput(rows, threads):
    """The FP64 CPU restatement of the sweep (oracle/mv_oracle.c) on a bounded sample of the workload."""
    sys.path.insert(0, str(ROOT / "oracle"))
    import pyoracle as po
    mus = planted_means(np.random.default_rng(SEED))
    views, z = make_rows_numpy(0, rows, mus)
    tab, dish, hyp = initial_state(z)
    o = po.OracleState(views, CAP, seed=SEED)
    o.alpha_v[:] = hyp["alpha_v"]; o.sigma_v[:] = hyp["sigma_v"]; o.tau_v[:] = hyp["tau_v"]
    o.set_assignment(tab, dish)
    t0 = time.perf_counter()
    o.sweep_n(1, threads=threads, do_hyper=True)
    dt = time.perf_counter() - t0
    return rows * len(DIMS) * CAP / dt, dt


def c1_views(n=500, seed=SEED):
    """BASELINE configs[0] / SURVEY.md §8d C1: view1 = N(3,1.3^2) U N(-3,1.3^2); view2 = three groups."""
    rng = np.random.default_rng(seed)
    h, q = n // 2, n // 4
    v1 = np.concatenate([rng.normal(3, 1.3, h), rng.normal(-3, 1.3, n - h)])
    v2 = np.concatenate([rng.normal(0, 1.3, q), rng.normal(-5, 1.3, h), rng.normal(5, 1.3, n - q - h)])
    return [v1, v2]


def c2_start(n, cap, chain=0):
    """Start of a count-view chain: cap/2 random tables, each with its own dish in every view.  (From the reference's
    T=4, K=2 start a count-view chain cannot split: a new dish starts at the uniform prior predictive W^-|x|, which
    never beats an existing dish in a 13k-word vocabulary; starting over-split lets the sampler merge instead.)"""
    rng = np.random.default_rng([SEED, chain])
    tab = rng.integers(0, cap // 2, n).astype(np.int32)
    dish = np.full((3, cap), -1, np.int32)
    dish[:, :cap // 2] = np.arange(cap // 2)
    return tab, dish


def run_c2(args, out):
    """Reuters-shaped sparse count views (BASELINE configs[1]; configs[4] with --chains 8) in sweeps/s."""
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    from mvc_b200 import reuters
    cached = reuters.load_cached()           # the real collection, ingested from the .sgm files (data_cache/, travels with the tree)
    if cached is not None and not args.synthetic_reuters:
        views, z = cached[0], None
        source = "Reuters-21578 (real: body / title / category-tag count views ingested from the .sgm files)"
    else:
        views, z = reuters.synthetic_like_reuters(seed=SEED)
        source = "synthetic topics with the shapes of Reuters-21578"
    n, steps, cap = len(views[0]["rowptr"]) - 1, args.steps, 64
    nnz = [int(len(v["col"])) for v in views]
    workload = ("C2: three CSR count views, %s (N=%d; vocab %s; nnz %s), cap %d"
                % (source, n, "/".join(str(v["vocab"]) for v in views), "/".join(map(str, nnz)), cap))
    if args.impl == "reference":
        if rank != 0:
            return
        sys.path.insert(0, str(ROOT / "oracle"))
        import pyoracle as po
        threads = os.cpu_count() or 1
        o = po.OracleState(views, cap, seed=SEED)
        tab0, dish0 = c2_start(n, cap)
        o.set_assignment(tab0, dish0)
        k = max(1, min(steps, 3))
        t0 = time.perf_counter()
        o.sweep_n(k, threads=threads, do_hyper=True)
        dt = time.perf_counter() - t0
        line = {"impl": "reference", "metric": "gibbs_sweeps_per_s", "value": k / dt, "unit": "sweeps/s", "n_gpus": args.gpus,
                "steps": k, "warmup": 0, "ms_per_step": 1e3 * dt / k, "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": "f64", "data": "synthetic", "config": {"workload": workload + ", one chain"},
                "cpu_baseline": {"value": k / dt, "unit": "sweeps/s", "cores": threads, "kind": "port",
                                 "sample": "%d FP64 sweeps of oracle/mv_oracle.c (the reference has no count likelihood)" % k},
                "e2e": {"value": k / dt, "unit": "sweeps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
        print(json.dumps(line), file=out)
        return
    import torch
    import mvc_b200
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the sweep has no CPU path")
    torch.cuda.set_device(local_rank)
    chains = []
    for ch in range(args.chains):
        s = mvc_b200.Sampler(n, [0, 0, 0], cap=cap, seed=SEED, chain=rank * args.chains + ch, device=local_rank, engine=1)
        for v, x in enumerate(views):
            s.upload_view_csr(v, x["rowptr"], x["col"], x["val"], x["vocab"])
        tab0, dish0 = c2_start(n, cap, chain=rank * args.chains + ch)
        s.set_state(tab0, dish0, [1.0] * 3, [0.5] * 3, [1.0] * 3, 1.0, 0.6)
        chains.append(s)
    block = 5
    def run(k):
        done = 0
        while done < k:
            b = min(block, k - done)
            for s in chains:
                s.sweep(b, True)
            done += b
        for s in chains:
            s.sync()
    run(args.warmup)
    l0 = sum(s.launch_count() for s in chains)
    t0 = time.perf_counter()
    run(steps)
    dt = time.perf_counter() - t0
    launches = sum(s.launch_count() for s in chains) - l0
    prof = chains[0].profile_sweep(True)
    ari = [chains[0].adjusted_rand_index(v, z)[0] for v in range(3)] if z is not None else None
    live = [int((s.get_state(with_rows=False)["n_t"] > 0).sum()) for s in chains]
    for s in chains:
        s.close()
    if rank == 0:
        # The count likelihood is a gather from the L2-resident, feature-major log2-theta tables (the data set itself fits
        # L2): cap floats per nonzero, plus the CSR stream and the [N][cap] result per view.  No HBM roofline applies;
        # the figure to read is the achieved L2 rate of the two kernels event-timed as "draw".
        l2_bytes = sum(nnz) * (cap * 4 + 8) + len(views) * n * (cap * 4 * 2 + 8)
        count_lik = {"bound": "l2 gather", "algorithmic_l2_bytes_per_sweep": l2_bytes, "kernel_ms": prof["draw"],
                     "achieved_gbs": l2_bytes / (prof["draw"] * 1e-3) / 1e9 if prof["draw"] > 0 else None,
                     "nonzeros": sum(nnz), "bytes_per_nonzero": cap * 4 + 8}
        line = {"metric": "gibbs_sweeps_per_s", "value": world * args.chains * steps / dt, "unit": "sweeps/s", "n_gpus": world,
                "steps": steps, "warmup": args.warmup, "ms_per_step": 1e3 * dt / steps, "higher_is_better": True,
                "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic" if z is not None else "Reuters-21578",
                "count_likelihood": count_lik,
                "config": {"workload": workload + ", %d independent chains per GPU, CUDA-core engine, hyper step on" % args.chains,
                           "timing": "wall clock around the launches of all chains and their final synchronisation"},
                "kernel_ms_one_chain": prof, "gpu_launches": int(launches), "tables_live": live,
                "ari_vs_planted_topics_chain0": ari}
        print(json.dumps(line), file=out)


def run_c5(args, out):
    """BASELINE configs[4]: independent chains of the Reuters configuration, --chains per GPU (64 = 8 per GPU on 8 GPUs),
    and the agreement of their pooled posterior co-clustering matrix with CPU chains of the FP64 restatement
    (oracle/mv_oracle.c; the reference has no count likelihood, so that restatement is the CPU reference here)."""
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    from mvc_b200 import reuters
    cached = reuters.load_cached()
    if cached is not None and not args.synthetic_reuters:
        views, source = cached[0], "Reuters-21578 (real, ingested from the .sgm files)"
    else:
        views, source = reuters.synthetic_like_reuters(seed=SEED)[0], "synthetic topics with the shapes of Reuters-21578"
    n, cap, V = len(views[0]["rowptr"]) - 1, 64, 3
    M, burn, thin = args.steps, args.steps // 2, max(1, args.steps // 20)      # the second half of the chain, ten kept states
    sub = np.sort(np.random.default_rng(SEED).choice(n, 1500, replace=False))   # documents whose pairs are compared

    def cocl_of(labels_list):
        acc = [np.zeros((len(sub), len(sub))) for _ in range(V)]
        for lab in labels_list:                                                  # lab: [V][n]
            for v in range(V):
                l = lab[v][sub]
                acc[v] += l[:, None] == l[None, :]
        return acc

    if args.impl == "reference":
        if rank != 0:
            return
        sys.path.insert(0, str(ROOT / "oracle"))
        import pyoracle as po
        threads = os.cpu_count() or 1
        t0 = time.perf_counter()
        o = po.OracleState(views, cap, seed=SEED, chain=1000)
        tab0, dish0 = c2_start(n, cap, chain=1000)
        o.set_assignment(tab0, dish0)
        k = max(1, min(M, 20))
        o.sweep_n(k, threads=threads, do_hyper=True)
        dt = time.perf_counter() - t0
        line = {"impl": "reference", "metric": "gibbs_sweeps_per_s", "value": k / dt, "unit": "sweeps/s", "n_gpus": args.gpus,
                "steps": k, "warmup": 0, "ms_per_step": 1e3 * dt / k, "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": "f64", "data": source, "config": {"workload": "C5: one CPU chain of the Reuters configuration"},
                "cpu_baseline": {"value": k / dt, "unit": "sweeps/s", "cores": threads, "kind": "port", "sample": "%d FP64 sweeps" % k},
                "e2e": {"value": k / dt, "unit": "sweeps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
        print(json.dumps(line), file=out)
        return
    import torch
    import mvc_b200
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the sweep has no CPU path")
    torch.cuda.set_device(local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("gloo")
    chains = []
    for ch in range(args.chains):
        cid = rank * args.chains + ch
        s = mvc_b200.Sampler(n, [0, 0, 0], cap=cap, seed=SEED, chain=cid, device=local_rank, engine=1)
        for v, x in enumerate(views):
            s.upload_view_csr(v, x["rowptr"], x["col"], x["val"], x["vocab"])
        tab0, dish0 = c2_start(n, cap, chain=cid)
        s.set_state(tab0, dish0, [1.0] * V, [0.5] * V, [1.0] * V, 1.0, 0.6)
        chains.append(s)
    kept = []
    t0 = time.perf_counter()
    done = 0
    while done < M:
        b = min(thin, M - done)
        for s in chains:
            s.sweep(b, True)
        done += b
        if done > burn:
            for s in chains:
                kept.append(s.cluster_labels())                                 # D2H of V x n labels per chain and kept state
    for s in chains:
        s.sync()
    dt = time.perf_counter() - t0
    launches = sum(s.launch_count() for s in chains)
    live = [int((s.get_state(with_rows=False)["n_t"] > 0).sum()) for s in chains]
    for s in chains:
        s.close()
    mine = cocl_of(kept)
    n_kept = len(kept)
    if dist is not None:
        parts = [None] * world
        dist.all_gather_object(parts, (mine, n_kept, dt, live))
        mine = [sum(p[0][v] for p in parts) for v in range(V)]
        n_kept = sum(p[1] for p in parts)
        dt = max(p[2] for p in parts)
        live = sum((p[3] for p in parts), [])
    if rank == 0:
        P_gpu = [m / n_kept for m in mine]
        # CPU chains of the FP64 restatement: the same schedule, two chains, all host threads
        sys.path.insert(0, str(ROOT / "oracle"))
        import pyoracle as po
        threads = os.cpu_count() or 1
        cpu_kept, t1 = [], time.perf_counter()
        n_cpu = 0 if args.no_cpu_baseline else 2
        for ch in range(n_cpu):
            o = po.OracleState(views, cap, seed=SEED, chain=1000 + ch)
            tab0, dish0 = c2_start(n, cap, chain=1000 + ch)
            o.set_assignment(tab0, dish0)
            done = 0
            while done < M:
                b = min(thin, M - done)
                o.sweep_n(b, threads=threads, do_hyper=True)
                done += b
                if done > burn:
                    cpu_kept.append(o.labels().T)
        cpu_dt = time.perf_counter() - t1
        agree = None
        if cpu_kept:
            P_cpu = [m / len(cpu_kept) for m in cocl_of(cpu_kept)]
            agree = {"mean_abs_dP_per_view": [float(np.abs(P_gpu[v] - P_cpu[v]).mean()) for v in range(V)],
                     "mean_P_gpu": [float(P_gpu[v].mean()) for v in range(V)], "mean_P_cpu": [float(P_cpu[v].mean()) for v in range(V)],
                     "documents_compared": int(len(sub)), "gpu_states": int(n_kept), "cpu_states": int(len(cpu_kept)),
                     "cpu_chains": n_cpu, "cpu_sweeps_per_s": n_cpu * M / cpu_dt, "cpu_threads": threads}
        total_chains = world * args.chains
        line = {"metric": "gibbs_sweeps_per_s", "value": total_chains * M / dt, "unit": "sweeps/s", "n_gpus": world,
                "steps": M, "warmup": 0, "ms_per_step": 1e3 * dt / M, "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": "f32", "data": source,
                "config": {"workload": "C5: %d independent chains of the Reuters configuration (%d per GPU), N=%d, cap %d; kept states "
                                       "every %d sweeps of the second half; wall clock incl. the D2H of the labels" % (total_chains, args.chains, n, cap, thin)},
                "gpu_launches": int(launches), "tables_live": live, "coclustering_vs_cpu": agree}
        print(json.dumps(line), file=out)
    if dist is not None:
        dist.destroy_process_group()


def run_c1(args, out):
    """Config 1 in sweeps/s.  b200 arm: --chains independent chains on one GPU (one handle and stream each,
    launches interleaved).  reference arm: the unmodified reference sampler compiled into oracle/_ref, 1 core."""
    rank = int(os.environ.get("RANK", "0"))
    views = c1_views()
    n, steps = len(views[0]), args.steps
    if args.impl == "reference":
        if rank != 0:
            return
        sys.path.insert(0, str(ROOT / "oracle"))
        import pyoracle as po
        y = np.stack(views)
        kind = "reference" if po.have_ref() else "port"
        t0 = time.perf_counter()
        if kind == "reference":
            po.ref_run_gibbs(y, steps, steps, 1, seed=SEED)           # M sweeps, nothing saved
        else:
            o = po.OracleState([v.astype(np.float32).reshape(-1, 1) for v in views], 32, seed=SEED)
            o.init_reference()
            o.sweep_n(steps, threads=1, do_hyper=True)
        dt = time.perf_counter() - t0
        line = {"impl": "reference", "metric": "gibbs_sweeps_per_s", "value": steps / dt, "unit": "sweeps/s", "n_gpus": args.gpus,
                "steps": steps, "warmup": 0, "ms_per_step": 1e3 * dt / steps, "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": "f64", "data": "synthetic",
                "config": {"workload": "C1: New_Simulation.R two scalar views, N=%d, one chain" % n},
                "cpu_baseline": {"value": steps / dt, "unit": "sweeps/s", "cores": 1, "kind": kind,
                                 "sample": "%d sweeps of one chain from the reference initialisation" % steps},
                "e2e": {"value": steps / dt, "unit": "sweeps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
        print(json.dumps(line), file=out)
        return
    import torch
    import mvc_b200
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the sweep has no CPU path")
    torch.cuda.set_device(local_rank)
    chains = []
    for ch in range(args.chains):
        s = mvc_b200.Sampler(n, [1, 1], cap=32, seed=SEED, chain=rank * args.chains + ch, device=local_rank, engine=1)
        for v, x in enumerate(views):
            s.upload_view(v, x.astype(np.float32).reshape(-1, 1))
        s.init_state_reference()
        chains.append(s)
    block = 25                                    # sweeps queued per chain before moving to the next stream
    def run(k):
        done = 0
        while done < k:
            b = min(block, k - done)
            for s in chains:
                s.sweep(b, True)
            done += b
        for s in chains:
            s.sync()
    run(args.warmup)
    l0 = sum(s.launch_count() for s in chains)
    t0 = time.perf_counter()
    run(steps)
    dt = time.perf_counter() - t0
    launches = sum(s.launch_count() for s in chains) - l0
    one_ms = chains[0].last_sweep_ms() / min(block, steps)
    live = [int((s.get_state(with_rows=False)["n_t"] > 0).sum()) for s in chains]
    for s in chains:
        s.close()
    if rank == 0:
        line = {"metric": "gibbs_sweeps_per_s", "value": world * args.chains * steps / dt, "unit": "sweeps/s", "n_gpus": world,
                "steps": steps, "warmup": args.warmup, "ms_per_step": 1e3 * dt / steps, "higher_is_better": True,
                "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                "config": {"workload": "C1: New_Simulation.R two scalar views, N=%d, %d independent chains per GPU "
                                       "(one stream each), CUDA-core engine, hyper step on" % (n, args.chains),
                           "timing": "wall clock around the launches of all chains and their final synchronisation"},
                "single_chain_ms_per_sweep_device": one_ms, "gpu_launches": int(launches), "tables_live": live}
        print(json.dumps(line), file=out)


def run_reference(args, out):
    """--impl reference: the reference's CPU implementation of the path on the host cores.  The
    reference sampler itself has no D > 1 likelihood (SURVEY.md §0), so on this configuration the
    CPU arm is the restated port of its arithmetic (oracle/mv_oracle.c, kind "port"), all host threads."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    threads = os.cpu_count() or 1
    rows = args.cpu_rows or 262144
    for _ in range(min(args.warmup, 1)):
        cpu_port_throughput(min(rows, 2048), threads)
    vals, dts = [], []
    for _ in range(max(1, min(args.steps, 5))):
        v, dt = cpu_port_throughput(rows, threads)
        vals.append(v); dts.append(dt)
    value = float(np.mean(vals))
    sample = f"one FP64 sweep over the first {rows} customers of the C3 workload per step, {threads} OpenMP threads"
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
            "steps": len(vals), "warmup": min(args.warmup, 1), "ms_per_step": 1e3 * float(np.mean(dts)),
            "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": "C3: 3-view Gaussian mixture N=1M D=64 K=64 (bounded CPU sample)", "rows_sampled": rows},
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": "port", "sample": sample},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), file=out)


def main():
    args = parse()
    # stdout carries exactly ONE JSON line: anything a library prints there while we run (NCCL's version banner,
    # for one) is sent to stderr instead, and the line is written to the real stdout at the end
    sys.stdout.flush()
    real_stdout = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    try:
        _main(args, real_stdout)
    finally:
        real_stdout.flush()


def _main(args, out):
    if args.workload == "c1":
        return run_c1(args, out)
    if args.workload == "c2":
        return run_c2(args, out)
    if args.workload == "c5":
        return run_c5(args, out)
    if args.impl == "reference":
        return run_reference(args, out)

    import torch
    import mvc_b200

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the sweep has no CPU path")
    torch.cuda.set_device(local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    mus = planted_means(np.random.default_rng(SEED))
    do_hyper = not args.no_hyper
    peak, peak_src = measured_peak()

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    def shard_of(n_total):
        return rank * n_total // world, (rank + 1) * n_total // world

    class Workload:
        """One chain of n_total customers, this rank's shard resident on its GPU."""
        def __init__(self, n_total, k_true, spread=None):
            self.n_total, self.k_true = n_total, k_true
            self.lo, self.hi = shard_of(n_total)
            self.n_local = self.hi - self.lo
            self.mus = mus if spread is None else planted_means(np.random.default_rng(SEED), spread)
            views_np, z = make_rows_numpy(self.lo, self.hi, self.mus, k_true=k_true)
            self.tab, self.dish, self.hyp = initial_state(z, k_true)
            self.pinned = [torch.from_numpy(v).pin_memory() for v in views_np]
            self.dev = [v.cuda(non_blocking=True) for v in self.pinned]
            torch.cuda.synchronize()

        def set_state(self, s):
            h = self.hyp
            s.set_state(self.tab, self.dish, h["alpha_v"], h["sigma_v"], h["tau_v"], h["alpha_g"], h["sigma_g"])

    comm_owner = []          # the first multi-GPU sampler owns the NCCL communicator; the others borrow it

    def make_sampler(w, attach, debug_export=0, single=False, incremental=None):
        """single: a one-GPU chain over this rank's rows only (checks that need no peers)."""
        ww, rr = (1, 0) if single else (world, rank)
        s = mvc_b200.Sampler(w.n_local, DIMS, cap=CAP, seed=SEED, device=local_rank, engine=args.engine, rank=rr,
                             world=ww, row_offset=0 if single else w.lo, n_rows_global=w.n_local if single else w.n_total,
                             debug_export=debug_export)
        if ww > 1:
            if comm_owner:
                s.comm_attach(comm_owner[0].comm_handle())
            else:
                uid = [mvc_b200.Sampler.nccl_unique_id() if rank == 0 else None]
                dist.broadcast_object_list(uid, src=0)
                s.comm_init_rank(uid[0])
                comm_owner.append(s)
        if attach:
            for v in range(len(DIMS)):
                s.attach_view_device(v, w.dev[v])
        if (args.stats == "incremental") if incremental is None else incremental:
            s.set_stats_mode(True, 64)
        return s

    transport = {"used": "none" if world == 1 else "nccl"}

    def enable_p2p(s):
        """Peer-memory exchange: every rank exports its receive buffer, all map all."""
        want = args.exchange if args.exchange != "auto" else "p2p"
        if world == 1 or want != "p2p":
            return
        ok = 1
        try:
            mine = s.p2p_export()
        except Exception as e:                                  # noqa: BLE001
            mine, ok = b"\0" * 64, 0
            print(f"[rank {rank}] p2p export failed, using NCCL: {e}", file=sys.stderr)
        handles = [None] * world
        dist.all_gather_object(handles, (ok, mine))
        if all(h[0] for h in handles):
            try:
                s.p2p_attach([h[1] for h in handles])
            except Exception as e:                              # noqa: BLE001
                ok = 0
                print(f"[rank {rank}] p2p attach failed, using NCCL: {e}", file=sys.stderr)
        else:
            ok = 0
        flag = torch.tensor([ok], device="cuda")
        dist.all_reduce(flag, op=dist.ReduceOp.MIN)
        if int(flag.item()) == 1:
            transport["used"] = "p2p"
        elif ok:
            s.p2p_disable()                                     # a peer could not map the buffers: everybody uses NCCL

    def timed_run(w, steps, warmup, sample_clocks, incremental=None, keep_state=False):
        """W warm-up sweeps, then `steps` sweeps timed on the device (CUDA events on the library's stream, barrier and
        synchronize on both sides, max over ranks).  keep_state: also return the state the last timed sweep left."""
        s = make_sampler(w, attach=True, debug_export=2 if args.role_profile else 0, incremental=incremental)
        enable_p2p(s)
        w.set_state(s)
        s.sweep(warmup, do_hyper)
        s.sync()
        for which in (0, 1):
            s.kernel_clock(which, reset=True)
        clocks = ClockSampler(local_rank) if sample_clocks else None
        barrier()
        if clocks:
            clocks.start()
        l0 = s.launch_count()
        t_wall = time.perf_counter()
        s.sweep(steps, do_hyper)
        s.sync()
        barrier()
        wall_ms = 1e3 * (time.perf_counter() - t_wall)
        if clocks:
            clocks.stop_flag = True
        state = s.get_state() if keep_state else None         # before profile_sweep below, which sweeps again
        t = torch.tensor([s.last_sweep_ms()], device="cuda")
        if dist is not None:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dev_ms = float(t.item())
        # the kernels of the timed sweeps themselves, by the library's in-kernel wall clocks (the sweeps are graph replays)
        d_ms, d_n = s.kernel_clock(0)
        d_last = s.kernel_clock_last
        f_ms, f_n = s.kernel_clock(1)
        f_last = s.kernel_clock_last
        inreg = {"draw": d_ms / d_n if d_n else None, "draw_launches": d_n,
                 "finalize": f_ms / f_n if f_n else None, "finalize_launches": f_n}
        if d_n > 1 and f_n > 0 and d_last[0] > f_last[1] > f_last[0] > d_last[2] > 0:
            # the last sweep's tail: draw out -> [pack, statistics, reduce + exchange] -> finalize in .. out -> next draw's inputs ready
            inreg["tail_us"] = {"draw_out_to_finalize_in": 1e-3 * (f_last[0] - d_last[2]), "finalize": 1e-3 * (f_last[1] - f_last[0]),
                                "finalize_out_to_draw_ready": 1e-3 * (d_last[0] - f_last[1])}
        prof = [s.profile_sweep(do_hyper) for _ in range(5)]      # per-kernel device times of a few extra sweeps
        kern = {k: float(np.median([p[k] for p in prof])) for k in prof[0]}
        return {"s": s, "dev_ms": dev_ms, "wall_ms": wall_ms, "launches": s.launch_count() - l0, "kern": kern, "inreg": inreg,
                "clocks": clocks.summary() if clocks else None, "state": state}

    def roofline_of(w, kern, traffic, inreg=None):
        alg_bytes = w.n_local * (sum(DIMS) * 4 + 8)
        achieved = alg_bytes / (kern["draw"] * 1e-3) / 1e9
        timed = None
        if inreg and inreg.get("draw"):
            a2 = alg_bytes / (inreg["draw"] * 1e-3) / 1e9
            timed = {"kernel_ms": {"draw": inreg["draw"], "finalize": inreg["finalize"]}, "launches": inreg["draw_launches"],
                     "last_sweep_tail_us": inreg.get("tail_us"),
                     "achieved": a2, "frac": a2 / peak,
                     "clock": "%globaltimer inside the kernel, first CTA in (once its grid dependency has resolved) to last CTA "
                              "out, averaged over every launch of the timed region (graph replays; events cannot be placed there)"}
        return {"in_timed_region": timed, "bound": "hbm", "kernel": "likelihood+draw", "achieved": achieved, "peak": peak, "unit": "GB/s",
                "frac": achieved / peak, "traffic": traffic,
                "traffic_source": "ncu --set full, dram__bytes_read.sum + dram__bytes_write.sum of k_draw_tc at N=1M "
                                  "(profiles/), scaled to this shard", "peak_source": peak_src,
                "algorithmic_bytes_per_launch": alg_bytes, "kernel_ms": kern, "planted_clusters": w.k_true,
                "free_table_slots": CAP - w.k_true}

    # ---------------- the headline run: `--scaling` (default strong: north_star's N = 1M split over the GPUs) ----------
    n_total = args.rows * world if args.scaling == "weak" else args.rows
    W = Workload(n_total, args.k_true)
    R = timed_run(W, args.steps, args.warmup, sample_clocks=True, keep_state=bool(args.dump_outputs))
    s = R["s"]
    if args.dump_outputs:
        dump_state(R["state"], W.lo, args.dump_outputs, dist, rank, world)
    ms_per_step = R["dev_ms"] / args.steps
    updates = n_total * len(DIMS) * CAP
    value = updates * args.steps / (R["dev_ms"] * 1e-3)
    traffic = NCU_TRAFFIC_BYTES * W.n_local / N_ROWS if args.engine in (0, 2, 3) else None
    roofline = roofline_of(W, R["kern"], traffic, R["inreg"])
    if args.role_profile and rank == 0:
        pr = s.get_debug_prof(n_ctas=256)
        for role in range(len(DIMS) + 1):                      # view CTAs, then the franchise CTA (cycles since the CTA began)
            print("finalize stamps, CTA %d:" % role, pr[200 + role, :13].tolist(), file=sys.stderr)
        print("epilogue phases of CTA 0 pair 0 (cycles; lower half | upper half): prologue, views, corr+max, rdv1, marg+weights, rdv2, "
              "scan, rdv3, write, [acc wait]:", pr[230, :10].tolist(), "|", pr[231, :10].tolist(), file=sys.stderr)
        pr = pr[:148]
        names = ["tma.wait_raw_empty", "tma.total", "mma.wait_d_empty", "mma.wait_raw_full", "mma.wait_lo_full", "mma.total",
                 "conv0.wait_raw_full", "conv0.wait_lo_empty", "conv0.total", "conv1.wait_raw_full", "conv1.wait_lo_empty",
                 "conv1.total", "epi0.wait", "epi0.total", "epi1.wait", "epi1.total"]
        med = np.median(pr, axis=0)
        print("role profile (median cycles over CTAs):", {n: int(m) for n, m in zip(names, med)}, file=sys.stderr)
    final = s.get_state(with_rows=False)
    state_check = {"tables_live": int((final["n_t"] > 0).sum()), "customers": int(final["n_t"].sum())}
    if not comm_owner or comm_owner[0] is not s:
        s.close()

    # ---------------- e2e: one chain through the C ABI with HOST buffers ---------------------------------------------------
    e2e = None
    if not args.no_e2e:
        k_e2e = args.steps
        thin = max(1, k_e2e // 4)
        s2 = make_sampler(W, attach=False)       # handle (+ borrowed communicator): set-up, not part of a chain's run
        barrier()
        t0 = time.perf_counter()
        for v in range(len(DIMS)):
            s2.upload_view(v, W.pinned[v].numpy())
        if transport["used"] == "p2p":
            enable_p2p(s2)
        t_up = time.perf_counter()
        W.set_state(s2)
        t_st = time.perf_counter()
        trace = s2.run(k_e2e, 0, thin)           # gibbs_sampler(M, burn_in, thin): D2H of table_of on every kept sweep
        barrier()
        dt = time.perf_counter() - t0
        parts_s = {"upload": t_up - t0, "set_state": t_st - t_up, "run": t0 + dt - t_st}
        tt = torch.tensor([dt], device="cuda")
        if dist is not None:
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        dt = float(tt.item())
        n_saved = int(trace["table_of"].shape[0])
        h2d = W.n_local * (sum(DIMS) * 4 + 4)
        d2h = W.n_local * 4 * n_saved
        e2e = {"value": updates * k_e2e / dt, "unit": UNIT, "h2d_bytes_per_step": h2d / k_e2e,
               "d2h_bytes_per_step": d2h / k_e2e, "sweeps": k_e2e, "saved_states": n_saved, "seconds": dt, "seconds_by_part": parts_s,
               "note": "one chain through the C ABI (mvg_upload_view_f32 from pinned host memory, mvg_set_state, mvg_run = "
                       "gibbs_sampler(M, burn_in=0, thin) with the D2H of table_of on every kept sweep); wall clock, device "
                       "allocation included; bytes are per sweep (total / M)"}
        assert int(np.bincount(trace["table_of"][-1], minlength=CAP).sum()) == W.n_local
        s2.close()
    # ---------------- the same kernel with free table slots (the new-table marginal is evaluated): one GPU only ---------
    roofline_free = None
    if world == 1 and not args.no_free_slots and args.k_true == CAP:
        Wf = Workload(n_total, CAP - 4)
        Rf = timed_run(Wf, min(args.steps, 200), min(args.warmup, 5), sample_clocks=False)
        roofline_free = roofline_of(Wf, Rf["kern"], None, Rf["inreg"])
        roofline_free["ms_per_step"] = Rf["dev_ms"] / min(args.steps, 200)
        Rf["s"].close()
        del Wf, Rf

    # ---------------- the other statistics mode, and a data set whose rows keep moving (overlapping clusters) ----------
    stats_other, moving = None, None
    if not args.no_extra:
        ks = min(args.steps, 200)
        other = args.stats != "incremental"
        Ro = timed_run(W, ks, min(args.warmup, 5), sample_clocks=False, incremental=other)
        stats_other = {"stats": "incremental" if other else "rebuild", "steps": ks, "ms_per_step": Ro["dev_ms"] / ks,
                       "value": updates * ks / (Ro["dev_ms"] * 1e-3), "unit": UNIT, "kernel_ms": Ro["kern"]}
        if not comm_owner or comm_owner[0] is not Ro["s"]:
            Ro["s"].close()
        del Ro
        if world == 1:
            Wm = Workload(n_total, args.k_true, spread=0.35)     # cluster centres ~4 sigma apart: a few per cent of the rows move every sweep
            Rm = timed_run(Wm, ks, 20, sample_clocks=False)
            t_a = Rm["s"].get_state()["table_of"]
            Rm["s"].sweep(1, do_hyper)
            t_b = Rm["s"].get_state()["table_of"]
            moving = {"workload": "same shape, planted means N(0, 0.35^2 I): overlapping clusters", "stats": args.stats, "steps": ks,
                      "ms_per_step": Rm["dev_ms"] / ks, "value": updates * ks / (Rm["dev_ms"] * 1e-3), "unit": UNIT,
                      "kernel_ms": Rm["kern"], "rows_moved_in_one_sweep": int((t_a != t_b).sum()),
                      "tables_live": int((Rm["s"].get_state(with_rows=False)["n_t"] > 0).sum())}
            Rm["s"].close()
            del Wm, Rm

    # ---------------- weak scaling beside it (N > 1): one C3-sized shard per GPU ---------------------------------------
    weak = None
    if world > 1 and args.scaling == "strong" and not args.no_weak:
        Ww = Workload(args.rows * world, args.k_true)
        kw = min(args.steps, 200)
        Rw = timed_run(Ww, kw, min(args.warmup, 5), sample_clocks=False)
        weak = {"scaling": "weak", "rows_total": Ww.n_total, "rows_per_gpu": Ww.n_local, "steps": kw,
                "ms_per_step": Rw["dev_ms"] / kw, "value": Ww.n_total * len(DIMS) * CAP * kw / (Rw["dev_ms"] * 1e-3),
                "unit": UNIT, "kernel_ms": Rw["kern"]}
        if not comm_owner or comm_owner[0] is not Rw["s"]:
            Rw["s"].close()
        del Ww, Rw

    # ---------------- checks outside every timed region ------------------------------------------------------------------
    # (1) sharded chain against the same chain on one GPU (N > 1): every rank runs K sweeps sharded, rank 0 replays them
    #     unsharded over all rows; the draws are addressed by global row, so sweep 1 must be identical.
    if world > 1 and not args.no_checks:
        kc = max(2, min(args.steps, 20))
        s3 = make_sampler(W, attach=True)
        if transport["used"] == "p2p":
            enable_p2p(s3)
        W.set_state(s3)
        s3.sweep(1, do_hyper)
        t1 = s3.get_state()["table_of"]
        s3.sweep(kc - 1, do_hyper)
        st3 = s3.get_state()
        parts = [None] * world
        dist.all_gather_object(parts, (W.lo, t1, st3["table_of"], st3["n_t"], st3["tau_v"]))
        s3.close()
        if rank == 0:
            parts.sort(key=lambda p: p[0])
            tab1 = np.concatenate([p[1] for p in parts])
            tabK = np.concatenate([p[2] for p in parts])
            full_views, zfull = make_rows_numpy(0, n_total, mus, k_true=args.k_true)
            tab0, dish0, hyp0 = initial_state(zfull, args.k_true)
            one = mvc_b200.Sampler(n_total, DIMS, cap=CAP, seed=SEED, device=local_rank, engine=args.engine)
            for v in range(len(DIMS)):
                one.upload_view(v, full_views[v])
            one.set_state(tab0, dish0, hyp0["alpha_v"], hyp0["sigma_v"], hyp0["tau_v"], hyp0["alpha_g"], hyp0["sigma_g"])
            one.sweep(1, do_hyper)
            a1 = float((one.get_state()["table_of"] == tab1).mean())
            one.sweep(kc - 1, do_hyper)
            ref = one.get_state()
            one.close()
            del full_views
            state_check.update({"sharded_vs_one_gpu_sweeps": kc, "first_sweep_identical": bool(a1 == 1.0),
                                "first_sweep_agreement": a1,
                                "agreement_after_K": float((ref["table_of"] == tabK).mean()),
                                "replicas_identical": bool(all(np.array_equal(p[3], parts[0][3]) and
                                                               np.array_equal(p[4], parts[0][4]) for p in parts)),
                                "tau_rel_diff_vs_one_gpu": float(np.max(np.abs(ref["tau_v"] - parts[0][4]) / ref["tau_v"]))})
    # (2) draws of one sweep at full size against the CPU mirror (oracle/mv_oracle.c), fed the device's dot products and
    #     the same Philox uniforms, on the rows of 12 CTAs spread over the grid (first, middle, last) plus the ragged tail.
    if rank == 0 and not args.no_checks:
        state_check.update(spot_check_draws(mvc_b200, W, local_rank, args.engine))

    for s_ in comm_owner:
        s_.close()

    cpu = None
    if rank == 0 and not args.no_cpu_baseline:
        rows = args.cpu_rows or 524288          # ~10 s of one core
        v1, dt1 = cpu_port_throughput(rows, 1)
        cpu = {"value": v1, "unit": UNIT, "cores": 1, "kind": "port",
               "sample": f"one FP64 sweep of oracle/mv_oracle.c over the first {rows} customers of the same workload, "
                         f"1 thread ({dt1:.2f} s); the reference sampler itself has no D>1 path (SURVEY.md §0)"}

    if rank == 0:
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None,
                "dtype": "f32", "data": "synthetic",
                "config": {"workload": "C3: synthetic 3-view Gaussian mixture, N=%d (%d per GPU), D=64/view, K(cap)=64, row-sharded, "
                                       "one exchange of the per-table statistics per sweep" % (n_total, W.n_local),
                           "rows_per_gpu": W.n_local, "hyper_step": do_hyper, "engine": args.engine, "planted_clusters": args.k_true,
                           "l2": "inputs (768 MB per sweep at N=1M) larger than L2; no flush", "exchange": transport["used"],
                           "statistics": args.stats + (" (moved rows only, full rebuild every 64 sweeps)" if args.stats == "incremental" else " (all rows every sweep)")},
                "sweeps_per_s": args.steps / (R["dev_ms"] * 1e-3), "wall_ms_per_step": R["wall_ms"] / args.steps,
                "clocks": R["clocks"], "gpu_launches": int(R["launches"]),
                "roofline": roofline, "roofline_free_slots": roofline_free, "stats_rebuild" if args.stats == "incremental" else "stats_incremental": stats_other,
                "moving_rows": moving, "weak": weak, "e2e": e2e, "cpu_baseline": cpu,
                "state_check": state_check}
        print(json.dumps(line), file=out)
    if dist is not None:
        dist.destroy_process_group()


def dump_state(st, lo, out_dir, dist, rank, world):
    """The state after the last timed sweep as <out_dir>/<name>.npy: table_of in row order (gathered from the ranks; every
    row up to 8M rows, beyond that every k-th row so that the dump stays under 64 MB), the per-table counts and sums and
    the hyperparameters, which every rank holds alike."""
    tab = st["table_of"]
    if dist is not None:
        parts = [None] * world
        dist.all_gather_object(parts, (lo, tab))
        tab = np.concatenate([p[1] for p in sorted(parts, key=lambda p: p[0])])
    if rank != 0:
        return
    tab = tab[::-(-len(tab) // 8_000_000)]
    out = {"table_of": tab.astype(np.float32), "n_t": st["n_t"].astype(np.float32),
           "dish_of": st["dish_of"].astype(np.float32), "n_vk": st["n_vk"].astype(np.float32),
           "l_vk": st["l_vk"].astype(np.float32), "sum_y": np.stack(st["S1"]), "sum_y2": st["sum_y2"],
           "alpha_v": st["alpha_v"], "sigma_v": st["sigma_v"], "tau_v": st["tau_v"],
           "alpha_sigma_global": np.array([st["alpha_g"], st["sigma_g"]])}
    d = Path(out_dir)
    d.mkdir(parents=True, exist_ok=True)
    for name, a in out.items():
        np.save(d / f"{name}.npy", a)


def spot_check_draws(mvc_b200, W, device, engine):
    """One sweep of a debug handle over this rank's rows (a one-GPU chain), then the CPU mirror of the draw stage on the
    rows of 12 CTAs of the draw kernel's grid and on the last tile: integer draws must be identical."""
    sys.path.insert(0, str(ROOT / "oracle"))
    import pyoracle as po
    n = W.n_local
    s = mvc_b200.Sampler(n, DIMS, cap=CAP, seed=SEED, device=device, engine=engine, debug_export=1)
    for v in range(len(DIMS)):
        s.attach_view_device(v, W.dev[v])
    W.set_state(s)
    s.sweep(1, True)                         # leave the planted state once, so that rows sit at wrong tables too
    pre = s.get_state()
    P = s.get_params()
    s.sweep(1, True)
    acc, xx, raw = s.get_debug_rows()
    lnew = s.get_debug_lnew()
    s.close()
    n_tiles = (n + 127) // 128
    grid = min(148, n_tiles)
    ctas = sorted({c for c in (0, 1, 2, 3, grid // 2 - 1, grid // 2, grid // 2 + 1, grid // 2 + 2, grid - 4, grid - 3,
                               grid - 2, grid - 1) if 0 <= c < grid})
    tiles = sorted({t for c in ctas for t in range(c, n_tiles, grid)} | {n_tiles - 1})
    rows = np.concatenate([np.arange(t * 128, min(n, (t + 1) * 128)) for t in tiles])
    ps = po.params_struct(P)
    L = po.lib()
    bad = 0
    for i in rows:
        u = L.mvo_uf(SEED, 0, 0, 0, pre["sweep"], int(i))
        bad += int(po.stageB_tc(ps, acc[i], xx[i], pre["table_of"][i], u, lnew[i]) != raw[i])
    # dot products against FP64 on a subset (tolerance: 2^-18 of sum |x||m|, DESIGN.md §5)
    sub = rows[:: max(1, len(rows) // 4096)]
    worst = 0.0
    for v in range(len(DIMS)):
        x = W.pinned[v].numpy()[sub].astype(np.float64)
        m = po.scaled_means(P["A"][v], P["m"][v]).astype(np.float64)      # the engine's B operand: b = float32(2 A m)
        ref = x @ m.T
        bound = np.abs(x) @ np.abs(m).T
        worst = max(worst, float(np.max(np.abs(acc[sub, v, :] - ref) / bound)))
    return {"draws_checked_rows": int(len(rows)), "draws_bit_exact_rows": int(len(rows) - bad), "draws_mismatched": int(bad),
            "dot_rel_err_max": worst, "dot_rel_err_bound": 2.0 ** -18, "rows_moved_in_checked_sweep": int((raw != pre["table_of"]).sum())}


if __name__ == "__main__":
    main()
