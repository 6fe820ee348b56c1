"""Config 4 on one GPU (SURVEY.md §8d C4): N = 4M customers, 4 dense views as C3 (D = 64) and 4 sparse count views
(vocab 16 384, nnz/row ~ Poisson(48), counts ~ 1 + Geometric(1/2)), table capacity K = 256, CUDA-core engine.

Data (seed 1999, generated on the GPU): 96 planted clusters z; dense x = mu_vz + N(0, I), mu ~ N(0, 2^2 I); a count row
draws half of its words from a 512-word band of its cluster and half uniformly.  Start: over-split — cluster z sits at
table z or z + 96 (coin flip), each table its own dish, 64 of the 256 slots free.  After a warm-up, a timed window of
--sweeps sweeps (CUDA events of the library's stream, mvg_last_sweep_ms), then a per-kernel split (mvg_profile_sweep),
the same split for a cap-64 handle on the same data (k_finalize at 256 vs 64), and a state check.
Prints one JSON object; --out writes it too.

    python profiles/c4_probe.py --out profiles/r03_c4_1gpu.json
"""
import argparse
import json
import subprocess
import sys
import time
from pathlib import Path

import numpy as np
import torch

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT / "multiview-clustering_b200"))
import mvc_b200  # noqa: E402

N, DENSE, D, CSR, VOCAB, NNZ_MEAN, K_TRUE, SEED = 4_000_000, 4, 64, 4, 16384, 48, 96, 1999


def device_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader,nounits",
                        "-i", "0"], capture_output=True, text=True).stdout.strip().split(", ")
    p = torch.cuda.get_device_properties(0)
    return {"name": q[0] if q and q[0] else p.name, "power_limit_w": float(q[1]), "max_sm_clock_mhz": float(q[2]),
            "sms": p.multi_processor_count}


def make_data(n):
    g = torch.Generator(device="cuda").manual_seed(SEED)
    z = torch.randint(0, K_TRUE, (n,), device="cuda", generator=g)
    dense = []
    for _ in range(DENSE):
        mu = torch.randn(K_TRUE, D, device="cuda", generator=g) * 2.0
        dense.append((mu[z] + torch.randn(n, D, device="cuda", generator=g)).contiguous())
    csr = []
    for _ in range(CSR):
        lens = torch.poisson(torch.full((n,), float(NNZ_MEAN), device="cuda"), generator=g).clamp_(min=1).to(torch.int64)
        rowptr = torch.zeros(n + 1, dtype=torch.int64, device="cuda")
        rowptr[1:] = torch.cumsum(lens, 0)
        nnz = int(rowptr[-1])
        row = torch.repeat_interleave(torch.arange(n, device="cuda"), lens)
        band = (z[row] * 160 + torch.randint(0, 512, (nnz,), device="cuda", generator=g)) % VOCAB
        uni = torch.randint(0, VOCAB, (nnz,), device="cuda", generator=g)
        col = torch.where(torch.rand(nnz, device="cuda", generator=g) < 0.5, band, uni).to(torch.int32)
        val = torch.empty(nnz, device="cuda").geometric_(0.5, generator=g)      # 1, 2, ... = 1 + Geometric
        csr.append((rowptr.to(torch.int32).cpu().numpy(), col.cpu().numpy(), val.cpu().numpy()))
        del lens, row, band, uni, col, val
    coin = torch.rand(n, device="cuda", generator=g) < 0.5
    tab = (z + K_TRUE * coin.to(z.dtype)).to(torch.int32).cpu().numpy()
    return z.cpu().numpy(), dense, csr, tab


def make_sampler(cap, dense, csr, tab, n):
    dims = [D] * DENSE + [0] * CSR
    s = mvc_b200.Sampler(n, dims, cap=cap, seed=SEED, engine=mvc_b200.ENGINE_AUTO)
    for v in range(DENSE):
        s.attach_view_device(v, dense[v])
    for j, (rp, col, val) in enumerate(csr):
        s.upload_view_csr(DENSE + j, rp, col, val, VOCAB)
    dish = np.full((DENSE + CSR, cap), -1, np.int32)
    live = int(tab.max()) + 1
    dish[:, :live] = np.arange(live)
    V = DENSE + CSR
    s.set_state(tab, dish, [1.0] * V, [0.5] * V, [1.0] * V, 1.0, 0.6)
    return s


def split(s, reps):
    runs = [s.profile_sweep(do_hyper=True) for _ in range(reps)]
    return {k: float(np.median([r[k] for r in runs])) for k in runs[0]}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rows", type=int, default=N)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--sweeps", type=int, default=40)
    ap.add_argument("--profile-reps", type=int, default=5)
    ap.add_argument("--out")
    a = ap.parse_args()
    n = a.rows
    dev = device_info()
    t0 = time.perf_counter()
    z, dense, csr, tab = make_data(n)
    nnz = [int(c[0][-1]) for c in csr]
    t_data = time.perf_counter() - t0

    s = make_sampler(256, dense, csr, tab, n)
    s.sweep(a.warmup, do_hyper=True)
    s.sync()
    launches0 = s.launch_count()
    s.sweep(a.sweeps, do_hyper=True)
    s.sync()
    ms_window = s.last_sweep_ms()
    launches = s.launch_count() - launches0
    prof256 = split(s, a.profile_reps)
    st = s.get_state()
    s.close()
    n_t = st["n_t"]
    state_check = {"n_t_sums_to_N": int(n_t.sum()) == n,
                   "customers_conserved": bool(np.array_equal(np.bincount(st["table_of"], minlength=256), n_t)),
                   "dish_counts_consistent": bool(all(np.array_equal(np.bincount(st["dish_of"][v][n_t > 0], minlength=256),
                                                                     st["l_vk"][v]) for v in range(DENSE + CSR)))}
    tables_live = int((n_t > 0).sum())

    # the same data at cap 64 (tables folded onto 64 slots): k_finalize and the rest of the split for comparison
    s64 = make_sampler(64, dense, csr, (tab % 64).astype(np.int32), n)
    s64.sweep(a.warmup, do_hyper=True)
    prof64 = split(s64, a.profile_reps)
    s64.close()

    ms = ms_window / a.sweeps
    # work per sweep from the shapes
    dense_flop = 2.0 * n * 256 * D * DENSE                            # x . m_t for every customer, table and dense view
    count_flop = 2.0 * sum(nnz) * 256                                 # x_j log2 theta[col_j][t] for every nonzero and table
    hbm_bytes = (2 * 4.0 * n * D * DENSE                              # dense features: draw kernel + statistics rebuild
                 + CSR * 2 * 4.0 * n * 256                            # cnt_acc written by k_counts_loglik, read by the draw
                 + sum(8.0 * x for x in nnz))                         # CSR (col, val) read by k_counts_loglik
    l2_bytes = sum(4.0 * 256 * x for x in nnz)                        # l2t rows gathered per nonzero (16 MB table per view)
    fp32_peak = dev["sms"] * 128 * 2 * dev["max_sm_clock_mhz"] * 1e6   # FP32 CUDA-core FMA lanes at the max SM clock
    hbm_peak = 7.7e12                                                  # HBM3e, NVIDIA HGX B200 data sheet, per GPU
    t_flop = (dense_flop + count_flop) / fp32_peak
    t_hbm = hbm_bytes / hbm_peak
    bound = "fp32_cuda_core" if t_flop >= t_hbm else "hbm"
    res = {
        "workload": f"C4: N={n}, 4 dense views D=64 + 4 CSR views (vocab {VOCAB}, nnz/row ~ Poisson({NNZ_MEAN}), counts 1+Geometric(1/2)), "
                    f"cap=256, {K_TRUE} planted clusters, over-split start (192 live tables, 64 free), seed {SEED}",
        "engine": "CUDA-core (MVG_ENGINE_AUTO at cap 256)",
        "device": dev,
        "data_generation_s": round(t_data, 2),
        "nnz_per_view": nnz,
        "warmup_sweeps": a.warmup, "timed_sweeps": a.sweeps,
        "ms_per_sweep": ms,
        "ms_per_sweep_source": "CUDA events on the library stream around the timed mvg_sweep call (mvg_last_sweep_ms) / sweeps",
        "per_kernel_ms_cap256": prof256,
        "per_kernel_ms_cap64_same_data": prof64,
        "per_kernel_source": f"mvg_profile_sweep (CUDA events per phase), median of {a.profile_reps} sweeps after the window; "
                             "draw includes k_counts_loglik",
        "launches_per_sweep": launches / a.sweeps,
        "work_per_sweep": {"dense_gflop": dense_flop / 1e9, "count_gflop": count_flop / 1e9, "hbm_gb": hbm_bytes / 1e9,
                           "l2_gather_gb": l2_bytes / 1e9},
        "share_of_peak": {
            "bound": bound,
            "min_time_ms": 1e3 * max(t_flop, t_hbm),
            "fraction": 1e3 * max(t_flop, t_hbm) / ms,
            "peaks": {"fp32_tflops": fp32_peak / 1e12, "fp32_note": "SMs x 128 FP32 lanes x 2 x max SM clock (read in this run)",
                      "hbm_tb_s": hbm_peak / 1e12},
            "note": "whole-sweep time against the larger of (all FLOPs at the FP32 CUDA-core peak) and (HBM bytes at data-sheet "
                    "bandwidth); an end-to-end figure, not a kernel's share. The l2t gathers (L2-resident) are not in the bound."},
        "tables_live": tables_live,
        "state_check": state_check,
    }
    print(json.dumps(res))
    if a.out:
        Path(a.out).write_text(json.dumps(res, indent=1) + "\n")


if __name__ == "__main__":
    main()
