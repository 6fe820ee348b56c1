"""tests/golden/make_chain_golden.py — regenerate tests/golden/reference_chains.npz from the UNMODIFIED reference.

Run where the reference sources exist (oracle/Makefile compiles them into oracle/_ref/libmvref.so):

    python tests/golden/make_chain_golden.py

Every chain is run_gibbs_cpp of the compiled reference (pyoracle.ref_run_gibbs) on config-1 data (conftest.c1_data);
the tests compare the sequential engine on the host and on the device, the host layer and the GPU chain's posterior
summaries with these saved states, so they run where the reference is absent.  The script refuses to run without
the compiled reference: the file must never be rewritten from the code it checks.  The file's "source" entry says
what produced its arrays.

One chain per key "<seed>_<n>_<M>_<burn>_<thin>": table_of [S, n], T [S], dish_of [S, 2, max T] (-1 past T),
hypers [S, 8] = alpha_v, sigma_v, tau_v, alpha_global, sigma_global, and calls (uniforms + normals drawn).
"""
import sys
from pathlib import Path

import numpy as np

TESTS = Path(__file__).resolve().parents[1]
ROOT = TESTS.parent
sys.path[:0] = [str(TESTS), str(ROOT / "oracle")]
import pyoracle as po  # noqa: E402
from conftest import c1_data  # noqa: E402

OUT = Path(__file__).with_name("reference_chains.npz")
SOURCE = "run_gibbs_cpp of the compiled, unmodified reference (oracle/_ref/libmvref.so via pyoracle.ref_run_gibbs)"
CHAINS = [
    (1999, 500, 300, 100, 10), (7, 500, 400, 0, 40), (42, 200, 500, 250, 25),    # test_seq_engine, CPU
    (7, 500, 600, 0, 50),                                                        # test_seq_engine, device
    (11, 300, 200, 100, 20),                                                     # test_host_layer
    (1999, 500, 1500, 1200, 10),                                                 # test_gpu_parity: posterior summaries
    *[(sd, 500, 2000, 1500, 10) for sd in (1999, 7, 42, 2024)],                 # test_gpu_parity: long-chain statistics
]


def run(seed, n, M, burn, thin):
    views, _ = c1_data(n)
    y = np.stack([v.astype(np.float64) for v in views])
    tr = po.ref_run_gibbs(y, M, burn, thin, seed=seed)
    calls = po.ref().ref_uniform_calls() + po.ref().ref_normal_calls()
    T = np.array([t["dish_of"].shape[1] for t in tr], np.int32)
    dish = np.full((len(tr), y.shape[0], T.max()), -1, np.int16)
    for s, t in enumerate(tr):
        dish[s, :, :T[s]] = t["dish_of"]
    hyp = np.array([np.concatenate([t["alpha_v"], t["sigma_v"], t["tau_v"], [t["alpha_global"], t["sigma_global"]]])
                    for t in tr])
    return {"table_of": np.stack([t["table_of"] for t in tr]).astype(np.int16), "T": T, "dish_of": dish, "hypers": hyp,
            "calls": np.uint64(calls)}


def main():
    if not po.have_ref():
        po.build()
    if not po.have_ref():
        raise SystemExit("the compiled reference (oracle/_ref/libmvref.so) is needed: see oracle/Makefile")
    out = {"source": np.array(SOURCE)}
    for key in CHAINS:
        name = "_".join(map(str, key))
        for k, a in run(*key).items():
            out[f"{name}/{k}"] = a
    np.savez_compressed(OUT, **out)
    print("wrote", OUT, OUT.stat().st_size, "bytes")


if __name__ == "__main__":
    main()
