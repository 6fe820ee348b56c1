"""MVG_ENGINE_SEQ (csrc/mv_seq_core.h): the reference's sequential sampler restated for one thread of control.
Chain-level parity with the UNMODIFIED reference (run_gibbs_cpp, saved states in tests/golden/reference_chains.npz) driven by
the same call-ordered Philox stream:

  * CPU (here): the same source compiled for the host (tests/seq_host_check.cpp, test scaffolding) visits the same states
    as the reference — table_of, dish_of of every kept sweep identical, hyperparameters bitwise equal, the same number of
    uniforms and normals consumed;
  * GPU (-m gpu): the device chain (mvg_seq_run through the C ABI) visits the same integer states; the hyperparameters
    agree to 1e-9 (the last bits of exp / log / cos differ between libm and the CUDA math library)."""
import ctypes as C
import subprocess
from pathlib import Path

import numpy as np
import pytest
from conftest import c1_data, reference_chain

ROOT = Path(__file__).resolve().parents[1]
OUT = ROOT / "tests" / "_build" / "libseqhost.so"


def _host_lib():
    OUT.parent.mkdir(exist_ok=True)
    cmd = ["g++", "-O2", "-std=c++17", "-fPIC", "-ffp-contract=off", "-shared", "-D__host__=", "-D__device__=",
           "-D__forceinline__=inline", f"-I{ROOT / 'multiview-clustering_b200' / 'csrc'}", "-o", str(OUT),
           str(ROOT / "tests" / "seq_host_check.cpp")]
    subprocess.run(cmd, check=True, capture_output=True, text=True)
    return C.CDLL(str(OUT))


def _data(n):
    views, truth = c1_data(n)
    return np.ascontiguousarray(np.stack([v.astype(np.float64) for v in views])), truth


def _compare(tr, tab, T, dish, hyp, d, exact_hypers):
    for s, ref in enumerate(tr):
        np.testing.assert_array_equal(tab[s], ref["table_of"], err_msg=f"table_of, kept state {s}")
        assert T[s] == ref["dish_of"].shape[1], (s, T[s], ref["dish_of"].shape)
        for v in range(d):
            np.testing.assert_array_equal(dish[s][v][:T[s]], ref["dish_of"][v], err_msg=f"dish_of view {v}, kept state {s}")
        got = np.concatenate([hyp[s][:3 * d], hyp[s][3 * d:]])
        want = np.concatenate([ref["alpha_v"], ref["sigma_v"], ref["tau_v"], [ref["alpha_global"], ref["sigma_global"]]])
        if exact_hypers:
            np.testing.assert_array_equal(got, want)
        else:
            np.testing.assert_allclose(got, want, rtol=1e-9)


@pytest.mark.parametrize("seed,n,M,burn,thin", [(1999, 500, 300, 100, 10), (7, 500, 400, 0, 40), (42, 200, 500, 250, 25)])
def test_sequential_core_follows_the_compiled_reference_state_for_state(seed, n, M, burn, thin):
    y, _ = _data(n)
    d = y.shape[0]
    tr, ref_calls = reference_chain(seed, n, M, burn, thin)
    S, t_cap, k_cap = len(tr), 1024, 2 * M + 64
    tab = np.zeros((S, n), np.int32); T = np.zeros(S, np.int32); dish = np.zeros((S, d, t_cap), np.int32)
    hyp = np.zeros((S, 3 * d + 2)); calls = C.c_ulonglong()
    L = _host_lib()
    rc = L.seq_host_run(n, d, y.ctypes.data_as(C.POINTER(C.c_double)), M, burn, thin, C.c_ulonglong(seed), t_cap, k_cap, S,
                        tab.ctypes.data_as(C.POINTER(C.c_int)), T.ctypes.data_as(C.POINTER(C.c_int)),
                        dish.ctypes.data_as(C.POINTER(C.c_int)), hyp.ctypes.data_as(C.POINTER(C.c_double)), C.byref(calls))
    assert rc == S, rc
    assert calls.value == ref_calls                      # the same number of uniforms and normals, in the same order
    _compare(tr, tab, T, [[dish[s, v] for v in range(d)] for s in range(S)], hyp, d, exact_hypers=True)


@pytest.mark.gpu
@pytest.mark.parametrize("seed,n,M,burn,thin", [(1999, 500, 300, 100, 10), (7, 500, 600, 0, 50)])
def test_sequential_engine_on_the_device_follows_the_reference(seed, n, M, burn, thin):
    import mvc_b200
    y, truth = _data(n)
    d = y.shape[0]
    tr, ref_calls = reference_chain(seed, n, M, burn, thin)
    res = mvc_b200.run_gibbs_seq([y[v] for v in range(d)], M, burn, thin, seed=seed)
    S = len(res["table_of"])
    assert S == len(tr) and res["stream_calls"] == ref_calls
    hyp = [np.concatenate([[res["alpha_v"][v][s] for v in range(d)], [res["sigma_v"][v][s] for v in range(d)],
                           [res["tau_v"][v][s] for v in range(d)], [res["alpha_global"][s], res["sigma_global"][s]]]) for s in range(S)]
    _compare(tr, res["table_of"], [len(res["dish_of"][s][0]) for s in range(S)], res["dish_of"], hyp, d, exact_hypers=False)
