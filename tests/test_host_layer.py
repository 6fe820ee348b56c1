"""The host layer (multiview-clustering_b200/host): the reference's C++ interface — run_gibbs_cpp,
gibbs_sampler, update_hyperparameters, struct ViewState and the mirrored globals — over the C ABI.
R is not installed in this image, so the sources are compiled against the stand-in Rcpp.h of
oracle/refshim and driven through the C hooks of tests/host_shim.cpp."""
import ctypes as C
import subprocess
from pathlib import Path

import numpy as np
import pytest
from conftest import c1_data, reference_chain

ROOT = Path(__file__).resolve().parents[1]
HOST = ROOT / "multiview-clustering_b200" / "host"
OUT = ROOT / "tests" / "_build" / "libmvhost_test.so"


def build_host():
    OUT.parent.mkdir(exist_ok=True)
    srcs = [str(HOST / f) for f in ("multiview_gibbs.cpp", "multiview_hyper.cpp", "multiview_state.cpp", "multiview_utils.cpp")]
    cmd = ["g++", "-O2", "-fPIC", "-std=c++17", "-Wall", "-DMVHOST_WITH_RCPP", f"-I{ROOT / 'oracle' / 'refshim'}", f"-I{HOST}",
           f"-I{ROOT / 'tests'}", "-shared", "-o", str(OUT), *srcs, str(ROOT / "tests" / "host_shim.cpp"),
           str(ROOT / "tests" / "host_shim_utils.cpp"),
           f"-L{ROOT / 'multiview-clustering_b200' / 'mvc_b200'}", "-lmvg_b200",
           f"-Wl,-rpath,{ROOT / 'multiview-clustering_b200' / 'mvc_b200'}"]
    subprocess.run(cmd, check=True, capture_output=True, text=True)
    return C.CDLL(str(OUT))


def test_host_layer_compiles_and_keeps_the_reference_names():
    """Every name of multiview_gibbs.h / multiview_hyper.h / multiview_state.h resolves in the built library."""
    import mvc_b200
    mvc_b200.lib()
    build_host()
    syms = subprocess.run(["nm", "-DC", str(OUT)], capture_output=True, text=True, check=True).stdout
    for name in ["run_gibbs_cpp(Rcpp::List const&, int, int, int)", "gibbs_sampler(int, int, int)", "update_hyperparameters()",
                 "update_tau_v_MH()", "log_EPPF(int, double, double)", "log_prior_alpha(double)", "log_prior_sigma(double)",
                 "log_posterior_given_tau(int, double)", "propose_tau(double)", "initialize_hyperparameters()",
                 "compute_log_likelihood()", "compute_f_vk(int, int, int)", "compute_f_vk_new(int, int)",
                 "compute_table_probs_with_cache(int, std::vector<double", "remove_customer(int)",
                 "add_customer_to_existing_table(int, int)", "create_empty_table()", "add_customer_to_new_table(int, int)",
                 "sample_dish_for_new_table(int, int)", "assign_dishes_new_table(int, int)", "save_state()", "uniform01()",
                 "rnorm_scalar(double, double)", "ensure_global_variances_calculated()", "saved_loglik", "table_of", "dish_of", "views", "saved_table_of", "alpha_global", "sigma_global"]:
        assert name in syms, name


def test_host_philox_stream_is_the_c_abi_stream():
    import mvc_b200
    L = build_host()
    L.host_uniform01.restype = C.c_double
    M = mvc_b200.lib()
    for skip in (0, 3, 17):
        u = L.host_uniform01(C.c_uint(7), skip)
        assert u == M.mvg_philox_uniform_f64(7, 0, 6, 0, 0, skip)


@pytest.mark.gpu
def test_run_gibbs_cpp_through_the_host_layer_equals_the_c_abi_chain():
    """run_gibbs_cpp (host C++) and the ctypes binding drive the same device chain: same saved partitions."""
    import mvc_b200
    views, _ = c1_data(400)
    y = np.ascontiguousarray(np.stack([v.astype(np.float64) for v in views]))
    L = build_host()
    L.host_last_error.restype = C.c_char_p
    S = L.host_run(400, 2, y.ctypes.data_as(C.POINTER(C.c_double)), 60, 40, 5, 32, C.c_ulonglong(1999))
    assert S == 4, L.host_last_error()
    ref = mvc_b200.run_gibbs([y[0], y[1]], 60, 40, 5, cap=32, seed=1999)
    for s in range(S):
        T = L.host_saved_T(s)
        tab = np.empty(400, np.int32)
        L.host_saved_table_of(s, tab.ctypes.data_as(C.POINTER(C.c_int)))
        rt = np.asarray(ref["table_of"][s])
        live = np.unique(rt)                                    # slots -> dense labels in slot order
        assert T == len(live)
        np.testing.assert_array_equal(tab, np.searchsorted(live, rt))
        for v in range(2):
            dish = np.empty(T, np.int32)
            L.host_saved_dish_of(s, v, dish.ctypes.data_as(C.POINTER(C.c_int)))
            rd = np.asarray(ref["dish_of"][s][v])[live]
            np.testing.assert_array_equal(dish, np.searchsorted(np.unique(rd), rd))
        hyp = np.empty(8)
        L.host_saved_hypers(s, 2, hyp.ctypes.data_as(C.POINTER(C.c_double)))
        np.testing.assert_array_equal(hyp[:2], [ref["alpha_v"][v][s] for v in range(2)])
        np.testing.assert_array_equal(hyp[4:6], [ref["tau_v"][v][s] for v in range(2)])
        assert hyp[6] == ref["alpha_global"][s] and hyp[7] == ref["sigma_global"][s]
    L.host_compute_log_likelihood.restype = C.c_double
    L.host_log_EPPF.restype = C.c_double
    assert np.isfinite(L.host_compute_log_likelihood())
    assert np.isfinite(L.host_log_EPPF(0, C.c_double(1.0), C.c_double(0.5)))


@pytest.mark.gpu
def test_utils_inspectors_on_the_mirrored_state_equal_the_fp64_restatement(oracle):
    """multiview_utils.h over the device chain: compute_table_probs_with_cache / compute_f_vk on the state mirrored from
    the GPU give the weights of the FP64 restatement (oracle/mv_oracle.c, whose row weights test_oracle_vs_reference pins
    to vectors from the compiled reference at 2e-11) for the same state; saved_loglik is filled on every kept sweep; the
    single-customer mutators raise."""
    views, _ = c1_data(300)
    y = np.ascontiguousarray(np.stack([v.astype(np.float64) for v in views]))
    L = build_host()
    L.host_last_error.restype = C.c_char_p
    S = L.host_run(300, 2, y.ctypes.data_as(C.POINTER(C.c_double)), 40, 30, 5, 32, C.c_ulonglong(7))
    assert S == 2, L.host_last_error()
    ll = np.empty(8)
    assert L.host_saved_loglik(ll.ctypes.data_as(C.POINTER(C.c_double))) == S and np.all(np.isfinite(ll[:S])) and np.all(ll[:S] < 0)
    tab = np.empty(300, np.int32)
    T = L.host_final_table_of(tab.ctypes.data_as(C.POINTER(C.c_int)))
    dish = np.empty((2, T), np.int32)
    for v in range(2):
        row = np.empty(T, np.int32)
        L.host_final_dish_of(v, row.ctypes.data_as(C.POINTER(C.c_int)))
        dish[v] = row
    hyp = np.empty(8)
    L.host_final_hypers(hyp.ctypes.data_as(C.POINTER(C.c_double)))
    cap = max(T, int(dish.max()) + 1) + 1                       # one slot free for a new table
    dish_cap = np.pad(dish, ((0, 0), (0, cap - T)), constant_values=-1)
    L.host_f_vk.restype = C.c_double
    L.host_f_vk_new.restype = C.c_double
    for i in (0, 17, 150, 299):
        # the weights of customer i while it is seated = the oracle's leave-one-out weights of a copy of row i at its table
        o = oracle.OracleState([np.append(y[v], y[v][i]).astype(np.float32) for v in range(2)], cap)
        o.alpha_v[:], o.sigma_v[:], o.tau_v[:] = hyp[0:2], hyp[2:4], hyp[4:6]
        o.alpha_g, o.sigma_g = hyp[6], hyp[7]
        o.set_assignment(np.append(tab, tab[i]), dish_cap)
        w = np.exp(o.row_logweights(len(tab)))
        pe, pn = w[:T], w[cap]
        hpe, hpn = np.zeros(T), C.c_double()
        assert L.host_table_probs(i, hpe.ctypes.data_as(C.POINTER(C.c_double)), C.byref(hpn)) == T, L.host_last_error()
        # the mirror holds the device's FP32-tree sums: the statistics agree to 1e-5, so do the weights
        np.testing.assert_allclose(hpe, pe, rtol=2e-4, atol=1e-300)
        np.testing.assert_allclose(hpn.value, pn, rtol=2e-4)
    for which in range(4):
        assert L.host_mutator_raises(which) == 1 and b"not supported on the device chain" in L.host_last_error()


@pytest.mark.gpu
def test_run_gibbs_cpp_sequential_engine_equals_the_compiled_reference():
    """mvhost::sequential = true: run_gibbs_cpp (host C++, the reference's signature) on MVG_ENGINE_SEQ returns the partitions
    the UNMODIFIED reference returns for the same data and seed — chain-level integer equality through the host layer."""
    views, _ = c1_data(300)
    y = np.ascontiguousarray(np.stack([v.astype(np.float64) for v in views]))
    L = build_host()
    L.host_last_error.restype = C.c_char_p
    S = L.host_run_seq(300, 2, y.ctypes.data_as(C.POINTER(C.c_double)), 200, 100, 20, C.c_ulonglong(11))
    tr, _ = reference_chain(11, 300, 200, 100, 20)
    assert S == len(tr) == 5, L.host_last_error()
    for s in range(S):
        tab = np.empty(300, np.int32)
        L.host_saved_table_of(s, tab.ctypes.data_as(C.POINTER(C.c_int)))
        np.testing.assert_array_equal(tab, tr[s]["table_of"])
        T = L.host_saved_T(s)
        assert T == tr[s]["dish_of"].shape[1]
        for v in range(2):
            dish = np.empty(T, np.int32)
            L.host_saved_dish_of(s, v, dish.ctypes.data_as(C.POINTER(C.c_int)))
            np.testing.assert_array_equal(dish, tr[s]["dish_of"][v])


@pytest.mark.gpu
def test_run_gibbs_cpp_accepts_matrices_and_dgCMatrix(oracle):
    """data_views may hold what dataset/reuters/data pre-process.R builds: a numeric matrix (column-major, n x D), a
    Matrix::dgCMatrix of counts (compressed COLUMNS) and a plain vector.  run_gibbs_cpp converts them (row-major dense,
    CSR) and the chain equals the ctypes chain on the same views."""
    import mvc_b200
    from conftest import make_count_view
    rng = np.random.default_rng(4)
    n, D, W, k = 300, 4, 60, 4
    z = rng.integers(0, k, n)
    dense = (rng.normal(0, 2, (k, D))[z] + rng.normal(0, 1, (n, D)))
    cv = make_count_view(n, W, z, k, seed=2, mean_len=12)
    vec = rng.normal(0, 2, k)[z] + rng.normal(0, 1, n)
    import scipy.sparse as sp
    csr = sp.csr_matrix((cv["val"].astype(np.float64), cv["col"], cv["rowptr"]), shape=(n, W))
    csc = csr.tocsc()
    colmajor = np.ascontiguousarray(dense.T).ravel()              # R stores matrices column-major
    L = build_host()
    L.host_last_error.restype = C.c_char_p
    pd, pi = C.POINTER(C.c_double), C.POINTER(C.c_int)
    ci, cp, cx = csc.indices.astype(np.int32), csc.indptr.astype(np.int32), csc.data.astype(np.float64)
    S = L.host_run_mixed(n, D, colmajor.ctypes.data_as(pd), W, int(csc.nnz), ci.ctypes.data_as(pi), cp.ctypes.data_as(pi),
                         cx.ctypes.data_as(pd), np.ascontiguousarray(vec).ctypes.data_as(pd), 30, 20, 5, 32, C.c_ulonglong(77))
    assert S == 2, L.host_last_error()
    ref = mvc_b200.run_gibbs([dense, cv, vec], 30, 20, 5, cap=32, seed=77)
    for s in range(S):
        tab = np.empty(n, np.int32)
        L.host_saved_table_of(s, tab.ctypes.data_as(pi))
        rt = np.asarray(ref["table_of"][s])
        np.testing.assert_array_equal(tab, np.searchsorted(np.unique(rt), rt))
