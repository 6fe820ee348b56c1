"""mvc_b200 — thin ctypes binding of libmvg_b200.so (the C ABI in include/mvg.h).

This is a binding, not an implementation: every call goes to the CUDA library.  If the shared
library is missing, or there is no CUDA device, construction raises — there is no CPU path here
(the CPU restatement under oracle/ is test infrastructure and is never imported from this package).

``Sampler`` mirrors the reference's chain object-in-globals (multiview_state.h:21-45) and its entry
points: ``init_state_reference`` = initialize_state_from_data (multiview_gibbs.cpp:12-103),
``sweep`` = the loop body of gibbs_sampler (multiview_gibbs.cpp:157-202), ``run`` = gibbs_sampler +
save_state, ``run_gibbs`` = run_gibbs_cpp (multiview_gibbs.cpp:105-131, same keys in the result).
"""
from __future__ import annotations

import ctypes as C
from pathlib import Path

import numpy as np

_HERE = Path(__file__).resolve().parent
LIB_PATH = _HERE / "libmvg_b200.so"

ENGINE_AUTO, ENGINE_SIMT, ENGINE_TCGEN05, ENGINE_TCGEN05_FAST = 0, 1, 2, 3
COUNT_LIKELIHOODS = {"plugin": 0, "dirmult": 1}   # MVG_COUNT_PLUGIN / MVG_COUNT_DIRMULT
NEW_TABLE = -1

_i32p = C.POINTER(C.c_int32)
_f32p = C.POINTER(C.c_float)
_f64p = C.POINTER(C.c_double)
_u32p = C.POINTER(C.c_uint32)


class MvgError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"mvg error {code}: {msg}")
        self.code = code


class _Config(C.Structure):
    _fields_ = [
        ("abi_version", C.c_int32), ("device", C.c_int32),
        ("n_rows", C.c_int64), ("n_rows_global", C.c_int64), ("row_offset", C.c_int64),
        ("n_views", C.c_int32), ("cap", C.c_int32),
        ("seed", C.c_uint64), ("chain", C.c_uint32),
        ("engine", C.c_int32), ("debug_export", C.c_int32), ("rank", C.c_int32), ("world", C.c_int32),
        ("reserved", C.c_int32 * 5),
    ]


class _StateHost(C.Structure):
    _fields_ = [
        ("table_of", _i32p), ("n_t", _i32p), ("dish_of", _i32p), ("n_vk", _i32p), ("l_vk", _i32p),
        ("sum_y", _f64p), ("sum_y2", _f64p), ("alpha_v", _f64p), ("sigma_v", _f64p), ("tau_v", _f64p),
        ("alpha_sigma_global", _f64p), ("sweep", _u32p),
    ]


class _ParamsHost(C.Structure):
    _fields_ = [
        ("dish", _i32p), ("A", _f32p), ("C", _f32p), ("A1", _f32p), ("C1", _f32p), ("W", _f32p), ("W1", _f32p),
        ("lone", _i32p), ("AN", _f32p), ("CN", _f32p), ("WN", _f32p), ("LD", _f32p), ("LM", _f32p),
        ("LM1", _f32p), ("single", _i32p), ("LMN", _f32p), ("m", _f32p),
    ]


class _ScreenHost(C.Structure):
    _fields_ = [
        ("mode", C.c_int32), ("sweep", C.c_uint32), ("valid", C.c_uint32), ("ref_sweep", C.c_uint32),
        ("k", C.c_float * 7), ("n_eval", C.c_int32), ("tiles", _i32p), ("margin", _f32p), ("ref", _ParamsHost),
        ("ref_b", _f32p),
    ]


_lib = None


def lib():
    """Load libmvg_b200.so (raises FileNotFoundError with build instructions if it was not built)."""
    global _lib
    if _lib is None:
        if not LIB_PATH.exists():
            raise FileNotFoundError(
                f"{LIB_PATH} is missing: build it with `python multiview-clustering_b200/build.py` "
                "(nvcc, sm_100a).  There is no CPU fallback.")
        L = C.CDLL(str(LIB_PATH))
        H = C.c_void_p
        L.mvg_last_error.restype = C.c_char_p
        L.mvg_last_error.argtypes = [H]
        L.mvg_create.argtypes = [C.POINTER(_Config), C.POINTER(H)]
        L.mvg_destroy.argtypes = [H]
        L.mvg_upload_view_f32.argtypes = [H, C.c_int32, _f32p, C.c_int32]
        L.mvg_upload_view_f64.argtypes = [H, C.c_int32, _f64p, C.c_int32]
        L.mvg_attach_view_device_f32.argtypes = [H, C.c_int32, C.c_void_p, C.c_int32]
        L.mvg_upload_view_csr.argtypes = [H, C.c_int32, _i32p, _i32p, _f32p, C.c_int64, C.c_int32]
        L.mvg_set_count_beta.argtypes = [H, C.c_double]
        L.mvg_get_count_tables.argtypes = [H, C.c_int32, _f32p, _i32p, _i32p]
        L.mvg_set_count_likelihood.argtypes = [H, C.c_int32]
        L.mvg_get_count_den.argtypes = [H, C.c_int32, _f32p, _i32p]
        L.mvg_set_count_beta_prior.argtypes = [H, C.c_double, C.c_double, C.c_double]
        L.mvg_get_count_beta.argtypes = [H, _f64p]
        L.mvg_get_count_beta_step.argtypes = [H, _f64p, _i32p]
        L.mvg_set_count_beta_trace.argtypes = [H, _f64p]
        L.mvg_get_debug_loo.argtypes = [H, _f32p]
        L.mvg_init_state_reference.argtypes = [H]
        L.mvg_set_state.argtypes = [H, C.POINTER(_StateHost)]
        L.mvg_get_state.argtypes = [H, C.POINTER(_StateHost)]
        L.mvg_save_checkpoint.argtypes = [H, C.c_char_p]
        L.mvg_load_checkpoint.argtypes = [H, C.c_char_p]
        L.mvg_sweep.argtypes = [H, C.c_int32, C.c_int32]
        L.mvg_hyper_step.argtypes = [H]
        L.mvg_set_sweep_blocks.argtypes = [H, C.c_int32]
        L.mvg_set_draw_screen.argtypes = [H, C.c_int32]
        L.mvg_get_draw_screen_stats.argtypes = [H, C.POINTER(C.c_int32), C.POINTER(C.c_int64), C.POINTER(C.c_int64)]
        L.mvg_get_draw_screen_record.argtypes = [H, C.POINTER(_ScreenHost)]
        L.mvg_get_draw_rows.argtypes = [H, _i32p, _i32p, _u32p, _u32p]
        L.mvg_set_stats_mode.argtypes = [H, C.c_int32, C.c_int32]
        L.mvg_hyper_step_parts.argtypes = [H, C.c_int32]
        L.mvg_sync.argtypes = [H]
        L.mvg_run.argtypes = [H, C.c_int32, C.c_int32, C.c_int32, C.c_int32, _i32p, _i32p, _f64p, _f64p, _i32p]
        L.mvg_comm_attach.argtypes = [H, C.c_void_p]
        L.mvg_comm_handle.restype = C.c_void_p
        L.mvg_comm_handle.argtypes = [H]
        L.mvg_comm_unique_id.argtypes = [C.c_void_p]
        L.mvg_comm_init_rank.argtypes = [H, C.c_void_p]
        L.mvg_prepare.argtypes = [H]
        L.mvg_comm_p2p_export.argtypes = [H, C.c_void_p]
        L.mvg_comm_p2p_attach.argtypes = [H, C.c_void_p]
        L.mvg_comm_p2p_disable.argtypes = [H]
        L.mvg_comm_p2p_enable.argtypes = [H]
        L.mvg_clear_fault.argtypes = [H]
        L.mvg_get_params.argtypes = [H, C.POINTER(_ParamsHost)]
        L.mvg_get_debug_rows.argtypes = [H, _f32p, _f32p, _i32p]
        L.mvg_get_debug_lnew.argtypes = [H, _f32p]
        L.mvg_get_debug_births.argtypes = [H, _i32p, C.POINTER(C.c_int64), _f64p]
        L.mvg_get_debug_prof.argtypes = [H, C.POINTER(C.c_int64), C.c_int32]
        L.mvg_last_sweep_ms.argtypes = [H, _f32p]
        L.mvg_kernel_clock.argtypes = [H, C.c_int32, C.POINTER(C.c_double), C.POINTER(C.c_int64), C.POINTER(C.c_int64), C.c_int32]
        L.mvg_launch_count.restype = C.c_int64
        L.mvg_launch_count.argtypes = [H]
        L.mvg_log_likelihood.argtypes = [H, _f64p, _f64p]
        L.mvg_cluster_labels.argtypes = [H, _i32p]
        L.mvg_coclustering_begin.argtypes = [H, C.c_int32]
        L.mvg_coclustering_accumulate.argtypes = [H]
        L.mvg_coclustering_get.argtypes = [H, _u32p, _i32p]
        L.mvg_adjusted_rand_index.argtypes = [H, C.c_int32, _i32p, C.c_int32, _f64p, _i32p]
        L.mvg_profile_sweep.argtypes = [H, C.c_int32, _f32p]
        L.mvg_stream.restype = C.c_void_p
        L.mvg_stream.argtypes = [H]
        L.mvg_seq_run.argtypes = [C.c_int32, C.c_int32, C.c_int32, _f64p, C.c_int32, C.c_int32, C.c_int32, C.c_uint64, C.c_int32,
                                  C.c_int32, C.c_int32, _i32p, _i32p, _i32p, _f64p, _i32p, C.POINTER(C.c_uint64)]
        L.mvg_seq_last_error.restype = C.c_char_p
        L.mvg_philox4x32_10.argtypes = [_u32p, _u32p, _u32p]
        args = [C.c_uint64, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint64]
        L.mvg_philox_uniform_f32.restype = C.c_float
        L.mvg_philox_uniform_f32.argtypes = args
        L.mvg_philox_uniform_f64.restype = C.c_double
        L.mvg_philox_uniform_f64.argtypes = args
        L.mvg_philox_normal.restype = C.c_double
        L.mvg_philox_normal.argtypes = args
        _lib = L
    return _lib


def _p(a, typ):
    return a.ctypes.data_as(typ)


class Sampler:
    """One chain (or one row shard of a chain) on one B200."""

    def __init__(self, n_rows, dims, cap=64, seed=1999, chain=0, device=0, engine=ENGINE_AUTO,
                 debug_export=False, rank=0, world=1, row_offset=0, n_rows_global=None):
        self.L = lib()
        self.n_rows = int(n_rows)
        self.dims = [int(d) for d in dims]
        self.V = len(self.dims)
        self.cap = int(cap)
        self.Dsum = sum(self.dims)
        self.doff = np.concatenate([[0], np.cumsum(self.dims)[:-1]]).astype(int)
        cfg = _Config()
        cfg.abi_version = 2
        cfg.device = device
        cfg.n_rows = self.n_rows
        cfg.n_rows_global = self.n_rows if n_rows_global is None else int(n_rows_global)
        cfg.row_offset = int(row_offset)
        cfg.n_views = self.V
        cfg.cap = self.cap
        cfg.seed = seed
        cfg.chain = chain
        cfg.engine = engine
        cfg.debug_export = int(debug_export)
        cfg.rank = rank
        cfg.world = world
        self.h = C.c_void_p()
        rc = self.L.mvg_create(C.byref(cfg), C.byref(self.h))
        if rc != 0:
            raise MvgError(rc, self.L.mvg_last_error(None).decode())
        self._keep = []
        self.count_likelihood = "plugin"
        self.count_beta_prior = None

    # -- plumbing ---------------------------------------------------------------------------
    def _ck(self, rc):
        if rc != 0:
            raise MvgError(rc, self.L.mvg_last_error(self.h).decode())

    def close(self):
        if getattr(self, "h", None) is not None and self.h:
            self.L.mvg_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # -- data -------------------------------------------------------------------------------
    def upload_view(self, v, x):
        x = np.ascontiguousarray(x)
        if x.ndim == 1:
            x = x.reshape(-1, 1)
        assert x.shape == (self.n_rows, self.dims[v]), (x.shape, self.n_rows, self.dims[v])
        if x.dtype == np.float64:
            self._ck(self.L.mvg_upload_view_f64(self.h, v, _p(x, _f64p), x.shape[1]))
        else:
            x = np.ascontiguousarray(x, dtype=np.float32)
            self._ck(self.L.mvg_upload_view_f32(self.h, v, _p(x, _f32p), x.shape[1]))

    def upload_view_csr(self, v, rowptr, col, val, vocab):
        """Sparse count view v (declare it with dim 0 in ``dims``): CSR arrays over a vocabulary of ``vocab`` words."""
        assert self.dims[v] == 0, "declare count views with dim 0"
        rowptr = np.ascontiguousarray(rowptr, np.int32)
        col = np.ascontiguousarray(col, np.int32)
        val = np.ascontiguousarray(val, np.float32)
        assert rowptr.shape == (self.n_rows + 1,) and col.shape == val.shape
        self.vocab = getattr(self, "vocab", {})
        self.vocab[v] = int(vocab)
        self._ck(self.L.mvg_upload_view_csr(self.h, v, _p(rowptr, _i32p), _p(col, _i32p), _p(val, _f32p), len(col), int(vocab)))

    def set_count_beta(self, beta):
        self._ck(self.L.mvg_set_count_beta(self.h, float(beta)))

    def set_count_likelihood(self, model):
        """"plugin" (default: the plug-in multinomial) or "dirmult" (the collapsed Dirichlet-multinomial) for every
        count view; before the first state call."""
        if model not in COUNT_LIKELIHOODS:
            raise MvgError(-1, f"unknown count likelihood {model!r}: expected one of {sorted(COUNT_LIKELIHOODS)}")
        self._ck(self.L.mvg_set_count_likelihood(self.h, COUNT_LIKELIHOODS[model]))
        self.count_likelihood = model

    def set_count_beta_prior(self, shape, rate, step=0.3):
        """Learn beta of every "dirmult" count view: a Gamma(shape, rate) prior and one log-normal random-walk
        Metropolis-Hastings step of scale ``step`` per view per hyper step (step 0.3 as the tau step's proposal).  Before
        the first state call."""
        self._ck(self.L.mvg_set_count_beta_prior(self.h, float(shape), float(rate), float(step)))
        self.count_beta_prior = (float(shape), float(rate), float(step))

    def get_count_beta(self):
        """[V] float64: beta of every count view (0 for a dense view)."""
        out = np.empty(self.V, np.float64)
        self._ck(self.L.mvg_get_count_beta(self.h, _p(out, _f64p)))
        return out

    def get_count_beta_step(self):
        """(log A [V], accepted [V]) of the most recent beta step."""
        la = np.empty(self.V, np.float64)
        acc = np.empty(self.V, np.int32)
        self._ck(self.L.mvg_get_count_beta_step(self.h, _p(la, _f64p), _p(acc, _i32p)))
        return la, acc

    def get_count_den(self, v):
        """"dirmult" count view v: (den [n_max + 1, cap], n_max), den[n][t] = sum_{j<n} log2(W beta + C_k + j) of the dish
        table slot t serves, for the NEXT sweep."""
        n_max = C.c_int32(0)
        self._ck(self.L.mvg_get_count_den(self.h, v, None, C.byref(n_max)))
        den = np.empty((n_max.value + 1, self.cap), np.float32)
        self._ck(self.L.mvg_get_count_den(self.h, v, _p(den, _f32p), C.byref(n_max)))
        return den, n_max.value

    def get_count_tables(self, v):
        """(log2 theta, dish counts, table counts), each [vocab, cap], of count view v for the NEXT sweep.  Under the
        "dirmult" likelihood the first holds log2(beta + c) of the dish's word count c instead of log2 theta."""
        W = self.vocab[v]
        l2t = np.empty((W, self.cap), np.float32)
        cd = np.empty((W, self.cap), np.int32)
        ct = np.empty((W, self.cap), np.int32)
        self._ck(self.L.mvg_get_count_tables(self.h, v, _p(l2t, _f32p), _p(cd, _i32p), _p(ct, _i32p)))
        return l2t, cd, ct

    def get_debug_loo(self):
        out = np.empty((self.n_rows, self.V), np.float32)
        self._ck(self.L.mvg_get_debug_loo(self.h, _p(out, _f32p)))
        return out

    def attach_view_device(self, v, tensor):
        """Use a CUDA torch tensor (float32, contiguous, [n_rows, dim]) in place."""
        assert tensor.is_cuda and tensor.is_contiguous() and tuple(tensor.shape) == (self.n_rows, self.dims[v])
        self._keep.append(tensor)
        self._ck(self.L.mvg_attach_view_device_f32(self.h, v, C.c_void_p(tensor.data_ptr()), self.dims[v]))

    # -- peer-memory exchange (optional transport of the per-sweep packets; NCCL otherwise) -------
    def p2p_export(self):
        buf = C.create_string_buffer(64)
        self._ck(self.L.mvg_comm_p2p_export(self.h, buf))
        return buf.raw

    def p2p_attach(self, handles):
        """handles: the 64-byte exports of all ranks, in rank order."""
        blob = b"".join(handles)
        assert len(blob) == 64 * len(handles)
        self._ck(self.L.mvg_comm_p2p_attach(self.h, C.c_char_p(blob)))

    def p2p_disable(self):
        self._ck(self.L.mvg_comm_p2p_disable(self.h))

    # -- state ------------------------------------------------------------------------------
    def p2p_enable(self):
        self._ck(self.L.mvg_comm_p2p_enable(self.h))

    def clear_fault(self):
        self._ck(self.L.mvg_clear_fault(self.h))

    def init_state_reference(self):
        self._ck(self.L.mvg_init_state_reference(self.h))

    def set_state(self, table_of, dish_of, alpha_v, sigma_v, tau_v, alpha_g, sigma_g, sweep=0):
        s = _StateHost()
        a = {
            "table_of": np.ascontiguousarray(table_of, np.int32),
            "dish_of": np.ascontiguousarray(dish_of, np.int32).reshape(self.V, self.cap),
            "alpha_v": np.ascontiguousarray(alpha_v, np.float64),
            "sigma_v": np.ascontiguousarray(sigma_v, np.float64),
            "tau_v": np.ascontiguousarray(tau_v, np.float64),
            "alpha_sigma_global": np.array([alpha_g, sigma_g], np.float64),
            "sweep": np.array([sweep], np.uint32),
        }
        assert a["table_of"].shape == (self.n_rows,)
        s.table_of = _p(a["table_of"], _i32p)
        s.dish_of = _p(a["dish_of"], _i32p)
        s.alpha_v = _p(a["alpha_v"], _f64p)
        s.sigma_v = _p(a["sigma_v"], _f64p)
        s.tau_v = _p(a["tau_v"], _f64p)
        s.alpha_sigma_global = _p(a["alpha_sigma_global"], _f64p)
        s.sweep = _p(a["sweep"], _u32p)
        self._ck(self.L.mvg_set_state(self.h, C.byref(s)))

    def get_state(self, with_rows=True):
        V, cap = self.V, self.cap
        o = {
            "table_of": np.empty(self.n_rows, np.int32) if with_rows else None,
            "n_t": np.empty(cap, np.int32), "dish_of": np.empty((V, cap), np.int32),
            "n_vk": np.empty((V, cap), np.int32), "l_vk": np.empty((V, cap), np.int32),
            "sum_y": np.empty(cap * self.Dsum, np.float64), "sum_y2": np.empty((V, cap), np.float64),
            "alpha_v": np.empty(V, np.float64), "sigma_v": np.empty(V, np.float64), "tau_v": np.empty(V, np.float64),
            "alpha_sigma_global": np.empty(2, np.float64), "sweep": np.empty(1, np.uint32),
        }
        s = _StateHost()
        if with_rows:
            s.table_of = _p(o["table_of"], _i32p)
        s.n_t = _p(o["n_t"], _i32p)
        s.dish_of = _p(o["dish_of"], _i32p)
        s.n_vk = _p(o["n_vk"], _i32p)
        s.l_vk = _p(o["l_vk"], _i32p)
        s.sum_y = _p(o["sum_y"], _f64p)
        s.sum_y2 = _p(o["sum_y2"], _f64p)
        s.alpha_v = _p(o["alpha_v"], _f64p)
        s.sigma_v = _p(o["sigma_v"], _f64p)
        s.tau_v = _p(o["tau_v"], _f64p)
        s.alpha_sigma_global = _p(o["alpha_sigma_global"], _f64p)
        s.sweep = _p(o["sweep"], _u32p)
        self._ck(self.L.mvg_get_state(self.h, C.byref(s)))
        o["S1"] = [o["sum_y"][cap * self.doff[v]: cap * (self.doff[v] + self.dims[v])].reshape(cap, self.dims[v])
                   for v in range(V)]
        o["alpha_g"], o["sigma_g"] = float(o["alpha_sigma_global"][0]), float(o["alpha_sigma_global"][1])
        o["sweep"] = int(o["sweep"][0])
        return o

    def save_checkpoint(self, path):
        self._ck(self.L.mvg_save_checkpoint(self.h, str(path).encode()))

    def load_checkpoint(self, path):
        self._ck(self.L.mvg_load_checkpoint(self.h, str(path).encode()))

    # -- hot path ---------------------------------------------------------------------------
    def sweep(self, n=1, do_hyper=True):
        self._ck(self.L.mvg_sweep(self.h, int(n), int(do_hyper)))

    def set_stats_mode(self, incremental, rebuild_every=64):
        """incremental: only moved rows are re-read each sweep (running FP64 sums, full rebuild every rebuild_every sweeps)."""
        self._ck(self.L.mvg_set_stats_mode(self.h, 1 if incremental else 0, int(rebuild_every)))

    def set_sweep_blocks(self, blocks):
        """One sweep = `blocks` passes over row blocks with the statistics refreshed in between (1 = synchronous)."""
        self._ck(self.L.mvg_set_sweep_blocks(self.h, int(blocks)))

    def set_draw_screen(self, on):
        """Exact draw screening on the tensor-core engines (on by default): rows whose draw is provably their own table
        skip the likelihood.  The chain is the same either way."""
        self._ck(self.L.mvg_set_draw_screen(self.h, 1 if on else 0))

    def draw_screen_stats(self):
        """{'enabled', 'rows_screened', 'tiles_evaluated'} of the most recent draw (tiles of 128 rows)."""
        en, rows, tiles = C.c_int32(0), C.c_int64(0), C.c_int64(0)
        self._ck(self.L.mvg_get_draw_screen_stats(self.h, C.byref(en), C.byref(rows), C.byref(tiles)))
        return {"enabled": bool(en.value), "rows_screened": rows.value, "tiles_evaluated": tiles.value}

    def get_draw_screen_record(self):
        """What the most recent screened draw decided and left behind (mvg_get_draw_screen_record): 'mode' (0 off,
        1 refresh, 2 skip), 'sweep' it belongs to, 'valid', 'ref_sweep', 'k' [7], 'n_eval', 'tiles', 'margin' [n_rows],
        'ref' (dish, A, C, A1, C1, lone [V, cap]; LM, LM1 [cap]) and 'ref_b' [2, cap*Dsum] (mean_hi, mean_lo)."""
        V, cap = self.V, self.cap
        ref = {"dish": np.empty((V, cap), np.int32), "A": np.empty((V, cap), np.float32), "C": np.empty((V, cap), np.float32),
               "A1": np.empty((V, cap), np.float32), "C1": np.empty((V, cap), np.float32),
               "lone": np.empty((V, cap), np.int32), "LM": np.empty(cap, np.float32), "LM1": np.empty(cap, np.float32)}
        tiles = np.empty((self.n_rows + 127) // 128, np.int32)
        margin = np.empty(self.n_rows, np.float32)
        ref_b = np.empty((2, cap * self.Dsum), np.float32)
        s = _ScreenHost()
        for k, a in ref.items():
            setattr(s.ref, k, _p(a, _i32p if a.dtype == np.int32 else _f32p))
        s.tiles, s.margin, s.ref_b = _p(tiles, _i32p), _p(margin, _f32p), _p(ref_b, _f32p)
        self._ck(self.L.mvg_get_draw_screen_record(self.h, C.byref(s)))
        return {"mode": s.mode, "sweep": s.sweep, "valid": s.valid, "ref_sweep": s.ref_sweep,
                "k": np.array(s.k[:], np.float32), "n_eval": s.n_eval, "tiles": tiles, "margin": margin, "ref": ref,
                "ref_b": ref_b}

    def get_draw_rows(self):
        """The draw's per-row buffers as the most recent sweep left them (mvg_get_draw_rows): 'choice', 'table_cur'
        [n_rows] and 'birthmask', 'movedmask' [ceil(n_rows / 32)] (bit r of word w: row 32 w + r)."""
        n, w = self.n_rows, (self.n_rows + 31) // 32
        out = {"choice": np.empty(n, np.int32), "table_cur": np.empty(n, np.int32),
               "birthmask": np.empty(w, np.uint32), "movedmask": np.empty(w, np.uint32)}
        self._ck(self.L.mvg_get_draw_rows(self.h, _p(out["choice"], _i32p), _p(out["table_cur"], _i32p),
                                          _p(out["birthmask"], _u32p), _p(out["movedmask"], _u32p)))
        return out

    def hyper_step(self):
        self._ck(self.L.mvg_hyper_step(self.h))

    def sync(self):
        self._ck(self.L.mvg_sync(self.h))

    def last_sweep_ms(self):
        ms = C.c_float()
        self._ck(self.L.mvg_last_sweep_ms(self.h, C.byref(ms)))
        return ms.value

    def profile_sweep(self, do_hyper=True):
        ms = (C.c_float * 6)()
        self._ck(self.L.mvg_profile_sweep(self.h, int(do_hyper), ms))
        return dict(zip(["draw", "pack", "stats", "reduce", "finalize", "collective"], list(ms)))

    def kernel_clock(self, which=0, reset=False):
        """(total ms, launches) of the in-kernel wall clock: 0 = tensor-core draw kernel, 1 = finalize."""
        ms, n, last = C.c_double(0.0), C.c_int64(0), (C.c_int64 * 3)()
        self._ck(self.L.mvg_kernel_clock(self.h, int(which), C.byref(ms), C.byref(n), last, int(reset)))
        self.kernel_clock_last = list(last)     # ns: start, end of the latest launch; end of the one before
        return ms.value, n.value

    def launch_count(self):
        return int(self.L.mvg_launch_count(self.h))

    def run(self, M, burn_in, thin):
        """gibbs_sampler(M, burn_in, thin): returns the saved trace (multiview_gibbs.cpp:134-212)."""
        n_saved_max = max(0, (M - burn_in + thin - 1) // thin) if M > burn_in else 0
        tab = np.empty((max(n_saved_max, 1), self.n_rows), np.int32)
        dish = np.empty((max(n_saved_max, 1), self.V, self.cap), np.int32)
        hyp = np.empty((max(n_saved_max, 1), 3 * self.V + 2), np.float64)
        ll = np.zeros(max(n_saved_max, 1), np.float64)
        ns = C.c_int32(0)
        beta = np.empty((max(n_saved_max, 1), self.V), np.float64) if self.count_beta_prior else None
        if beta is not None:
            self._ck(self.L.mvg_set_count_beta_trace(self.h, _p(beta, _f64p)))
        # the log-likelihood kernel covers the Gaussian views and the Dirichlet-multinomial count views
        dense = all(d > 0 for d in self.dims) or self.count_likelihood == "dirmult"
        self._ck(self.L.mvg_run(self.h, M, burn_in, thin, n_saved_max, _p(tab, _i32p), _p(dish, _i32p),
                                _p(hyp, _f64p), _p(ll, _f64p) if dense else None, C.byref(ns)))
        if beta is not None:
            self._ck(self.L.mvg_set_count_beta_trace(self.h, None))
        S = ns.value
        out = {"table_of": tab[:S], "dish_of": dish[:S], "hypers": hyp[:S], "loglik": ll[:S] if dense else ll[:0]}
        if beta is not None:
            out["count_beta"] = beta[:S]
        return out

    # -- multi-GPU ----------------------------------------------------------------------------
    @staticmethod
    def nccl_unique_id() -> bytes:
        buf = C.create_string_buffer(128)
        rc = lib().mvg_comm_unique_id(buf)
        if rc != 0:
            raise MvgError(rc, lib().mvg_last_error(None).decode())
        return buf.raw

    def comm_init_rank(self, unique_id: bytes):
        buf = C.create_string_buffer(unique_id, 128)
        self._ck(self.L.mvg_comm_init_rank(self.h, buf))

    def comm_handle(self):
        """The NCCL communicator of this handle (an integer address) for comm_attach on another handle."""
        return self.L.mvg_comm_handle(self.h)

    def comm_attach(self, comm):
        self._ck(self.L.mvg_comm_attach(self.h, C.c_void_p(comm)))

    # -- posterior summaries ------------------------------------------------------------------
    def log_likelihood(self):
        """(total, per view): log marginal likelihood of the data given the current partition."""
        tot = C.c_double()
        pv = np.empty(self.V, np.float64)
        self._ck(self.L.mvg_log_likelihood(self.h, C.byref(tot), _p(pv, _f64p)))
        return tot.value, pv

    def cluster_labels(self):
        """[V, n_rows] dish of every customer in every view (get_final_clusters, New_Simulation.R:135-149)."""
        out = np.empty((self.V, self.n_rows), np.int32)
        self._ck(self.L.mvg_cluster_labels(self.h, _p(out, _i32p)))
        return out

    def coclustering_begin(self, view=-1):
        self._ck(self.L.mvg_coclustering_begin(self.h, int(view)))

    def coclustering_accumulate(self):
        self._ck(self.L.mvg_coclustering_accumulate(self.h))

    def coclustering_get(self):
        """(counts [n, n] uint32, number of accumulated states)."""
        out = np.empty((self.n_rows, self.n_rows), np.uint32)
        ns = C.c_int32(0)
        self._ck(self.L.mvg_coclustering_get(self.h, _p(out, _u32p), C.byref(ns)))
        return out, ns.value

    def adjusted_rand_index(self, view, truth, n_classes=None):
        """(ARI, contingency [cap, n_classes]) of the current clustering of `view` (-1: tables) vs truth."""
        truth = np.ascontiguousarray(truth, np.int32)
        n_classes = int(truth.max()) + 1 if n_classes is None else int(n_classes)
        ari = C.c_double()
        tab = np.empty((self.cap, n_classes), np.int32)
        self._ck(self.L.mvg_adjusted_rand_index(self.h, int(view), _p(truth, _i32p), n_classes, C.byref(ari), _p(tab, _i32p)))
        return ari.value, tab

    # -- inspection ---------------------------------------------------------------------------
    def get_params(self):
        V, cap = self.V, self.cap
        P = {
            "dish": np.empty((V, cap), np.int32), "A": np.empty((V, cap), np.float32), "C": np.empty((V, cap), np.float32),
            "A1": np.empty((V, cap), np.float32), "C1": np.empty((V, cap), np.float32), "W": np.empty((V, cap), np.float32),
            "W1": np.empty((V, cap), np.float32), "lone": np.empty((V, cap), np.int32), "AN": np.empty(V, np.float32),
            "CN": np.empty(V, np.float32), "WN": np.empty((V, 2), np.float32), "LD": np.empty((V, 2), np.float32),
            "LM": np.empty(cap, np.float32), "LM1": np.empty(cap, np.float32), "single": np.empty(cap, np.int32),
            "LMN": np.empty(2, np.float32),
        }
        mflat = np.empty(cap * self.Dsum, np.float32)
        s = _ParamsHost()
        for k, a in P.items():
            setattr(s, k, _p(a, _i32p if a.dtype == np.int32 else _f32p))
        s.m = _p(mflat, _f32p)
        self._ck(self.L.mvg_get_params(self.h, C.byref(s)))
        P["m"] = [mflat[cap * self.doff[v]: cap * (self.doff[v] + self.dims[v])].reshape(cap, self.dims[v]).copy()
                  for v in range(V)]
        return P

    def get_debug_rows(self):
        acc = np.empty((self.n_rows, self.V, self.cap), np.float32)
        xx = np.empty((self.n_rows, self.V), np.float32)
        ch = np.empty(self.n_rows, np.int32)
        self._ck(self.L.mvg_get_debug_rows(self.h, _p(acc, _f32p), _p(xx, _f32p), _p(ch, _i32p)))
        return acc, xx, ch

    def get_debug_lnew(self):
        out = np.empty(self.n_rows, np.float32)
        self._ck(self.L.mvg_get_debug_lnew(self.h, _p(out, _f32p)))
        return out

    def get_debug_prof(self, n_ctas=148):
        """Role wait counters of the last tcgen05 draw (needs debug_export & 2): [n_ctas, 16] cycles."""
        out = np.zeros((n_ctas, 16), np.int64)
        self._ck(self.L.mvg_get_debug_prof(self.h, _p(out, C.POINTER(C.c_int64)), n_ctas))
        return out

    def get_debug_births(self):
        ns = C.c_int32(0)
        rows = np.empty(self.cap, np.int64)
        w = np.empty((self.cap, self.V, self.cap + 1), np.float64)
        self._ck(self.L.mvg_get_debug_births(self.h, C.byref(ns), _p(rows, C.POINTER(C.c_int64)), _p(w, _f64p)))
        return ns.value, rows[:ns.value].copy(), w[:ns.value].copy()


def _as_csr(v):
    """A sparse count view as (rowptr, col, val, vocab): a dict with those keys, or a scipy.sparse matrix."""
    if isinstance(v, dict):
        return (np.asarray(v["rowptr"], np.int32), np.asarray(v["col"], np.int32), np.asarray(v["val"], np.float32), int(v["vocab"]))
    if hasattr(v, "tocsr"):
        m = v.tocsr()
        m.sum_duplicates()
        m.sort_indices()
        return (m.indptr.astype(np.int32), m.indices.astype(np.int32), m.data.astype(np.float32), int(m.shape[1]))
    return None


def run_gibbs(data_views, M, burn_in, thin, cap=64, seed=1999, device=0, engine=ENGINE_AUTO, start=None, blocks=1,
              count_likelihood="plugin", count_beta_prior=None):
    """run_gibbs_cpp(data_views, M, burn_in, thin) on the GPU (multiview_gibbs.cpp:105-131).

    ``data_views`` is a list of per-view arrays (vectors as in New_Simulation.R:105-111, or [n, D]
    matrices); a sparse count view (the X_body / X_title / X_topics of dataset/reuters/data pre-process.R) is a
    scipy.sparse matrix or a dict {"rowptr", "col", "val", "vocab"}.  ``start`` = (table_of, dish_of) replaces the
    reference's random T = 4 / K = 2 start.  Returns a dict with the reference's eight keys; ``table_of`` is
    0-based, ``dish_of`` is indexed [saved][view][table slot] with -1 for a free slot.  ``count_likelihood`` is
    "plugin" or "dirmult" (Sampler.set_count_likelihood).  ``count_beta_prior`` = (shape, rate) or (shape, rate, step)
    learns beta of every "dirmult" count view (Sampler.set_count_beta_prior); the result then has "count_beta" [S][V].
    """
    csr = [_as_csr(v) for v in data_views]
    views = [None if c is not None else np.asarray(v, dtype=np.float64).reshape(len(v), -1) for v, c in zip(data_views, csr)]
    n = len(csr[0][0]) - 1 if csr[0] is not None else views[0].shape[0]
    s = Sampler(n, [0 if x is None else x.shape[1] for x in views], cap=cap, seed=seed, device=device, engine=engine)
    try:
        for v, x in enumerate(views):
            if x is None:
                s.upload_view_csr(v, *csr[v])
            else:
                s.upload_view(v, x)
        if blocks > 1:
            s.set_sweep_blocks(blocks)
        if count_likelihood != "plugin":
            s.set_count_likelihood(count_likelihood)
        if count_beta_prior is not None:
            s.set_count_beta_prior(*count_beta_prior)
        if start is None:
            s.init_state_reference()
        else:
            V = len(views)
            s.set_state(start[0], start[1], [1.0] * V, [0.5] * V, [1.0] * V, 1.0, 0.6)
        tr = s.run(M, burn_in, thin)
    finally:
        s.close()
    V = len(views)
    hyp = tr["hypers"]
    out = {
        "table_of": [t for t in tr["table_of"]],
        "dish_of": [[d[v] for v in range(V)] for d in tr["dish_of"]],
        "loglik": list(tr["loglik"]),                   # the reference declares it and never fills it (multiview_state.h:38)
        "alpha_v": [hyp[:, v] for v in range(V)],
        "sigma_v": [hyp[:, V + v] for v in range(V)],
        "tau_v": [hyp[:, 2 * V + v] for v in range(V)],
        "alpha_global": hyp[:, 3 * V],
        "sigma_global": hyp[:, 3 * V + 1],
    }
    if "count_beta" in tr:
        out["count_beta"] = tr["count_beta"]
    return out


def run_gibbs_seq(data_views, M, burn_in, thin, seed=1999, device=0, t_cap=1024, k_cap=None):
    """MVG_ENGINE_SEQ: run_gibbs_cpp of the reference, rule for rule, on the device (scalar views; one thread per chain).
    Returns the reference's eight keys; table_of is 0-based and dense, dish_of[s][v] has one entry per live table."""
    y = np.ascontiguousarray(np.stack([np.asarray(v, np.float64).reshape(-1) for v in data_views]))
    d, n = y.shape
    S = max(0, (M - burn_in + thin - 1) // thin) if M > burn_in else 0
    k_cap = int(k_cap or (2 * M + 64))
    tab = np.zeros((max(S, 1), n), np.int32)
    T = np.zeros(max(S, 1), np.int32)
    dish = np.zeros((max(S, 1), d, t_cap), np.int32)
    hyp = np.zeros((max(S, 1), 3 * d + 2), np.float64)
    ns, calls = C.c_int32(0), C.c_uint64(0)
    L = lib()
    rc = L.mvg_seq_run(device, n, d, _p(y, _f64p), M, burn_in, thin, seed, t_cap, k_cap, S, _p(tab, _i32p), _p(T, _i32p),
                       _p(dish, _i32p), _p(hyp, _f64p), C.byref(ns), C.byref(calls))
    if rc != 0:
        raise MvgError(rc, L.mvg_seq_last_error().decode())
    S = ns.value
    return {"table_of": [tab[s] for s in range(S)], "dish_of": [[dish[s, v, :T[s]] for v in range(d)] for s in range(S)],
            "loglik": [], "alpha_v": [hyp[:S, v] for v in range(d)], "sigma_v": [hyp[:S, d + v] for v in range(d)],
            "tau_v": [hyp[:S, 2 * d + v] for v in range(d)], "alpha_global": hyp[:S, 3 * d], "sigma_global": hyp[:S, 3 * d + 1],
            "stream_calls": int(calls.value)}
