"""oracle/pydirmult.py — TEST INFRASTRUCTURE, not product code.

ctypes access to oracle/mv_oracle_dm.c, the CPU restatement of the Dirichlet-multinomial count likelihood
(MVG_COUNT_DIRMULT): ``DirmultState`` is an ``pyoracle.OracleState`` whose count views are scored by the collapsed
Dirichlet-multinomial conditional in the draw, the reseat (births) and the marginal likelihood, and
``stageA_counts_dm_f32`` is the FP32 mirror of the device's stage A.  The library (mv_oracle_dm.c linked with
mv_oracle.c) is built into oracle/_ref/ by ``build()``; only tests/ may load it.
"""
from __future__ import annotations

import ctypes as C
import subprocess

import numpy as np

import pyoracle
from pyoracle import ORACLE_DIR, REF_DIR, _f32p, _f64p, _i32p, _ptr

LIB = REF_DIR / "libmvoracle_dm.so"
_SRCS = [ORACLE_DIR / "mv_oracle_dm.c", ORACLE_DIR / "mv_oracle.c"]
# the flags of oracle/Makefile: the FP32 mirror must not have a*b+c fused behind its back
_CFLAGS = ["-O2", "-fPIC", "-std=gnu11", "-ffp-contract=off", "-fno-fast-math", "-Wall", "-Wextra", "-fopenmp", "-shared"]


def build() -> None:
    REF_DIR.mkdir(exist_ok=True)
    subprocess.run(["gcc", *_CFLAGS, "-o", str(LIB), *map(str, _SRCS), "-lm"], check=True)


_lib = None


def lib():
    global _lib
    if _lib is None:
        if not LIB.exists() or any(s.stat().st_mtime > LIB.stat().st_mtime for s in _SRCS):
            build()
        L = C.CDLL(str(LIB))
        S = C.POINTER(pyoracle._MvoState)
        L.mvod_counts_log_f_vk.restype = C.c_double
        L.mvod_counts_log_f_vk.argtypes = [S, C.c_int, C.c_int, C.c_int, C.c_int]
        L.mvod_counts_log_f_new.restype = C.c_double
        L.mvod_counts_log_f_new.argtypes = [S, C.c_int, C.c_int]
        L.mvod_log_marginal_counts.restype = C.c_double
        L.mvod_log_marginal_counts.argtypes = [S, C.c_int]
        L.mvod_row_logweights.argtypes = [S, C.c_int, _f64p, _f64p]
        L.mvod_draw_rows.argtypes = [S, _i32p, C.c_int]
        L.mvod_reseat.argtypes = [S, _i32p, _i32p, _i32p, _f64p]
        L.mvod_stageA_counts_f32.argtypes = [_i32p, _f32p, C.c_int, _f32p, _i32p, _f32p, C.c_int, C.c_int, C.c_float,
                                             C.c_float, _f32p, _f32p]
        _lib = L
    return _lib


class DirmultState(pyoracle.OracleState):
    """An OracleState whose count views follow the Dirichlet-multinomial model (dense views as in OracleState)."""

    def counts_log_f_vk(self, v, k, i, loo=False):
        """Natural log f of row i of count view v under dish k (loo: row i removed from the dish first)."""
        return lib().mvod_counts_log_f_vk(self.ref(), int(v), int(k), int(i), int(loo))

    def counts_log_f_new(self, v, i):
        return lib().mvod_counts_log_f_new(self.ref(), int(v), int(i))

    def log_marginal_counts(self, v):
        """Collapsed log marginal of the partition in count view v (no multinomial coefficients)."""
        return lib().mvod_log_marginal_counts(self.ref(), int(v))

    def row_logweights(self, i, want_L=False):
        lw = np.empty(self.cap + 1, dtype=np.float64)
        L = np.empty((self.V, self.cap + 1), dtype=np.float64) if want_L else None
        lib().mvod_row_logweights(self.ref(), int(i), _ptr(lw, _f64p), _ptr(L, _f64p) if want_L else None)
        return (lw, L) if want_L else lw

    def draw_rows(self, threads=1):
        choice = np.empty(self.n, dtype=np.int32)
        lib().mvod_draw_rows(self.ref(), _ptr(choice, _i32p), threads)
        return choice

    def reseat(self, choice, want_births=False):
        choice = np.ascontiguousarray(choice, dtype=np.int32)
        n_seated = C.c_int32(0)
        rows = np.full(self.cap, -1, dtype=np.int32)
        w = np.zeros((self.cap, self.V, self.cap + 1), dtype=np.float64)
        rc = lib().mvod_reseat(self.ref(), _ptr(choice, _i32p), C.byref(n_seated), _ptr(rows, _i32p), _ptr(w, _f64p))
        if rc:
            raise ValueError(f"mvod_reseat rc={rc}")
        ns = n_seated.value
        return (ns, rows[:ns].copy(), w[:ns].copy()) if want_births else ns

    def make_params(self):
        """The FP32 parameter block: as OracleState's, with AN = 1, CN = 0 for the count views (their draw reads
        -log2 f_new itself where the plug-in reads the token total)."""
        P = super().make_params()
        P["AN"][self.kind == 1] = 1.0
        P["CN"][self.kind == 1] = 0.0
        return P


def stageA_counts_dm_f32(col, val, l2c, cdt, den, t0, beta, wbeta_plus_ctot):
    """Stage A of one CSR row against the device's tables l2c / cdt ([vocab, cap]) and den ([n_max + 1, cap]);
    returns (acc [cap], leave-one-out value)."""
    col = np.ascontiguousarray(col, np.int32)
    val = np.ascontiguousarray(val, np.float32)
    l2c = np.ascontiguousarray(l2c, np.float32)
    cdt = np.ascontiguousarray(cdt, np.int32)
    den = np.ascontiguousarray(den, np.float32)
    cap = l2c.shape[1]
    acc = np.empty(cap, np.float32)
    loo = C.c_float()
    lib().mvod_stageA_counts_f32(_ptr(col, _i32p), _ptr(val, _f32p), len(col), _ptr(l2c, _f32p), _ptr(cdt, _i32p),
                                 _ptr(den, _f32p), cap, int(t0), C.c_float(float(beta)), C.c_float(float(wbeta_plus_ctot)),
                                 _ptr(acc, _f32p), C.byref(loo))
    return acc, np.float32(loo.value)
