"""pytest configuration: the `gpu` marker, import paths, shared synthetic data."""
import sys
from pathlib import Path

import numpy as np
import pytest

ROOT = Path(__file__).resolve().parents[1]
for p in (ROOT, ROOT / "oracle", ROOT / "multiview-clustering_b200"):
    if str(p) not in sys.path:
        sys.path.insert(0, str(p))


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")


def _cuda_device_present():
    """True when the product library is built and a CUDA device answers (cheap: one driver query)."""
    try:
        import ctypes
        cuda = ctypes.CDLL("libcuda.so.1")
        n = ctypes.c_int(0)
        return cuda.cuInit(0) == 0 and cuda.cuDeviceGetCount(ctypes.byref(n)) == 0 and n.value > 0
    except OSError:
        return False


def pytest_collection_modifyitems(config, items):
    """A plain `pytest tests` on a host without a GPU skips the gpu-marked tests instead of failing in mvg_create."""
    if _cuda_device_present():
        return
    skip = pytest.mark.skip(reason="no CUDA device: the sweep has no CPU path (run with -m gpu on the B200 box)")
    for item in items:
        if "gpu" in item.keywords:
            item.add_marker(skip)


def make_mixture(n, dims, k_true, seed, spread=2.0, noise=1.0):
    """Synthetic multiview Gaussian mixture in the style of New_Simulation.R:47-60 / SURVEY.md §8d (C3)."""
    rng = np.random.default_rng(seed)
    z = rng.integers(0, k_true, n)
    views = []
    for d in dims:
        mu = rng.normal(0.0, spread, (k_true, d))
        views.append((mu[z] + rng.normal(0.0, noise, (n, d))).astype(np.float32))
    return views, z


def c1_data(n=500, seed=1999):
    """Config 1: two scalar views (SURVEY.md §8d): view1 = N(3,1.3^2) U N(-3,1.3^2); view2 three groups."""
    rng = np.random.default_rng(seed)
    h, q = n // 2, n // 4
    v1 = np.concatenate([rng.normal(3, 1.3, h), rng.normal(-3, 1.3, n - h)])
    v2 = np.concatenate([rng.normal(0, 1.3, q), rng.normal(-5, 1.3, h), rng.normal(5, 1.3, n - q - h)])
    z1 = np.concatenate([np.zeros(h, int), np.ones(n - h, int)])
    z2 = np.concatenate([np.zeros(q, int), np.ones(h, int), np.full(n - q - h, 2)])
    return [v1.astype(np.float32), v2.astype(np.float32)], [z1, z2]


def reference_chain(seed, n, M, burn, thin):
    """Saved states of the reference's run_gibbs_cpp on c1_data(n) (tests/golden/reference_chains.npz; its "source" entry
    says what wrote them), in the form pyoracle.ref_run_gibbs returns them, and the number of uniforms + normals drawn."""
    z = np.load(Path(__file__).parent / "golden" / "reference_chains.npz")
    key = f"{seed}_{n}_{M}_{burn}_{thin}"
    tab, T, dish, hyp = (z[f"{key}/{k}"] for k in ("table_of", "T", "dish_of", "hypers"))
    d = dish.shape[1]
    states = [{"table_of": tab[s].astype(np.int32), "dish_of": dish[s, :, :T[s]].astype(np.int32),
               "alpha_v": hyp[s, :d], "sigma_v": hyp[s, d:2 * d], "tau_v": hyp[s, 2 * d:3 * d],
               "alpha_global": hyp[s, 3 * d], "sigma_global": hyp[s, 3 * d + 1]} for s in range(len(T))]
    return states, int(z[f"{key}/calls"])


@pytest.fixture(scope="session")
def oracle():
    import pyoracle
    pyoracle.lib()
    return pyoracle


def make_count_view(n, vocab, z, k_true, seed=0, mean_len=30, concentration=0.05):
    """Synthetic bag-of-words view: row i draws Poisson(mean_len) tokens from the multinomial of its cluster z[i]
    (some rows are empty, as in Reuters).  Returns a CSR dict {"rowptr", "col", "val", "vocab"}."""
    rng = np.random.default_rng(seed)
    theta = rng.dirichlet(np.full(vocab, concentration), k_true)
    rp, col, val = [0], [], []
    for i in range(n):
        ln = rng.poisson(mean_len) if rng.random() > 0.05 else 0
        r = rng.multinomial(ln, theta[z[i]])
        nz = np.nonzero(r)[0]
        col += list(nz)
        val += list(r[nz])
        rp.append(len(col))
    return {"rowptr": np.array(rp, np.int32), "col": np.array(col, np.int32), "val": np.array(val, np.float32), "vocab": int(vocab)}
