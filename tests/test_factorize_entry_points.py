"""The four factorize entry points of the C ABI against each other.

cnmf_factorize (device or host RNG), cnmf_factorize_seeds_dev, cnmf_factorize_init and cnmf_factorize_dev share one
host path: started from the same factors they must return the same bits.  Every GPU test here is marked `gpu`; the
symbol-table test at the end runs without a GPU.
"""
import os
import re
import shutil
import subprocess

import numpy as np
import pytest

from cnmf_golden import load_golden

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

KS = np.array([3, 7, 32, 1, 10], np.int32)                      # mixed K: both Gram widths, several GEMM tiles
SEEDS = np.array([1, 2 ** 31 - 2, 123456789, 42, 59886188], np.uint32)
CASES = [(tag, precision) for tag in ("sim_mu", "sim_cd") for precision in ("f16x2", "tf32x3-general", "fp32")]
SENTINEL = 7.0


@pytest.fixture(scope="module")
def eng():
    from cnmf_b200.engine import Engine
    return Engine(0)


@pytest.fixture(scope="module", params=CASES, ids=["%s-%s" % c for c in CASES])
def case(request, eng):
    """Dataset, solver arguments and the reference result: cnmf_factorize with the device RNG."""
    tag, precision = request.param
    g = load_golden(tag)
    ds = eng.dataset(g["X"], precision=precision)
    kw = dict(solver=g["solver"], tol=1e-4, max_iter=1000)
    sp, us, n_iter, err = ds.factorize(KS, SEEDS, kw, return_usages=True)
    return dict(ds=ds, kw=kw, spectra=np.vstack(sp), usages=np.vstack([u.T for u in us]), n_iter=n_iter, err=err)


def assert_same(a, b):
    assert a.dtype == b.dtype and a.shape == b.shape
    assert np.array_equal(a, b), int((a != b).sum())


def device_starts(ds):
    """random_init_dev into padded device buffers that start out as SENTINEL."""
    import torch
    ld_r, ld_c = ds.ld()
    SK = int(KS.sum())
    Wt = torch.full((SK, ld_r), SENTINEL, dtype=torch.float32, device="cuda:0")
    H = torch.full((SK, ld_c), SENTINEL, dtype=torch.float32, device="cuda:0")
    ds.random_init_dev(KS, SEEDS, Wt.data_ptr(), H.data_ptr())
    return Wt, H


@pytest.mark.gpu
def test_seeds_dev_matches_factorize(case):
    """Device-resident spectra with a row stride wider than n_cols: same bits, padding columns left alone."""
    import torch
    ds = case["ds"]
    G = ds.shape[1]
    ld_out = ds.ld()[1] + 40
    out = torch.full((int(KS.sum()), ld_out), SENTINEL, dtype=torch.float32, device="cuda:0")
    n_iter, err = ds.factorize_seeds_dev(KS, SEEDS, out.data_ptr(), ld_out, case["kw"])
    o = out.cpu().numpy()
    assert (o[:, G:] == SENTINEL).all()
    assert_same(o[:, :G], case["spectra"])
    assert_same(n_iter, case["n_iter"])
    assert_same(err, case["err"])


@pytest.mark.gpu
def test_factorize_dev_matches_factorize(case):
    """random_init_dev + factorize_dev (padded device factors in, full padded rows out) = factorize."""
    import torch
    ds = case["ds"]
    G = ds.shape[1]
    Wt, H = device_starts(ds)
    out = torch.full(H.shape, SENTINEL, dtype=torch.float32, device="cuda:0")
    n_iter, err = ds.factorize_dev(KS, Wt.data_ptr(), H.data_ptr(), out.data_ptr(), case["kw"])
    o = out.cpu().numpy()
    assert not (o[:, G:] == SENTINEL).any()          # every row is written out to ld_cols
    assert_same(o[:, :G], case["spectra"])
    assert_same(n_iter, case["n_iter"])
    assert_same(err, case["err"])


@pytest.mark.gpu
def test_factorize_init_from_device_starts_matches_factorize(case):
    """The device generator's factors, copied to the host without padding, through cnmf_factorize_init."""
    ds = case["ds"]
    n, G = ds.shape
    Wt, H = device_starts(ds)
    W0, H0 = Wt.cpu().numpy()[:, :n].copy(), H.cpu().numpy()[:, :G].copy()
    sp, us, n_iter, err = ds.factorize(KS, SEEDS, case["kw"], return_usages=True, W0=W0, H0=H0)
    assert_same(np.vstack(sp), case["spectra"])
    assert_same(np.vstack([u.T for u in us]), case["usages"])
    assert_same(n_iter, case["n_iter"])
    assert_same(err, case["err"])


@pytest.mark.gpu
def test_host_rng_matches_factorize_init(case):
    """rng='host' (pinned restart groups) = cnmf_factorize_init started from cnmf_random_init_host's factors."""
    from cnmf_b200 import _lib
    ds = case["ds"]
    n, G = ds.shape
    kw = dict(case["kw"], rng="host")
    sp, us, n_iter, err = ds.factorize(KS, SEEDS, kw, return_usages=True)
    s, _ = ds.sums()
    mean = s / (n * float(G))
    W0 = np.zeros((int(KS.sum()), n), np.float32)
    H0 = np.zeros((int(KS.sum()), G), np.float32)
    o = 0
    lib = _lib.load()
    for k, seed in zip(KS, SEEDS):
        _lib.check(lib.cnmf_random_init_host(int(seed), float(np.sqrt(mean / k)), n, G, int(k),
                                             _lib.ptr(W0[o:o + k]), n, _lib.ptr(H0[o:o + k]), G))
        o += k
    sp0, us0, n_iter0, err0 = ds.factorize(KS, SEEDS, case["kw"], return_usages=True, W0=W0, H0=H0)
    assert_same(np.vstack(sp), np.vstack(sp0))
    assert_same(np.vstack([u.T for u in us]), np.vstack([u.T for u in us0]))
    assert_same(n_iter, n_iter0)
    assert_same(err, err0)


@pytest.mark.gpu
def test_factorize_init_resets_timing(eng):
    """Every factorize entry point starts its timing afresh: supplied factors draw nothing, so rng_ms reads 0 even
    right after a call that did draw."""
    g = load_golden("sim_mu")
    ds = eng.dataset(g["X"])
    n, G = ds.shape
    kw = dict(solver="mu", tol=1e-4, max_iter=50)
    ds.factorize(KS, SEEDS, dict(kw, rng="host"))
    assert eng.last_timing()["rng_ms"] > 0
    SK = int(KS.sum())
    rng = np.random.RandomState(0)
    W0 = np.abs(rng.randn(SK, n)).astype(np.float32)
    H0 = np.abs(rng.randn(SK, G)).astype(np.float32)
    ds.factorize(KS, SEEDS, kw, W0=W0, H0=H0)
    t = eng.last_timing()
    assert t["rng_ms"] == 0
    assert t["solve_ms"] > 0


def test_library_exports_exactly_the_header_symbols():
    """The shared library's dynamic symbol table holds the header's cnmf_ functions and no other cnmf_ symbol."""
    from cnmf_b200 import _lib
    nm = shutil.which("nm")
    if nm is None:
        pytest.skip("nm not available")
    header = open(os.path.join(ROOT, "include", "cnmf_b200.h")).read()
    declared = set(re.findall(r"\b(cnmf_[a-z0-9_]+)\s*\(", header)) - {"cnmf_nmf_params"}
    out = subprocess.run([nm, "-D", "--defined-only", _lib.LIB_PATH], capture_output=True, text=True, check=True).stdout
    exported = {line.split()[-1] for line in out.splitlines() if line.split() and line.split()[-1].startswith("cnmf_")}
    assert exported == declared, (sorted(exported - declared), sorted(declared - exported))
