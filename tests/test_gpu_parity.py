"""GPU parity tests (`-m gpu`): the CUDA path, called through the C ABI (ctypes), against the oracle
and against the fixtures produced by the unmodified reference.

Tolerances (BASELINE.json north_star): spectra within 1e-4 rel-L2 of the reference (float64
scikit-learn) on identical seeds, identical iteration counts -- for EVERY restart of every fixture and of the
sampled BASELINE configurations, with one exemption stated by name (ILL_CONDITIONED below).
"""
import os
import warnings

import numpy as np
import pytest

from cnmf_golden import load_golden

pytestmark = pytest.mark.gpu

TOL_SPECTRA = 1e-4       # north star: spectra within 1e-4 rel-L2
TOL_GEMM = 2e-6          # fp32-class GEMM vs float64
# The single exemption from TOL_SPECTRA: fixture sim_mu, K=4, iter 0 (360 MU iterations along a nearly flat valley).  scikit-learn's OWN float32 path ends 1.75e-4 away from its float64 path on this restart
# (fixture `fp32dev_k4[0]`; every other restart of every fixture: <= 1e-5), so no implementation that stores its
# factors in fp32 can hold 1e-4 here; it is held to 1e-3 and must still reproduce the iteration count.
ILL_CONDITIONED = {("sim_mu", 4, 0): 1e-3}


def rel(a, b):
    a = np.asarray(a, dtype=np.float64)
    return float(np.linalg.norm(a - b) / np.linalg.norm(b))


@pytest.fixture(scope="module")
def eng():
    from cnmf_b200.engine import Engine
    return Engine(0)


# ------------------------------------------------------------------------------------ GEMM
@pytest.mark.parametrize("precision", ["tf32x3", "fp32"])
@pytest.mark.parametrize("shape", [(128, 256, 32, 1), (128, 256, 2048, 1), (200, 300, 100, 1), (7, 1000, 500, 1),
                                   (70, 40, 33, 1), (1, 5, 4, 1), (1000, 2000, 2000, 1), (300, 500, 4000, 4),
                                   (129, 257, 65, 2)])
def test_gemm_against_float64(eng, precision, shape):
    M, N, K, sp = shape
    rng = np.random.RandomState(M + N + K)
    A = np.abs(rng.randn(M, K)).astype(np.float32)
    B = np.abs(rng.randn(N, K)).astype(np.float32)
    C, _ = eng.gemm_abt(A, B, precision=precision, splits=sp)
    ref = A.astype(np.float64) @ B.astype(np.float64).T
    assert not np.isnan(C).any()
    assert rel(C, ref) < TOL_GEMM


@pytest.mark.parametrize("shape", [(128, 256, 64, 1), (128, 256, 2048, 1), (200, 300, 100, 1), (7, 1000, 500, 1),
                                   (70, 40, 33, 1), (1, 5, 4, 1), (1000, 2000, 2000, 1), (300, 500, 4000, 4),
                                   (129, 257, 65, 2), (1000, 2000, 20000, 9)])
def test_gemm_f16x2_against_float64(eng, shape):
    """kind::f16 path: A = two fp16 pieces of its row-normalised values (rows spanning 12 orders of magnitude and
    heavy-tailed entries), B = integer counts; same tolerance as the tf32 pair."""
    M, N, K, sp = shape
    rng = np.random.RandomState(M + N + K)
    A = (np.abs(rng.standard_cauchy((M, K))) * 10.0 ** rng.uniform(-6, 6, size=(M, 1))).astype(np.float32)
    A[:, ::7] = 0.0
    B = rng.poisson(1.5, size=(N, K)).astype(np.float32)
    B[0, 0] = 2048.0
    C, _ = eng.gemm_abt(A, B, precision="f16x2", splits=sp)
    ref = A.astype(np.float64) @ B.astype(np.float64).T
    assert not np.isnan(C).any()
    assert rel(C, ref) < TOL_GEMM
    rows = np.linalg.norm(C - ref, axis=1) / np.maximum(np.linalg.norm(ref, axis=1), 1e-300)
    assert rows.max() < 4 * TOL_GEMM, rows.max()          # every row, whatever its scale


def test_gemm_properties_full_size(eng):
    """BASELINE c2 shapes: split-K invariance, linearity, signed inputs (size-independent properties)."""
    rng = np.random.RandomState(0)
    M, N, K = 1000, 2000, 20000
    A = np.abs(rng.randn(M, K)).astype(np.float32)
    B = np.abs(rng.randn(N, K)).astype(np.float32)
    C1, _ = eng.gemm_abt(A, B, splits=1)
    C9, _ = eng.gemm_abt(A, B, splits=9)
    assert rel(C9, C1.astype(np.float64)) < 1e-6
    A2 = rng.randn(M, K).astype(np.float32)
    Cs, _ = eng.gemm_abt(A + A2, B, splits=9)
    C2, _ = eng.gemm_abt(A2, B, splits=9)
    assert rel(Cs, C9.astype(np.float64) + C2) < 1e-5
    ref_row = A[:3].astype(np.float64) @ B.astype(np.float64).T
    assert rel(C1[:3], ref_row) < TOL_GEMM


# ------------------------------------------------------------------------------------ random init
def test_device_rng_reproduces_numpy_legacy_stream(eng):
    """The on-device generator (MT19937 + polar gauss, one block per restart) against the host generator, which
    is bit-exact with numpy (tests/test_host_logic.py).  Only log() may differ from glibc in its last fp64 bit:
    at most a handful of fp32 values per million may differ, and then by one ulp."""
    import torch
    from cnmf_b200 import _lib
    g = load_golden("sim_mu")
    X = g["X"]
    ds = eng.dataset(X)
    n, G = ds.shape
    ks = np.array([3, 7, 32, 1, 10], np.int32)
    seeds = np.array([1, 2 ** 31 - 2, 123456789, 42, 59886188], np.uint32)
    ld_r, ld_c = ds.ld()
    SK = int(ks.sum())
    Wt = torch.full((SK, ld_r), 7.0, dtype=torch.float32, device="cuda:0")
    H = torch.full((SK, ld_c), 7.0, dtype=torch.float32, device="cuda:0")
    ds.random_init_dev(ks, seeds, Wt.data_ptr(), H.data_ptr())
    Wd, Hd = Wt.cpu().numpy(), H.cpu().numpy()
    s, _ = ds.sums()
    mean = s / (n * float(G))
    lib = _lib.load()
    Wh = np.zeros((SK, ld_r), np.float32)
    Hh = np.zeros((SK, ld_c), np.float32)
    o = 0
    for k, seed in zip(ks, seeds):
        _lib.check(lib.cnmf_random_init_host(int(seed), float(np.sqrt(mean / k)), n, G, int(k),
                                             _lib.ptr(Wh[o:o + k]), ld_r, _lib.ptr(Hh[o:o + k]), ld_c))
        o += k
    for dev, host in ((Wd, Wh), (Hd, Hh)):
        assert not dev[:, -1].any() or dev.shape[1] in (n, G)          # padding columns are zero
        diff = dev != host
        assert diff.sum() <= max(2, int(2e-6 * dev.size)), int(diff.sum())
        if diff.any():
            assert (np.abs(dev[diff] - host[diff]) <= np.abs(host[diff]) * 2.0 ** -22).all()


# ------------------------------------------------------------------------------------ factorize
def test_exact_count_detection(eng):
    """HVG-normalised counts (counts / std) and TPM (counts * 1e6 / total) are recognised as scaled integers and
    take the 2-pass products; arbitrary real data and 'tf32x3-general' stay on the general 3-pass path."""
    g = load_golden("sim_mu")
    assert eng.dataset(g["X"]).exact
    assert eng.dataset(g["tpm"]).exact
    assert not eng.dataset(g["X"], precision="tf32x3-general").exact
    assert not eng.dataset(g["X"], precision="fp32").exact
    rng = np.random.RandomState(0)
    assert not eng.dataset(np.abs(rng.randn(300, 120))).exact
    big = g["X"].copy()
    big[0, 0] = big[big[:, 0] > 0, 0].min() * 5000        # a count above 2048 is not tf32-exact
    assert not eng.dataset(big).exact


def _fixture_cases():
    out = []
    for tag in ("sim_mu", "sim_cd"):
        for precision in ("tf32x3", "f16x2", "tf32x3-hostrng", "tf32x3-general", "fp32"):
            out.append((tag, precision))
    for tag in ("c1_mu", "c1_cd"):          # BASELINE configs[0] in full: 1 000 x 500, K=7, 10 restarts
        for precision in ("f16x2", "tf32x3-general"):
            out.append((tag, precision))
    for precision in ("f16x2", "tf32x3-general"):      # `--init nndsvd` (cnmf.py:1252), the reference's default solver
        out.append(("sim_nndsvd", precision))
    return out


@pytest.mark.parametrize("tag,precision", _fixture_cases())
def test_factorize_matches_reference_fixture(eng, precision, tag):
    """Every restart of the reference's own factorize() run (fixture): same n_iter, spectra within 1e-4."""
    from oracle import nmf_ref
    g = load_golden(tag)
    rng = "host" if precision.endswith("-hostrng") else "device"
    precision = precision.replace("-hostrng", "")
    ds = eng.dataset(g["X"], precision=precision)
    kw = dict(solver=g["solver"], tol=1e-4, max_iter=1000, alpha_W=0.0, alpha_H=0.0, l1_ratio=0.0,
              beta_loss=2.0 if g["solver"] == "mu" else "frobenius", init=g["init"], rng=rng)
    table = g["table"]
    sp, us, n_iter, err = ds.factorize(table[:, 0], table[:, 2], kw, return_usages=True, X_host=g["X"])
    errs = []
    for r, (k, it, seed) in enumerate(table):
        ref = g["merged_k%d" % k][it * k:(it + 1) * k]
        e = rel(sp[r], ref)
        errs.append(e)
        limit = ILL_CONDITIONED.get((tag, int(k), int(it)), TOL_SPECTRA)
        assert e < limit, (tag, precision, k, it, e, limit)
        Wo, Ho, n_o = nmf_ref.nmf(g["X"], int(k), int(seed), solver=g["solver"], init=g["init"])
        assert n_o == int(n_iter[r]), (tag, precision, k, it, n_o, int(n_iter[r]))
        # reported final error = ||X - W H||_F of the returned factors
        e_true = nmf_ref.frobenius_error(g["X"], us[r].astype(np.float64), sp[r].astype(np.float64))
        assert abs(err[r] - e_true) / e_true < 1e-5
    assert np.median(errs) < 1e-5, errs


# ------------------------------------------------------------------------------------ BASELINE configurations, sampled
def _big_samples():
    z = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "big_samples.npz"))
    out = {}
    for key in z.files:
        if key.startswith("H_"):
            tag = key[2:]
            out[tag] = (z[key], int(z["it_" + tag]), z["meta_" + tag])
    return out


@pytest.mark.parametrize("case", ["c2", "c3", "k20", "k30"])
def test_factorize_baseline_configs_sampled(eng, case):
    """BASELINE.json configs[1] (20k x 2k, K=10), configs[2] (50k x 2k, K=5..13) and the K > 16 kernel path
    (configs[3]/[4]-shaped: K=20 on 4k x 2k, K=30 on 2k x 1k): restarts sampled from the configuration's own job table,
    solved in ONE mixed batch together with their neighbours in the table, against the reference's own call
    (sklearn non_negative_factorization float64 as cnmf.py:672 issues it; outputs stored by oracle/make_golden_big.py):
    identical n_iter, spectra within 1e-4."""
    from oracle.make_golden_big import CASES, case_inputs
    X, table = case_inputs(case)
    lookup = {(k, it): seed for k, it, seed in table}
    samples = {t: v for t, v in _big_samples().items() if t.startswith(case + "_")}
    assert samples
    ds = eng.dataset(X)
    assert ds.f16                                     # the default path: exact counts -> 2 kind::f16 passes
    for solver in ("mu", "cd"):
        want = [(t, v) for t, v in samples.items() if t.endswith("_" + solver)]
        if not want:
            continue
        jobs = [(int(v[2][2]), int(v[2][3])) for _, v in want]
        # neighbours from the same job table: other K's / seeds share the batch (mixed-K packing, compaction)
        extra = [(k, it) for (k, it, _) in table[1::max(1, len(table) // 6)] if (k, it) not in jobs][:5]
        batch = jobs + extra
        kw = dict(solver=solver, tol=1e-4, max_iter=1000, beta_loss=2.0 if solver == "mu" else "frobenius")
        sp, _, n_iter, _ = ds.factorize([k for k, _ in batch], [lookup[j] for j in batch], kw)
        for i, (t, (H, it_ref, meta)) in enumerate(want):
            assert meta[0] == X.shape[0] and meta[1] == X.shape[1] and meta[4] == lookup[jobs[i]]
            e = rel(sp[i], H)
            assert int(n_iter[i]) == it_ref, (t, int(n_iter[i]), it_ref)
            assert e < TOL_SPECTRA, (t, e)
        # the same restarts alone: a restart's result does not depend on the batch it ran in
        sp1, _, n1, _ = ds.factorize([k for k, _ in jobs[:1]], [lookup[jobs[0]]], kw)
        assert int(n1[0]) == int(n_iter[0])
        assert rel(sp1[0], sp[0].astype(np.float64)) < 1e-6, rel(sp1[0], sp[0].astype(np.float64))


def test_factorize_batching_invariance(eng):
    """A restart's result does not depend on what else is in the batch (bit-exact)."""
    g = load_golden("sim_mu")
    ds = eng.dataset(g["X"])
    kw = dict(solver="mu", tol=1e-4, max_iter=200)
    t = g["table"]
    sp_all, _, it_all, _ = ds.factorize(t[:6, 0], t[:6, 2], kw)
    sp_one, _, it_one, _ = ds.factorize(t[3:4, 0], t[3:4, 2], kw)
    assert it_one[0] == it_all[3]
    assert np.array_equal(sp_one[0], sp_all[3])


@pytest.mark.parametrize("solver", ["mu", "cd"])
def test_factorize_edge_shapes(eng, solver):
    """Ragged sizes (not multiples of any tile), K = 1 and K = 32 (the maximum), a single restart."""
    from oracle import nmf_ref
    from cnmf_b200.synth import make_counts, normalise
    X64, _ = normalise(make_counts(333, 97, k_true=3, seed=3, libsize=500.0), np.float64)
    ds = eng.dataset(X64)
    for k, seed in ((1, 11), (32, 12), (3, 13)):
        kw = dict(solver=solver, tol=1e-4, max_iter=60)
        sp, _, n_iter, _ = ds.factorize([k], [seed], kw)
        W, H, it = nmf_ref.nmf(X64, k, seed, solver=solver, max_iter=60)
        assert it == int(n_iter[0])
        assert rel(sp[0], H) < 5e-4, (solver, k, rel(sp[0], H))     # 60 iterations far from converged: looser
    with pytest.raises(Exception, match=r"\[1, 32\]"):
        ds.factorize([33], [1], dict(solver=solver, tol=1e-4, max_iter=10))


def test_factorize_with_regularisation(eng):
    from oracle import nmf_ref
    g = load_golden("sim_mu")
    X = g["X"]
    ds = eng.dataset(X)
    for solver in ("mu", "cd"):
        kw = dict(solver=solver, tol=1e-4, max_iter=150, alpha_W=0.002, alpha_H=0.001, l1_ratio=0.3)
        sp, _, n_iter, _ = ds.factorize([5], [99], kw)
        W, H, it = nmf_ref.nmf(X, 5, 99, solver=solver, max_iter=150, alpha_W=0.002, alpha_H=0.001, l1_ratio=0.3)
        assert it == int(n_iter[0])
        assert rel(sp[0], H) < TOL_SPECTRA


# ------------------------------------------------------------------------------------ beta-divergence losses
@pytest.mark.parametrize("precision", ["tf32x3", "fp32"])
def test_factorize_kl_matches_reference_fixture(eng, precision):
    """--beta-loss kullback-leibler (cnmf.py:629-631 -> solver 'mu', beta = 1): every restart of the reference's own
    run, same n_iter, spectra within the north-star tolerance; reported errors = sqrt(2 KL) is not returned, the
    Frobenius residual of the final factors is."""
    from oracle import nmf_ref
    g = load_golden("sim_kl")
    assert g["beta"] == 1 and g["solver"] == "mu"
    ds = eng.dataset(g["X"], precision=precision)
    kw = dict(solver="mu", beta_loss="kullback-leibler", tol=1e-4, max_iter=1000)
    table = g["table"]
    sp, us, n_iter, err = ds.factorize(table[:, 0], table[:, 2], kw, return_usages=True)
    errs = []
    for r, (k, it, seed) in enumerate(table):
        ref = g["merged_k%d" % k][it * k:(it + 1) * k]
        e = rel(sp[r], ref)
        errs.append(e)
        assert e < TOL_SPECTRA, (precision, k, it, e)
        Wo, Ho, n_o = nmf_ref.nmf(g["X"], int(k), int(seed), solver="mu", beta=1)
        assert n_o == int(n_iter[r]), (precision, k, it, n_o, int(n_iter[r]))
        e_true = nmf_ref.frobenius_error(g["X"], us[r].astype(np.float64), sp[r].astype(np.float64))
        assert abs(err[r] - e_true) / e_true < 1e-5
    assert np.median(errs) < 2e-5, errs


def test_kl_refit_regularisation_and_edge_shapes(eng):
    from oracle import nmf_ref
    from cnmf_b200.synth import make_counts, normalise
    g = load_golden("sim_kl")
    X, tpm = g["X"], g["tpm"]
    k = int(g["ks"][1])
    kw = dict(solver="mu", beta_loss="kullback-leibler", tol=1e-4, max_iter=1000)
    ds = eng.dataset(X)
    # refit_usage / refit_spectra with the loss of the run (cnmf.py:792 re-reads the yaml)
    H = g["cspectra_k%d" % k]
    W, it, err = ds.refit(H, kw)
    Wr, itr = nmf_ref.refit(X, H, "mu", beta=1)
    assert it == itr and rel(W, Wr) < TOL_SPECTRA
    assert abs(err - nmf_ref.frobenius_error(X, Wr, H)) / err < 1e-5
    U = Wr / Wr.sum(axis=1, keepdims=True)
    tds = eng.dataset(tpm)
    Ht, it2, _ = tds.refit(np.ascontiguousarray(U.T), kw, transposed=True)
    Hr, itr2 = nmf_ref.refit(tpm.T, U.T, "mu", beta=1)
    assert it2 == itr2 and rel(Ht, Hr) < TOL_SPECTRA
    # regularised
    kwr = dict(kw, max_iter=150, alpha_W=0.002, alpha_H=0.001, l1_ratio=0.3)
    sp, _, n_iter, _ = ds.factorize([5], [99], kwr)
    _, Hreg, itreg = nmf_ref.nmf(X, 5, 99, solver="mu", beta=1, max_iter=150, alpha_W=0.002, alpha_H=0.001, l1_ratio=0.3)
    assert itreg == int(n_iter[0]) and rel(sp[0], Hreg) < TOL_SPECTRA
    # ragged sizes, K = 1 / 17 / 32 in ONE batch (three register classes of the kernel)
    X64, _ = normalise(make_counts(333, 97, k_true=3, seed=3, libsize=500.0), np.float64)
    ds2 = eng.dataset(X64)
    ks, seeds = [1, 17, 32, 3], [11, 12, 13, 14]
    sp, _, n_iter, _ = ds2.factorize(ks, seeds, dict(kw, max_iter=40))
    for r, (kk, seed) in enumerate(zip(ks, seeds)):
        _, Ho, ito = nmf_ref.nmf(X64, kk, seed, solver="mu", beta=1, max_iter=40)
        assert ito == int(n_iter[r])
        assert rel(sp[r], Ho) < 5e-4, (kk, rel(sp[r], Ho))
    with pytest.raises(ValueError):          # sklearn: 'cd' does not handle beta_loss != frobenius
        ds.factorize([3], [1], dict(kw, solver="cd"))


def test_itakura_saito(eng):
    """beta = 0: sklearn refuses X with zeros (_nmf.py:1675-1680) -- count data always has them; on strictly
    positive X the updates (gamma = 1/2, both factors clipped) match the oracle."""
    from oracle import nmf_ref
    g = load_golden("sim_kl")
    kw = dict(solver="mu", beta_loss="itakura-saito", tol=1e-4, max_iter=300)
    with pytest.raises(ValueError, match="contains zeros"):
        eng.dataset(g["X"]).factorize([4], [1], kw)
    Xp = g["X"] + 0.1
    ds = eng.dataset(Xp)
    assert abs(ds.min() - Xp.min()) < 1e-6
    sp, us, n_iter, err = ds.factorize([4, 9], [5, 6], kw, return_usages=True)
    for r, (k, seed) in enumerate(((4, 5), (9, 6))):
        Wo, Ho, ito = nmf_ref.nmf(Xp, k, seed, solver="mu", beta=0, max_iter=300)
        assert ito == int(n_iter[r]), (k, ito, int(n_iter[r]))
        assert rel(sp[r], Ho) < 5e-4, (k, rel(sp[r], Ho))
    Wr, itr = nmf_ref.refit(Xp, Ho, "mu", beta=0, max_iter=300)
    W, it, _ = ds.refit(Ho, kw)
    assert it == itr and rel(W, Wr) < 5e-4



# ------------------------------------------------------------------------------------ refits
@pytest.mark.parametrize("precision", ["tf32x3", "f16x2", "tf32x3-general"])
@pytest.mark.parametrize("tag", ["sim_mu", "sim_cd"])
def test_refits_match_oracle(eng, tag, precision):
    from oracle import nmf_ref
    g = load_golden(tag)
    k = int(g["ks"][1])
    X, tpm = g["X"], g["tpm"]
    kw = dict(solver=g["solver"], tol=1e-4, max_iter=1000)
    ds = eng.dataset(X, precision=precision)
    H = g["cspectra_k%d" % k]
    W, it, err = ds.refit(H, kw)
    Wr, itr = nmf_ref.refit(X, H, g["solver"])
    assert it == itr and rel(W, Wr) < TOL_SPECTRA
    assert abs(err - nmf_ref.frobenius_error(X, Wr, H)) / err < 1e-5
    # refit_spectra: transposed problem on the TPM matrix (cnmf.py:805-820, 952)
    U = Wr / Wr.sum(axis=1, keepdims=True)
    tds = eng.dataset(tpm, precision=precision)
    Ht, it2, _ = tds.refit(np.ascontiguousarray(U.T), kw, transposed=True)
    Hr, itr2 = nmf_ref.refit(tpm.T, U.T, g["solver"])
    assert it2 == itr2 and rel(Ht, Hr) < TOL_SPECTRA
    # column-subset dataset (cnmf.py:965-969: tpm[:, hvgs] / std) keeps its exactness and its values
    hv = g["hvg_idx"]
    std1 = tpm[:, hv].std(axis=0, ddof=1)
    sub = tds.from_columns(hv, 1.0 / std1)
    assert sub.exact == tds.exact
    Xs = tpm[:, hv] / std1
    Hs = np.abs(np.random.RandomState(1).randn(k, len(hv))) + 0.1
    Ws, its, _ = sub.refit(Hs, kw)
    Wsr, itsr = nmf_ref.refit(Xs, Hs, g["solver"])
    assert its == itsr and rel(Ws, Wsr) < TOL_SPECTRA
    # OLS projection accumulator (cnmf.py:119): Ut @ X with signed (centred) Ut
    Ut = np.random.RandomState(2).randn(k, tpm.shape[0])
    assert rel(tds.project_rows(Ut), Ut @ tpm) < 1e-5


# ------------------------------------------------------------------------------------ consensus kernels
def test_consensus_kernels_match_oracle(eng):
    from cnmf_b200 import consensus as cs
    from oracle import consensus_ref as cr
    g = load_golden("sim_mu")
    for k in g["ks"]:
        k = int(k)
        merged = g["merged_k%d" % k]
        S = cs.SpectraMatrix(eng, merged).l2_normalize()
        l2 = cr.l2_normalize_rows(merged)
        assert rel(S.numpy(), l2) < 1e-6
        n_nb = int(0.3 * merged.shape[0] / k)
        dens, D = S.local_density(n_nb, return_dist=True)
        assert rel(dens, g["density_k%d" % k]) < 1e-5           # the reference's own cache file
        assert np.abs(D - cr.euclidean_distances(l2)).max() < 2e-6
        assert (np.diag(D) == 0).all()
        labels, labels_t, inertia, _ = cs.kmeans(S, k)
        lref, iref, _ = cr.kmeans(l2, k)
        assert np.array_equal(labels, lref) and abs(inertia - iref) / iref < 1e-4
        assert rel(cs.cluster_medians(S, labels_t, k), cr.cluster_medians(l2, lref, k)) < 1e-6


def test_consensus_kernels_larger_random(eng):
    """R = 3000 x G = 2000 with planted clusters + outliers: density, filter, KMeans partition, medians."""
    from cnmf_b200 import consensus as cs
    from oracle import consensus_ref as cr
    rng = np.random.RandomState(5)
    cen = np.abs(rng.randn(12, 2000))
    pts = np.vstack([c + 0.05 * np.abs(rng.randn(240, 2000)) for c in cen] + [np.abs(rng.randn(120, 2000))])
    S = cs.SpectraMatrix(eng, pts).l2_normalize()
    l2 = cr.l2_normalize_rows(pts)
    dens, _ = S.local_density(72)
    dref = cr.local_density(cr.euclidean_distances(l2), 72)
    assert rel(dens, dref) < 1e-5
    keep = dens < 0.5
    assert np.array_equal(keep, dref < 0.5)
    S2 = S.take_rows(np.where(keep)[0])
    labels, labels_t, inertia, _ = cs.kmeans(S2, 12)
    lref, iref, _ = cr.kmeans(l2[keep], 12)
    assert np.array_equal(labels, lref)
    assert rel(cs.cluster_medians(S2, labels_t, 12), cr.cluster_medians(l2[keep], lref, 12)) < 1e-6
    # idempotence: normalising twice changes nothing beyond fp32 rounding
    before = S.numpy().copy()
    S.l2_normalize()
    assert np.abs(S.numpy() - before).max() < 1e-7


# ------------------------------------------------------------------------------------ end to end through the facade
@pytest.mark.parametrize("tag", ["sim_mu", "sim_cd", "sim_kl", "sim_nndsvd", "c1_mu", "c1_cd"])
def test_pipeline_matches_reference_outputs(tmp_path, tag):
    """prepare -> factorize -> combine -> consensus through cnmf_b200.cNMF on the fixture's counts; every
    file the reference wrote is reproduced within tolerance (the reference test's own criterion is a sum of
    squared differences < 1e-4, tests/test_reproducibility.py:111-112; relative bounds here are tighter)."""
    import pandas as pd
    from cnmf_b200 import cNMF, load_df_from_npz, save_df_to_npz
    g = load_golden(tag)
    counts = g["counts"].astype(np.float64)
    df = pd.DataFrame(counts, index=["c%d" % i for i in range(counts.shape[0])],
                      columns=["g%d" % i for i in range(counts.shape[1])])
    fn = str(tmp_path / "counts.df.npz")
    save_df_to_npz(df, fn)
    obj = cNMF(output_dir=str(tmp_path), name="run")
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        obj.prepare(fn, components=list(g["ks"]), n_iter=int(g["n_iter"]), seed=int(g["seed"]), densify=True,
                    beta_loss=g["beta_loss_arg"], num_highvar_genes=len(g["hvg_idx"]), init=g["init"])
        obj.factorize()
        obj.combine()
        dt = float(g["dt"])
        for k in g["ks"]:
            k = int(k)
            merged = load_df_from_npz(obj.paths["merged_spectra"] % k)
            assert merged.shape == g["merged_k%d" % k].shape
            assert list(merged.index[:2]) == ["iter0_topic1", "iter0_topic2"]
            stats = obj.consensus(k, skip_density_and_return_after_stats=True, show_clustering=False)
            ref_stats = g["stats_k%d" % k]
            assert abs(stats.loc["silhouette", "stats"] - ref_stats[2]) < 1e-4
            assert abs(stats.loc["prediction_error", "stats"] - ref_stats[3]) / ref_stats[3] < 1e-5
            obj.consensus(k, density_threshold=dt, show_clustering=False)
            dts = str(dt).replace(".", "_")
            for key, name in (("consensus_spectra", "cspectra"), ("consensus_usages", "cusages"),
                              ("gene_spectra_tpm", "tpmspec"), ("gene_spectra_score", "score"),
                              ("starcat_spectra", "starcat")):
                got = load_df_from_npz(obj.paths[key] % (k, dts)).values
                ref = g["%s_k%d" % (name, k)]
                e = rel(got, ref)
                # the K=4 consensus of sim_mu contains the ill-conditioned restart named above (1 of its 8)
                limit = 3e-4 if (tag, k) == ("sim_mu", 4) else TOL_SPECTRA
                assert e < limit, (tag, k, key, e)
                assert os.path.exists(obj.paths[key + "__txt"] % (k, dts))


# ------------------------------------------------------------------------------------ facade behaviour on the GPU
def _prepared(tmp_path, g, name="run", n_iter=None):
    import pandas as pd
    from cnmf_b200 import cNMF, save_df_to_npz
    counts = g["counts"].astype(np.float64)
    df = pd.DataFrame(counts, index=["c%d" % i for i in range(counts.shape[0])],
                      columns=["g%d" % i for i in range(counts.shape[1])])
    tmp_path.mkdir(parents=True, exist_ok=True)
    fn = str(tmp_path / "counts.df.npz")
    save_df_to_npz(df, fn)
    obj = cNMF(output_dir=str(tmp_path), name=name)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        obj.prepare(fn, components=list(g["ks"]), n_iter=int(g["n_iter"]) if n_iter is None else n_iter,
                    seed=int(g["seed"]), densify=True, beta_loss=g["beta_loss_arg"],
                    num_highvar_genes=len(g["hvg_idx"]))
    return obj


def test_worker_split_and_resume_give_identical_files(tmp_path):
    """factorize(worker_i, total_workers) over two workers, and a resumed run with skip_completed_runs, write
    the files a single worker writes (cnmf.py:692-745, 729-733): same (k, iter) -> same seed -> same spectra,
    whatever batch the restart was solved in (the split-K partition is a function of the matrix shape only, the
    operand pieces a function of the factor values only).  Held to 1e-6 rel-L2 rather than bitwise: the fp64
    reduction order of the K x K Gram partials follows the launch geometry, which can move an fp32 rounding."""
    from cnmf_b200 import load_df_from_npz
    g = load_golden("sim_mu")
    a = _prepared(tmp_path / "a", g, n_iter=4)
    b = _prepared(tmp_path / "b", g, n_iter=4)
    c = _prepared(tmp_path / "c", g, n_iter=4)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        a.factorize()
        b.factorize(worker_i=0, total_workers=2)
        b.factorize(worker_i=1, total_workers=2)
        c.factorize(worker_i=1, total_workers=3)            # a partial run ...
        c.update_nmf_iter_params()
        c.factorize(skip_completed_runs=True)               # ... resumed
    for k in g["ks"]:
        for it in range(4):
            ref = load_df_from_npz(a.paths["iter_spectra"] % (k, it))
            for other in (b, c):
                got = load_df_from_npz(other.paths["iter_spectra"] % (k, it))
                assert got.shape == ref.shape and list(got.index) == list(range(1, k + 1))
                rel = np.linalg.norm(got.values - ref.values) / np.linalg.norm(ref.values)
                assert rel < 1e-6, (k, it, rel)


def test_consensus_errors_and_density_cache(tmp_path):
    """Zero surviving spectra raises the reference's RuntimeError (cnmf.py:905-906); the local-density cache is
    written once and reused, keyed by k only (cnmf.py:887-899)."""
    import os as _os
    from cnmf_b200 import load_df_from_npz
    g = load_golden("sim_mu")
    obj = _prepared(tmp_path, g)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        obj.factorize()
        obj.combine()
        k = int(g["ks"][0])
        with pytest.raises(RuntimeError, match="Zero components remain"):
            obj.consensus(k, density_threshold=1e-9, show_clustering=False)
        cache = obj.paths["local_density_cache"] % k
        assert _os.path.exists(cache)
        before = load_df_from_npz(cache)
        mtime = _os.path.getmtime(cache)
        obj.consensus(k, density_threshold=0.5, local_neighborhood_size=0.9, show_clustering=False)   # cache wins
        assert _os.path.getmtime(cache) == mtime and load_df_from_npz(cache).equals(before)
        usage, scores, tpm, top = obj.load_results(k, 0.5, n_top_genes=5)
        assert np.allclose(usage.sum(axis=1), 1.0) and top.shape == (5, k)


def test_k_selection_statistics(tmp_path):
    """k_selection_plot statistics (cnmf.py:1119-1135) against the reference's own stats branch output."""
    g = load_golden("sim_mu")
    obj = _prepared(tmp_path, g)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        obj.factorize()
        obj.combine()
        stats = obj.k_selection_plot(close_fig=True)
    for row, k in enumerate(sorted(int(x) for x in g["ks"])):
        ref = g["stats_k%d" % k]
        assert int(stats.loc[row, "k"]) == k
        assert abs(stats.loc[row, "silhouette"] - ref[2]) < 1e-4
        assert abs(stats.loc[row, "prediction_error"] - ref[3]) / ref[3] < 1e-5


# ------------------------------------------------------------------------------------ device-side prepare
def test_prepare_primitives_match_numpy(eng):
    """Cell totals, row-scaled column statistics and the row-scaled dataset against float64 numpy."""
    rng = np.random.RandomState(5)
    C = rng.poisson(0.7, size=(3001, 517)).astype(np.float64)
    C[:, 3] = 0.0                                   # an all-zero gene
    C[7] = 0.0
    C[7, 0] = 2.0
    ds = eng.dataset(C)
    tot = ds.row_sums()
    assert np.array_equal(tot, C.sum(axis=1))       # integers: exact
    rs = 1e6 / tot
    T = C * rs[:, None]
    mean, var = ds.col_stats(row_scale=rs)
    assert np.allclose(mean, T.mean(axis=0), rtol=1e-13, atol=0)
    assert np.allclose(var, T.var(axis=0), rtol=1e-10, atol=1e-9)
    m0, v0 = ds.col_stats()
    assert np.allclose(m0, C.mean(axis=0), rtol=1e-13) and np.allclose(v0, C.var(axis=0), rtol=1e-11, atol=1e-14)
    tds = ds.scale_rows(rs)
    assert tds.exact                                # TPM = integers x per-cell factor: 2-pass products
    s, q = tds.sums()
    assert abs(s - T.sum()) / T.sum() < 1e-6 and abs(q - (T ** 2).sum()) / (T ** 2).sum() < 1e-6
    # columns of a tall matrix (> 65535 rows went through a per-row grid before)
    big = eng.dataset(rng.poisson(1.0, size=(70001, 40)).astype(np.float64))
    sub = big.from_columns([5, 1, 39], [0.5, 2.0, 1.0])
    assert sub.shape == (70001, 3)
    m, _ = sub.col_stats()
    mb, _ = big.col_stats()
    assert np.allclose(m, mb[[5, 1, 39]] * np.array([0.5, 2.0, 1.0]), rtol=1e-12)


@pytest.mark.parametrize("tag", ["sim_mu"])
def test_prepare_on_device_matches_reference_outputs(tmp_path, tag):
    """prepare(on_device=True): HVG choice, normalised counts and TPM statistics equal what the reference wrote
    (fixture), and factorize() consumes the matrix prepare left in HBM."""
    import pandas as pd
    from cnmf_b200 import cNMF, load_df_from_npz, save_df_to_npz
    from cnmf_b200 import io as cio
    g = load_golden(tag)
    counts = g["counts"].astype(np.float64)
    df = pd.DataFrame(counts, index=["c%d" % i for i in range(counts.shape[0])],
                      columns=["g%d" % i for i in range(counts.shape[1])])
    fn = str(tmp_path / "counts.df.npz")
    save_df_to_npz(df, fn)
    obj = cNMF(output_dir=str(tmp_path), name="dev")
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        obj.prepare(fn, components=list(g["ks"]), n_iter=int(g["n_iter"]), seed=int(g["seed"]), densify=True,
                    beta_loss=g["beta_loss_arg"], num_highvar_genes=len(g["hvg_idx"]), on_device=True)
    hvgs = open(obj.paths["nmf_genes_list"]).read().split("\n")
    assert [int(x[1:]) for x in hvgs] == list(g["hvg_idx"])
    norm = cio.read_matrix(obj.paths["normalized_counts"])
    assert np.allclose(norm.X, g["X"], rtol=1e-12, atol=0)
    stats = load_df_from_npz(obj.paths["tpm_stats"])
    assert np.allclose(stats["__std"].values, g["tpm_std"], rtol=1e-10)
    assert obj._resident_norm is not None and obj._resident_norm.shape == norm.X.shape
    s, _ = obj._resident_norm.sums()
    assert abs(s - g["X"].sum()) / g["X"].sum() < 1e-6
    n0 = obj.engine().launch_count
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        obj.factorize()
    assert obj.engine().launch_count > n0
    obj.combine()
    k = int(g["ks"][0])
    merged = load_df_from_npz(obj.paths["merged_spectra"] % k).values
    ref = g["merged_k%d" % k]
    errs = [rel(merged[i * k:(i + 1) * k], ref[i * k:(i + 1) * k]) for i in range(ref.shape[0] // k)]
    assert np.median(errs) < 1e-5, errs


# ------------------------------------------------------------------------------------ round-2 additions
def test_density_filter_decision_near_tight_threshold(eng):
    """BASELINE configs[3] runs consensus at density_threshold = 0.01: replicate spectra whose local densities
    straddle the threshold (every cluster holds replicates with relative noise 1e-3 ... 3e-2, so the filter cuts
    through each of them: ~2/3 kept, nearest margin 8e-4 relative).  The keep/drop decision of every
    row must equal the oracle's (sklearn euclidean_distances + argpartition, float64); this is the regime the
    direct-difference distance kernel exists for (a Gram-form fp32 distance has ~3e-4 absolute error here)."""
    from cnmf_b200 import consensus as cs
    from oracle import reference_path
    rng = np.random.RandomState(11)
    K, reps, G = 20, 60, 2000
    cen = rng.gamma(0.3, 1.0, size=(K, G)) + 1e-3
    spread = np.geomspace(1e-3, 3e-2, reps)            # per-replicate noise: local densities from 0.002 to 0.03
    pts = np.vstack([cen[c] * (1.0 + spread[:, None] * rng.randn(reps, G)).clip(0.0) for c in range(K)])
    pts = pts[rng.permutation(len(pts))]
    dref, keep_ref, labels_ref, med_ref = reference_path.consensus_cluster(pts, K, density_threshold=0.01)
    assert 0.5 < keep_ref.mean() < 0.8                 # the threshold cuts through every cluster
    S = cs.SpectraMatrix(eng, pts).l2_normalize()
    dens, _ = S.local_density(int(0.3 * len(pts) / K))
    margin = np.abs(dref - 0.01) / 0.01
    assert rel(dens, dref) < 2e-5
    keep = dens < 0.01
    assert np.array_equal(keep, keep_ref), (int((keep != keep_ref).sum()), float(margin.min()))
    S2 = S.take_rows(np.where(keep)[0])
    k_kept = len(set(labels_ref))
    labels, labels_t, _, _ = cs.kmeans(S2, K)
    assert np.array_equal(labels, labels_ref)
    med = cs.cluster_medians(S2, labels_t, K)
    assert rel(med, med_ref) < 1e-6 and k_kept == K


def test_sparse_norm_counts_round_trip(tmp_path):
    """The reference keeps X sparse (CSR) unless --densify (cnmf.py:399-405, 534-538).  prepare(densify=False)
    stores CSR norm_counts / tpm, factorize and consensus consume them, and every output equals the dense run."""
    import scipy.sparse as sp
    from cnmf_b200 import cNMF, load_df_from_npz
    from cnmf_b200 import io as cio
    g = load_golden("sim_cd")
    a = _prepared(tmp_path / "dense", g, n_iter=4)
    import pandas as pd
    from cnmf_b200 import save_df_to_npz
    counts = g["counts"].astype(np.float64)
    df = pd.DataFrame(counts, index=["c%d" % i for i in range(counts.shape[0])],
                      columns=["g%d" % i for i in range(counts.shape[1])])
    (tmp_path / "sparse").mkdir()
    fn = str(tmp_path / "sparse" / "counts.df.npz")
    save_df_to_npz(df, fn)
    b = cNMF(output_dir=str(tmp_path / "sparse"), name="run")
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        b.prepare(fn, components=list(g["ks"]), n_iter=4, seed=int(g["seed"]), densify=False,
                  beta_loss=g["beta_loss_arg"], num_highvar_genes=len(g["hvg_idx"]))
    nb = cio.read_matrix(b.paths["normalized_counts"])
    assert sp.issparse(nb.X) and sp.issparse(cio.read_matrix(b.paths["tpm"]).X)
    na = cio.read_matrix(a.paths["normalized_counts"])
    assert np.array_equal(nb.X.toarray(), na.X)
    k = int(g["ks"][1])
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        for obj in (a, b):
            obj.factorize()
            obj.combine()
            obj.consensus(k, density_threshold=2.0, show_clustering=False)
    for key in ("consensus_spectra", "consensus_usages", "gene_spectra_tpm", "gene_spectra_score"):
        ra = load_df_from_npz(a.paths[key] % (k, "2_0")).values
        rb = load_df_from_npz(b.paths[key] % (k, "2_0")).values
        assert rel(rb, ra) < 1e-6, key


def test_clustergram_order_matches_reference_rule(tmp_path):
    """cnmf.py:986-1010: clusters in label order, average-linkage leaf order inside a cluster, on the distances of
    the density-filtered spectra.  Oracle: the same scipy calls on sklearn's float64 distances."""
    from scipy.cluster.hierarchy import leaves_list, linkage
    from scipy.spatial.distance import squareform
    from sklearn.metrics.pairwise import euclidean_distances
    from cnmf_b200 import load_df_from_npz
    from oracle import consensus_ref as cr
    g = load_golden("c1_mu")
    obj = _prepared(tmp_path, g)
    k = int(g["ks"][0])
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        obj.factorize()
        obj.combine()
        obj.consensus(k, density_threshold=float(g["dt"]), show_clustering=True, close_clustergram_fig=True)
    order = list(obj.last_clustergram_order)
    merged = load_df_from_npz(obj.paths["merged_spectra"] % k).values
    l2 = cr.l2_normalize_rows(merged)
    D = euclidean_distances(l2)
    n_nb = int(0.3 * merged.shape[0] / k)
    dens = cr.local_density(D, n_nb)
    keep = dens < float(g["dt"])
    labels, _, _ = cr.kmeans(l2[keep], k)
    Df = D[keep][:, keep]
    ref = []
    for cl in sorted(set(labels)):
        f = labels == cl
        if f.sum() > 1:
            d = squareform(Df[f][:, f], checks=False)
            d[d < 0] = 0
            ref += list(np.where(f)[0][leaves_list(linkage(d, "average"))])
        else:
            ref += list(np.where(f)[0])
    assert sorted(order) == list(range(int(keep.sum())))
    assert order == ref


def test_two_gpu_sharded_factorize_allgather_consensus():
    """tests/gpu_dist_check.py under torchrun with 2 ranks: restarts sharded idx % 2, ONE NCCL all-gather through the C
    ABI (cnmf_allgather_spectra on a communicator made by cnmf_comm_create), merged spectra equal the reference fixture
    on both ranks, consensus Ks sharded over the ranks.  Needs 2 GPUs (skipped on a single-GPU box)."""
    import subprocess
    import sys
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs >= 2 GPUs")
    script = os.path.join(os.path.dirname(os.path.abspath(__file__)), "gpu_dist_check.py")
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2",
                        "--master-addr", "127.0.0.1", "--master-port", "29571", script],
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-4000:]
    assert r.stdout.count("merged spectra match the reference fixture") == 2, r.stdout[-2000:]


def test_mixed_k_multi_tile_batch_matches_oracle(eng):
    """A multi-tile, mixed-K batch (45 restarts, K = 5..13, 405 packed rows over four 128-row GEMM tiles) against the
    numpy oracle on every fourth restart: identical n_iter, spectra within 1e-4."""
    from cnmf_b200.synth import make_counts, normalise, restart_table
    from oracle import nmf_ref
    X, _ = normalise(make_counts(1000, 500, k_true=7, seed=0, libsize=800.0), np.float64)
    rows = restart_table(list(range(5, 14)), 5, seed=14)
    assert sum(r[0] for r in rows) == 405
    ds = eng.dataset(X)
    sp, _, n_iter, _ = ds.factorize([r[0] for r in rows], [r[2] for r in rows],
                                    dict(solver="mu", beta_loss=2.0, tol=1e-4, max_iter=400))
    bad = []
    for i in range(0, len(rows), 4):
        k, _, seed = rows[i]
        _, H, it = nmf_ref.nmf(X, k, seed, solver="mu", max_iter=400)
        e = rel(sp[i], H)
        if it != int(n_iter[i]) or e >= TOL_SPECTRA:
            bad.append((i, k, it, int(n_iter[i]), e))
    assert bad == []
