"""CPU tests: C-ABI surface, host RNG, file ledger, prepare(), job sharding, gloo all-gather."""
import ctypes
import os
import re
import subprocess
import sys

import numpy as np
import pandas as pd
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

from cnmf_b200 import _lib, cNMF, load_df_from_npz, save_df_to_npz  # noqa: E402
from cnmf_b200.parallel import shard_jobs  # noqa: E402
from cnmf_b200.pipeline import worker_filter  # noqa: E402


def test_library_exports_every_declared_symbol():
    header = open(os.path.join(ROOT, "include", "cnmf_b200.h")).read()
    declared = set(re.findall(r"\b(cnmf_[a-z0-9_]+)\s*\(", header))
    declared -= {"cnmf_nmf_params"}
    assert len(declared) >= 20
    lib = ctypes.CDLL(_lib.LIB_PATH)
    for name in sorted(declared):
        assert hasattr(lib, name), "libcnmf_b200.so does not export %s" % name
    # and the Python binding table covers exactly the header
    assert set(_lib.SIGNATURES) == declared


def test_no_cpu_fallback_without_gpu():
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    from cnmf_b200.engine import Engine
    with pytest.raises(_lib.CnmfError, match="no CPU fallback"):
        Engine()


def test_host_rng_bit_exact_with_numpy_legacy_stream():
    lib = _lib.load()
    for seed, n, g, k in ((1, 50, 30, 3), (2 ** 31 - 2, 333, 77, 7), (123456789, 1000, 300, 13)):
        avg = 0.731
        ldw, ldh = n + 5, g + 3
        Wt = np.zeros((k, ldw), np.float32)
        H = np.zeros((k, ldh), np.float32)
        rc = lib.cnmf_random_init_host(seed, avg, n, g, k, _lib.ptr(Wt), ldw, _lib.ptr(H), ldh)
        assert rc == 0
        rng = np.random.RandomState(seed)        # sklearn _nmf.py:296-307: H first, then W
        H2 = np.abs(avg * rng.standard_normal((k, g))).astype(np.float32)
        W2 = np.abs(avg * rng.standard_normal((n, k))).astype(np.float32)
        assert np.array_equal(H[:, :g], H2)
        assert np.array_equal(Wt[:, :n], W2.T)
        assert not Wt[:, n:].any() and not H[:, g:].any()


def test_df_npz_codec_layout(tmp_path):
    df = pd.DataFrame(np.arange(6.0).reshape(2, 3), index=[1, 2], columns=["a", "b", "c"])
    fn = str(tmp_path / "x.df.npz")
    save_df_to_npz(df, fn)
    with np.load(fn, allow_pickle=True) as f:
        assert sorted(f.files) == ["columns", "data", "index"]      # cnmf.py:31-32
    back = load_df_from_npz(fn)
    assert back.equals(df)


def test_path_table_matches_reference(tmp_path):
    obj = cNMF(output_dir=str(tmp_path), name="run")
    assert obj.paths["iter_spectra"] % (7, 3) == os.path.join(str(tmp_path), "run", "cnmf_tmp", "run.spectra.k_7.iter_3.df.npz")
    assert obj.paths["consensus_usages__txt"] % (7, "0_1") == os.path.join(str(tmp_path), "run", "run.usages.k_7.dt_0_1.consensus.txt")
    # the reference's own table for the same name (oracle/make_golden.py path_table), relative to output_dir
    import json
    with open(os.path.join(ROOT, "tests", "golden", "path_table.json")) as f:
        ref = json.load(f)
    assert {key: os.path.relpath(p, str(tmp_path)) for key, p in obj.paths.items()} == ref


def test_worker_split_rules():
    assert list(worker_filter(range(10), 1, 3)) == [1, 4, 7]          # cnmf.py:52-53
    jobs = [shard_jobs(23, r, 4) for r in range(4)]
    assert sorted(sum(jobs, [])) == list(range(23))
    assert jobs[2] == list(worker_filter(range(23), 2, 4))


def test_prepare_matches_reference_outputs(tmp_path, golden):
    """prepare() on the golden counts reproduces what the reference wrote: HVG choice, seed table, solver."""
    counts = golden["counts"].astype(np.float64)
    df = pd.DataFrame(counts, index=["c%d" % i for i in range(counts.shape[0])],
                      columns=["g%d" % i for i in range(counts.shape[1])])
    fn = str(tmp_path / "counts.df.npz")
    save_df_to_npz(df, fn)
    obj = cNMF(output_dir=str(tmp_path), name="p")
    beta = golden["beta_loss_arg"]
    import warnings
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        obj.prepare(fn, components=list(golden["ks"]), n_iter=int(golden["n_iter"]), seed=int(golden["seed"]),
                    beta_loss=beta, num_highvar_genes=len(golden["hvg_idx"]), densify=True)
    hvgs = open(obj.paths["nmf_genes_list"]).read().split("\n")
    assert [int(g[1:]) for g in hvgs] == list(golden["hvg_idx"])
    table = load_df_from_npz(obj.paths["nmf_replicate_parameters"])
    assert np.array_equal(table[["n_components", "iter", "nmf_seed"]].values.astype(np.int64), golden["table"])
    import yaml
    kw = yaml.load(open(obj.paths["nmf_run_parameters"]), Loader=yaml.FullLoader)
    assert kw["solver"] == golden["solver"] and kw["tol"] == 1e-4 and kw["max_iter"] == 1000
    from cnmf_b200 import io as cio
    norm = cio.read_matrix(obj.paths["normalized_counts"])
    assert np.allclose(norm.X, golden["X"], rtol=1e-12, atol=0)
    stats = load_df_from_npz(obj.paths["tpm_stats"])
    assert np.allclose(stats["__std"].values, golden["tpm_std"], rtol=1e-12)


_GLOO_SCRIPT = r"""
import os, sys
import numpy as np
sys.path.insert(0, %(root)r)
from cnmf_b200.parallel import init_process_group, allgather_spectra, shard_jobs, dist_info
dist = init_process_group("gloo")
rank, world, _ = dist_info()
ks = [3, 3, 3, 4, 4, 4, 5]
G = 11
def spec(j):   # deterministic content per job
    return (np.arange(ks[j] * G, dtype=np.float32).reshape(ks[j], G) + 1000 * j)
jobs = shard_jobs(len(ks), rank, world)
full = allgather_spectra([spec(j) for j in jobs], jobs, ks, G)
ok = all(np.array_equal(full[j], spec(j)) for j in range(len(ks)))
dist.barrier()
print("RANK%%d_OK=%%s" %% (rank, ok))
dist.destroy_process_group()
"""


def test_allgather_spectra_gloo_world2(tmp_path):
    script = tmp_path / "gloo_case.py"
    script.write_text(_GLOO_SCRIPT % {"root": ROOT})
    env = dict(os.environ, MASTER_ADDR="127.0.0.1", MASTER_PORT="29533", WORLD_SIZE="2")
    procs = []
    for r in range(2):
        e = dict(env, RANK=str(r), LOCAL_RANK=str(r))
        procs.append(subprocess.Popen([sys.executable, str(script)], env=e, stdout=subprocess.PIPE, stderr=subprocess.STDOUT))
    outs = [p.communicate(timeout=180)[0].decode() for p in procs]
    for r, o in enumerate(outs):
        assert "RANK%d_OK=True" % r in o, o


def _fake_run(tmp_path, ks=(3,), n_iter=4, genes=6):
    """A cNMF directory with a params table and hand-written per-restart spectra files (no GPU needed)."""
    obj = cNMF(output_dir=str(tmp_path), name="fake")
    rp, kw = obj.get_nmf_iter_params(ks=list(ks), n_iter=n_iter, random_state_seed=3, beta_loss="frobenius")
    obj.save_nmf_iter_params(rp, kw)
    cols = ["g%d" % i for i in range(genes)]
    for _, p in rp.iterrows():
        k, it = int(p["n_components"]), int(p["iter"])
        df = pd.DataFrame(np.full((k, genes), float(it)), index=np.arange(1, k + 1), columns=cols)
        save_df_to_npz(df, obj.paths["iter_spectra"] % (k, it))
    return obj, rp


def test_combine_layout_and_missing_files(tmp_path):
    """combine_nmf (cnmf.py:748-773): row labels iter%d_topic%d, iter-major order, missing-file semantics."""
    obj, rp = _fake_run(tmp_path)
    merged = obj.combine_nmf(3)
    assert list(merged.index[:4]) == ["iter0_topic1", "iter0_topic2", "iter0_topic3", "iter1_topic1"]
    assert merged.shape == (12, 6) and (merged.iloc[3:6].values == 1.0).all()
    assert load_df_from_npz(obj.paths["merged_spectra"] % 3).equals(merged)
    os.remove(obj.paths["iter_spectra"] % (3, 2))
    with pytest.raises(FileNotFoundError):
        obj.combine_nmf(3)
    m2 = obj.combine_nmf(3, skip_missing_files=True)
    assert m2.shape == (9, 6) and "iter2_topic1" not in m2.index
    obj.combine(components=3, skip_missing_files=True)      # int / list / None forms of `components` (cnmf.py:474-480)
    obj.combine(components=[3], skip_missing_files=True)


def test_completed_ledger_and_skip(tmp_path):
    """update_nmf_iter_params / skip_completed_runs bookkeeping (cnmf.py:605-616, 636-651, 729-733)."""
    obj, rp = _fake_run(tmp_path, n_iter=3)
    assert not rp["completed"].any()                      # table was built before the files existed
    obj.update_nmf_iter_params()
    rp2 = load_df_from_npz(obj.paths["nmf_replicate_parameters"])
    assert rp2["completed"].all()
    os.remove(obj.paths["iter_spectra"] % (3, 1))
    obj.update_nmf_iter_params()
    rp3 = load_df_from_npz(obj.paths["nmf_replicate_parameters"])
    assert list(rp3["completed"]) == [True, False, True]
    todo = list(worker_filter(rp3.index[rp3["completed"] == False], 0, 1))   # noqa: E712
    assert todo == [1]
    import warnings
    with warnings.catch_warnings(record=True) as w:
        warnings.simplefilter("always")
        obj.get_nmf_iter_params(ks=[3], n_iter=3, random_state_seed=3)
        assert any("already appear completed" in str(x.message) for x in w)


def test_solver_selection_rule():
    """cnmf.py:629-631: beta_loss='frobenius' -> 'cd' (the default); anything else keeps 'mu'."""
    import tempfile
    obj = cNMF(output_dir=tempfile.mkdtemp(), name="x")
    assert obj.get_nmf_iter_params([3], 1, 1, beta_loss="frobenius")[1]["solver"] == "cd"
    assert obj.get_nmf_iter_params([3], 1, 1, beta_loss=2.0)[1]["solver"] == "mu"
    from cnmf_b200.engine import make_params
    assert make_params(dict(solver="mu", beta_loss="kullback-leibler"), 10, 10, "tf32x3").beta_loss == 1
    assert make_params(dict(solver="mu", beta_loss="itakura-saito"), 10, 10, "tf32x3").beta_loss == 2
    assert make_params(dict(solver="cd", beta_loss="frobenius"), 10, 10, "tf32x3").beta_loss == 0
    with pytest.raises(ValueError):             # sklearn _nmf.py:1195-1199: 'cd' only handles frobenius
        make_params(dict(solver="cd", beta_loss="kullback-leibler"), 10, 10, "tf32x3")
    with pytest.raises(NotImplementedError):
        make_params(dict(solver="mu", beta_loss=0.5), 10, 10, "tf32x3")
    with pytest.raises(ValueError, match="Invalid init"):      # sklearn's message for an unknown init
        make_params(dict(solver="cd", init="svd"), 10, 10, "tf32x3")
    assert make_params(dict(solver="cd", init="nndsvd"), 10, 10, "tf32x3").solver == 1
    p = make_params(dict(solver="cd", alpha_W=0.5, alpha_H="same", l1_ratio=0.25, tol=1e-3, max_iter=7), 100, 40, "fp32")
    assert (p.solver, p.max_iter, p.tol) == (1, 7, 1e-3)
    assert p.l1_reg_W == 40 * 0.5 * 0.25 and p.l2_reg_H == 100 * 0.5 * 0.75      # sklearn _nmf.py:1249-1260


def test_precision_names_and_hvg_ranking_from_stats():
    """Host-side pieces of the f16x2 precision and of prepare(on_device=True) that need no GPU."""
    from cnmf_b200 import _lib
    from cnmf_b200.engine import precision_code, _params_precision, _DEFAULT_PRECISION
    from cnmf_b200.pipeline import _highvar_from_stats, _highvar_genes
    assert precision_code("f16x2") == _lib.PRECISION_F16X2 == 3 and _DEFAULT_PRECISION == _lib.PRECISION_F16X2
    # params.precision names the arithmetic class (split-operand tensor-core products): 1 for both tf32x3 and f16x2
    assert _params_precision(precision_code("f16x2")) == _params_precision(precision_code("tf32x3")) == _lib.PRECISION_TF32X3
    assert _params_precision(precision_code("tf32x3-general")) == _lib.PRECISION_TF32X3
    assert _params_precision(precision_code("fp32")) == _lib.PRECISION_FP32
    rng = np.random.RandomState(3)
    C = rng.poisson(rng.gamma(0.5, 2.0, size=(1, 400)), size=(300, 400)).astype(np.float64) + rng.poisson(0.05, size=(300, 400))
    C = C[:, C.sum(axis=0) > 0]
    T = C / C.sum(axis=1, keepdims=True) * 1e6
    a = _highvar_genes(T, 50)
    b = _highvar_from_stats(T.mean(axis=0), T.var(axis=0), 50)
    assert a.sum() == 50 and np.array_equal(a, b)


def test_fp16_two_piece_split_bounds():
    """The operand representation of the default precision, restated in numpy (what emit_f16_kernel / emit_tile_f16
    compute): a row divided by the power of two that puts its maximum in [2^14, 2^15), then hi = fp16(x),
    mid = fp16(x - hi).  Entries down to 2^-18 of the row maximum keep >= 21 significant bits like a tf32 pair; smaller
    ones are off by at most 2^-39 of the row maximum; integer counts <= 2048 are exact in fp16."""
    rng = np.random.RandomState(0)
    A = (np.abs(rng.standard_cauchy((64, 4096))) * 10.0 ** rng.uniform(-8, 8, size=(64, 1))).astype(np.float32).astype(np.float64)
    A[:, ::11] = 0.0
    rowmax = A.max(axis=1, keepdims=True)
    mant, exp = np.frexp(rowmax)                       # rowmax = mant * 2^exp, mant in [0.5, 1)
    sc = np.ldexp(1.0, exp - 15)
    x = A / sc
    assert x.max() < 2 ** 15 and (x.max(axis=1) >= 2 ** 14).all()
    hi = x.astype(np.float16).astype(np.float64)
    mid = (x - hi).astype(np.float16).astype(np.float64)
    assert np.isfinite(hi).all() and np.isfinite(mid).all()
    err = np.abs((hi + mid) * sc - A)
    big = x >= 2.0 ** -3                               # both pieces normal fp16 numbers
    assert (err[big] <= A[big] * 2.0 ** -21).all()     # two 11-bit pieces
    assert ((err / sc)[~big] <= 2.0 ** -25).all()      # subnormal `mid`: half an fp16 subnormal step, in scaled units ...
    assert ((err / rowmax)[~big] <= 2.0 ** -39).all()  # ... which is 2^-39 of a row maximum >= 2^14
    C = np.arange(0, 2049, dtype=np.float64)
    assert np.array_equal(C.astype(np.float16).astype(np.float64), C)
    # a product against integer counts: same error class as the tf32 pair
    X = rng.poisson(0.7, size=(4096, 32)).astype(np.float64)
    P = A @ X
    Pr = ((hi + mid) * sc) @ X
    assert np.abs(Pr - P).max() / np.abs(P).max() < 2e-7


def test_binding_table_matches_header_prototypes():
    """Every prototype in include/cnmf_b200.h has the same number of parameters as its ctypes signature, the ABI
    version constants agree, and struct cnmf_nmf_params has the size the ctypes mirror assumes."""
    header = open(os.path.join(ROOT, "include", "cnmf_b200.h")).read()
    header = re.sub(r"/\*.*?\*/", " ", header, flags=re.S)
    protos = re.findall(r"\b(?:int|long long|const char\*)\s+(cnmf_[a-z0-9_]+)\s*\(([^;{]*?)\)\s*;", header, flags=re.S)
    assert len(protos) >= 30
    for name, args in protos:
        args = args.strip()
        n = 0 if args in ("", "void") else len([a for a in args.split(",") if a.strip()])
        assert n == len(_lib.SIGNATURES[name][1]), (name, n, len(_lib.SIGNATURES[name][1]))
    ver = int(re.search(r"#define CNMF_B200_ABI_VERSION (\d+)", header).group(1))
    assert ver == _lib.ABI_VERSION == ctypes.CDLL(_lib.LIB_PATH).cnmf_abi_version()
    assert ctypes.sizeof(_lib.NmfParams) == 4 * 4 + 5 * 8 + 2 * 4


# ------------------------------------------------------------------------------------ round-2 host logic
def _counts_file(tmp_path, counts, name="counts.df.npz"):
    df = pd.DataFrame(counts.astype(np.float64), index=["c%d" % i for i in range(counts.shape[0])],
                      columns=["g%d" % i for i in range(counts.shape[1])])
    fn = str(tmp_path / name)
    save_df_to_npz(df, fn)
    return fn


def test_prepare_sparse_semantics_and_zero_std_rule(tmp_path):
    """Without --densify the reference converts text / npz input to CSR (cnmf.py:399-405) and scales the HVG
    matrix with sc.pp.scale(zero_center=False) (cnmf.py:538), which maps a zero standard deviation to 1; with
    --densify it divides by the std (cnmf.py:542).  The facade keeps both behaviours and stores CSR like the
    reference; the stored values are otherwise identical."""
    import warnings
    import scipy.sparse as sp
    from cnmf_b200 import io as cio
    from cnmf_b200.synth import make_counts
    counts = make_counts(300, 60, k_true=3, seed=2, libsize=300.0).astype(np.float64)
    counts[:, 5] = 1.0                         # a constant gene: zero variance
    genes = ["g%d" % i for i in range(counts.shape[1])]
    fn = _counts_file(tmp_path, counts)
    gf = str(tmp_path / "genes.txt")
    open(gf, "w").write("\n".join(genes[:30]))
    out = {}
    for densify in (False, True):
        obj = cNMF(output_dir=str(tmp_path), name="d%d" % densify)
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            obj.prepare(fn, components=[3], n_iter=2, seed=1, densify=densify, genes_file=gf)
        out[densify] = cio.read_matrix(obj.paths["normalized_counts"])
        assert sp.issparse(out[densify].X) == (not densify)
        assert sp.issparse(cio.read_matrix(obj.paths["tpm"]).X) == (not densify)
    Xs, Xd = out[False].X.toarray(), out[True].X
    keep = np.arange(30) != 5
    assert np.array_equal(Xs[:, keep], Xd[:, keep])
    assert np.array_equal(Xs[:, 5], np.ones(300))          # std 0 -> 1: the column keeps its counts
    assert not np.isfinite(Xd[:, 5]).any()                 # dense branch: 1 / 0, as the reference (it only warns)


def test_unsupported_options_are_refused_at_prepare(tmp_path):
    """K > 32 and an init scikit-learn does not know fail when the user states them (prepare / get_nmf_iter_params /
    the CLI), not in factorize; the NNDSVD family is accepted (cnmf.py:1252); a refit ignores `init` (no initialisation
    when update_H=False, sklearn _nmf.py:1223-1228)."""
    from cnmf_b200.engine import check_supported, make_params
    from cnmf_b200.synth import make_counts
    fn = _counts_file(tmp_path, make_counts(120, 40, k_true=3, seed=2, libsize=300.0))
    obj = cNMF(output_dir=str(tmp_path), name="u")
    with pytest.raises(ValueError, match=r"\[1, 32\]"):
        obj.prepare(fn, components=[5, 40], n_iter=2, seed=1, densify=True)
    with pytest.raises(ValueError, match="Invalid init"):
        obj.prepare(fn, components=[5], n_iter=2, seed=1, densify=True, init="svd")
    with pytest.raises(ValueError, match=r"\[1, 32\]"):
        obj.get_nmf_iter_params(ks=[33], n_iter=2)
    with pytest.raises(NotImplementedError):
        check_supported([5], "random", 0.5)
    with pytest.raises(ValueError, match="Invalid init"):
        make_params(dict(solver="cd", init="svd"), 10, 10, "tf32x3")
    for init in ("random", "nndsvd", "nndsvda", "nndsvdar", None):
        check_supported([5], init, "frobenius")
    p = make_params(dict(solver="cd", init="svd"), 10, 10, "tf32x3", for_refit=True)
    assert p.solver == 1
    from cnmf_b200 import pipeline
    import sys
    argv = sys.argv
    try:
        sys.argv = ["cnmf", "prepare", "--init", "svd", "-c", fn, "-k", "5"]
        with pytest.raises(SystemExit):
            pipeline.main()
    finally:
        sys.argv = argv


def test_restart_groups_follow_the_memory_budget():
    from cnmf_b200.pipeline import plan_groups
    ks = [5] * 4 + [6] * 4 + [13] * 3
    assert plan_groups(ks, 10 ** 9) == [(0, len(ks))]
    groups = plan_groups(ks, 20)
    assert groups[0] == (0, 4) and groups[-1][1] == len(ks)
    assert all(sum(ks[a:b]) <= 20 or b - a == 1 for a, b in groups)
    assert [a for a, _ in groups][1:] == [b for _, b in groups][:-1]      # consecutive, nothing skipped
    assert plan_groups([40], 10) == [(0, 1)] and plan_groups([], 10) == []


def test_kmeans_draws_are_data_independent_and_in_sklearn_order():
    """cnmf_kmeans_fit receives every random number k-means++ will use up front.  That is only legitimate if the count
    and order of the draws do not depend on the data: consume the pre-drawn numbers in a numpy restatement of
    sklearn's k-means++ (SK/cluster/_kmeans.py:180-278) and check the chosen centres against sklearn's own
    kmeans_plusplus for the same RandomState, run after run."""
    from sklearn.cluster import kmeans_plusplus
    from cnmf_b200.consensus import _kmeans_draws
    rng0 = np.random.RandomState(3)
    X = np.abs(rng0.randn(240, 30)) + np.repeat(np.eye(6, 30) * 4, 40, axis=0)
    k, n_init = 6, 4
    first, unif, n_trials = _kmeans_draws(np.random.RandomState(1), X.shape[0], k, n_init)
    assert n_trials == 2 + int(np.log(k))
    ref_rng = np.random.RandomState(1)
    x_sq = (X * X).sum(axis=1)
    for t in range(n_init):
        _, ref_idx = kmeans_plusplus(X, k, random_state=ref_rng, x_squared_norms=x_sq)
        idx = [int(first[t])]
        closest = ((X - X[idx[0]]) ** 2).sum(axis=1)
        pot = closest.sum()
        for c in range(1, k):
            cand = np.searchsorted(np.cumsum(closest), unif[t, c - 1] * pot)
            np.clip(cand, None, len(closest) - 1, out=cand)
            d = np.minimum(closest, ((X[None, :, :] - X[cand][:, None, :]) ** 2).sum(axis=2))
            best = int(np.argmin(d.sum(axis=1)))
            pot, closest = d[best].sum(), d[best]
            idx.append(int(cand[best]))
        assert idx == list(ref_idx), (t, idx, list(ref_idx))


def test_slab_layout_matches_the_worker_filter_rule():
    """parallel._slab_layout (cached) against the definition: rank r owns the jobs idx % world == r (cnmf.py:52-53), its
    slab holds their spectra in job order, every slab padded to the largest per-rank row count."""
    from cnmf_b200.parallel import _slab_layout, shard_jobs
    ks_all = [k for k in (5, 7, 13, 6) for _ in range(11)]
    for world in (1, 2, 3, 8):
        rows_per_rank, max_rows, first_row, per_rank = _slab_layout(ks_all, world)
        assert per_rank == [shard_jobs(len(ks_all), r, world) for r in range(world)]
        assert rows_per_rank == [sum(ks_all[j] for j in jobs) for jobs in per_rank]
        assert max_rows == max(rows_per_rank)
        seen = set()
        for r, jobs in enumerate(per_rank):
            o = 0
            for j in jobs:
                assert first_row[j] == r * max_rows + o
                rows = set(range(first_row[j], first_row[j] + ks_all[j]))
                assert not (rows & seen)
                seen |= rows
                o += ks_all[j]
        assert _slab_layout(list(ks_all), world) is _slab_layout(tuple(ks_all), world)      # cached by value


def test_symmetric_gram_plan_covers_every_entry_once():
    """Index arithmetic of the update kernels' symmetric Gram (nmf_kernels.cu: SymGramMap, sym_gram_accumulate's block
    lists, sym_gram_plan), restated: the 10 blocks on or above the diagonal go 3 + 3 + 3 + 1 to the four warps; every
    entry (row, i) of the KP x KP Gram receives exactly one sum, read from a scratch slot that its owner warp wrote, and
    the mirror image of an entry reads the same slot."""
    lists = {0: [(0, 0), (0, 1), (0, 2)], 1: [(0, 3), (1, 1), (1, 2)], 2: [(1, 3), (2, 2), (2, 3)], 3: [(3, 3)]}

    def owner(bi, bj):
        idx = bi * 4 + bj - (bi * (bi + 1)) // 2
        return idx // 3, idx % 3

    for w, blocks in lists.items():                     # the compile-time lists and the closed form agree
        for slot, (bi, bj) in enumerate(blocks):
            assert owner(bi, bj) == (w, slot)
    assert sorted(b for bl in lists.values() for b in bl) == [(i, j) for i in range(4) for j in range(i, 4)]

    threads = 128
    for KP in (12, 16):
        RB = KP // 4
        stride = 3 * RB * RB + 1
        assert threads * stride <= KP * 512             # the scratch aliases the KP x 512 tile
        nup = KP * (KP + 1) // 2
        written = {}
        slots = set()
        for t in range(nup):
            row, rem = 0, t
            while row < KP - 1 and rem >= KP - row:
                rem -= KP - row
                row += 1
            i = row + rem
            assert row <= i < KP
            w, slot = owner(row // RB, i // RB)
            src = (w * 32) * stride + (slot * RB + row % RB) * RB + i % RB
            assert slot < len(lists[w]) and (slot * RB + row % RB) * RB + i % RB < stride - 1
            assert src not in slots                     # one distinct slot per distinct entry
            slots.add(src)
            for e in {row * KP + i, i * KP + row}:
                assert e not in written
                written[e] = src
        assert sorted(written) == list(range(KP * KP))
        for row in range(KP):
            for i in range(KP):
                assert written[row * KP + i] == written[i * KP + row]


def test_nndsvd_starting_factors_equal_scikit_learns():
    """cnmf_b200.nndsvd (numpy / scipy.linalg restatement of SK/decomposition/_nmf.py:309-369 and of randomized_svd,
    SK/utils/extmath.py) against scikit-learn's own `_initialize_nmf` -- what the reference's call with init='nndsvd'
    (cnmf.py:672, 1252) starts from: bit-identical in float64 (the dtype the reference runs in), dense and CSR, tall
    and wide; the packed layout handed to cnmf_factorize_init holds W^T rows then H rows per restart."""
    import scipy.sparse as sp
    from sklearn.decomposition._nmf import _initialize_nmf
    from cnmf_b200.engine import nndsvd_starts
    from cnmf_b200.nndsvd import nndsvd_init, resolve_init
    rng = np.random.RandomState(0)
    for shape in ((400, 200), (150, 300)):
        X = rng.poisson(1.0, size=shape).astype(np.float64) / (1.0 + rng.rand(shape[1]))
        for init in ("nndsvd", "nndsvda", "nndsvdar"):
            for k, seed in ((5, 14), (13, 123456)):
                W0, H0 = _initialize_nmf(X, k, init=init, random_state=seed)
                W1, H1 = nndsvd_init(X, k, seed, init)
                assert np.array_equal(W0, W1) and np.array_equal(H0, H1), (shape, init, k)
        X32 = X.astype(np.float32)
        W0, H0 = _initialize_nmf(X32, 7, init="nndsvd", random_state=3)
        W1, H1 = nndsvd_init(X32, 7, 3, "nndsvd")
        assert W1.dtype == np.float32 and np.abs(W0 - W1).max() <= 4e-7 * np.abs(W0).max()
        assert np.abs(H0 - H1).max() <= 4e-7 * np.abs(H0).max()
    Xs = sp.csr_matrix(rng.poisson(0.3, size=(300, 120)).astype(np.float64))
    W0, H0 = _initialize_nmf(Xs, 6, init="nndsvd", random_state=3)
    W1, H1 = nndsvd_init(Xs, 6, 3, "nndsvd")
    assert np.array_equal(W0, W1) and np.array_equal(H0, H1)
    # packed starts of a mixed batch
    X = rng.poisson(1.0, size=(120, 60)).astype(np.float64)
    ks, seeds = [3, 5, 4], [11, 12, 13]
    Wp, Hp = nndsvd_starts(X, ks, seeds, "nndsvd")
    assert Wp.shape == (12, 120) and Hp.shape == (12, 60) and Wp.dtype == np.float32
    o = 0
    for k, seed in zip(ks, seeds):
        W0, H0 = _initialize_nmf(X, k, init="nndsvd", random_state=seed)
        assert np.array_equal(Wp[o:o + k], W0.T.astype(np.float32)) and np.array_equal(Hp[o:o + k], H0.astype(np.float32))
        o += k
    assert resolve_init(None, 5, 100, 50) == "nndsvda" and resolve_init(None, 60, 100, 50) == "random"
    with pytest.raises(ValueError, match="can only be used"):
        resolve_init("nndsvd", 60, 100, 50)
