#!/usr/bin/env python
"""GPU bring-up probe (not a pytest file): run one stage per process so that a hung kernel
only costs its own `timeout`.  Usage on the GPU box:

    for s in gemm_fp32 gemm_tf32 nmf_fp32 nmf_tf32 perf; do timeout 300 python tests/gpu_probe.py $s; done
"""
import json
import os
import sys
import time
import warnings

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

from cnmf_b200.engine import Engine  # noqa: E402
from cnmf_golden import load_golden  # noqa: E402


def rel(a, b):
    return float(np.linalg.norm(a.astype(np.float64) - b) / np.linalg.norm(b))


def stage_gemm(precision):
    eng = Engine()
    rng = np.random.RandomState(0)
    shapes = [(128, 256, 32, 1), (128, 256, 64, 1), (128, 256, 2048, 1), (256, 512, 128, 1), (200, 300, 100, 1),
              (7, 1000, 500, 1), (70, 40, 33, 1), (1000, 2000, 2000, 1), (300, 500, 4000, 4), (1000, 2000, 20000, 9)]
    for (M, N, K, sp) in shapes:
        A = np.abs(rng.randn(M, K)).astype(np.float32)
        B = np.abs(rng.randn(N, K)).astype(np.float32)
        C, _ = eng.gemm_abt(A, B, precision=precision, splits=sp)
        ref = A.astype(np.float64) @ B.astype(np.float64).T
        bad = int(np.isnan(C).sum())
        print("gemm %s M=%d N=%d K=%d splits=%d rel=%.3e maxabs=%.3e nan=%d" % (
            precision, M, N, K, sp, rel(C, ref), float(np.abs(C - ref).max()), bad), flush=True)
    # signed inputs as well (the OLS projection uses centred usages)
    A = rng.randn(64, 1000).astype(np.float32)
    B = rng.randn(300, 1000).astype(np.float32)
    C, _ = eng.gemm_abt(A, B, precision=precision)
    print("gemm %s signed rel=%.3e" % (precision, rel(C, A.astype(np.float64) @ B.astype(np.float64).T)), flush=True)


def stage_nmf(precision):
    eng = Engine()
    for tag in ("sim_mu", "sim_cd"):
        g = load_golden(tag)
        ds = eng.dataset(g["X"], precision=precision)
        kw = dict(solver=g["solver"], tol=1e-4, max_iter=1000, alpha_W=0.0, alpha_H=0.0, l1_ratio=0.0)
        table = g["table"]
        t0 = time.time()
        sp, us, n_iter, err = ds.factorize(table[:, 0], table[:, 2], kw, return_usages=True)
        dt = time.time() - t0
        worst = 0.0
        for r, (k, it, seed) in enumerate(table):
            ref = g["merged_k%d" % k][it * k:(it + 1) * k]
            worst = max(worst, rel(sp[r], ref))
        print("nmf %s %s: %d restarts in %.3fs, worst rel-L2 vs reference spectra %.3e, n_iter %s" % (
            precision, tag, len(table), dt, worst, n_iter.tolist()), flush=True)
        from oracle import nmf_ref
        its = [nmf_ref.nmf(g["X"], int(k), int(seed), solver=g["solver"])[2] for (k, it, seed) in table]
        print("   oracle n_iter %s  match=%s" % (its, its == n_iter.tolist()), flush=True)
        # refit
        k = int(g["ks"][0])
        H = g["cspectra_k%d" % k]
        W, it, e = ds.refit(H, kw)
        Wr, itr = nmf_ref.refit(g["X"], H, g["solver"])
        print("   refit: n_iter %d (oracle %d) rel %.3e err %.6f (oracle %.6f)" % (
            it, itr, rel(W, Wr), e, nmf_ref.frobenius_error(g["X"], Wr, H)), flush=True)


def stage_gemmperf():
    eng = Engine()
    rng = np.random.RandomState(0)
    for name, (M, N, K, sp) in {"XHt_c2": (1000, 20000, 2000, 1), "WtX_c2": (1000, 2000, 20000, 9)}.items():
        A = np.abs(rng.randn(M, K)).astype(np.float32)
        B = np.abs(rng.randn(N, K)).astype(np.float32)
        C, ms = eng.gemm_abt(A, B, precision="tf32x3", splits=sp, reps=10)
        ref = A.astype(np.float64) @ B.astype(np.float64).T
        print("gemmperf %s: %.3f ms %.1f algo TFLOP/s rel=%.3e" % (
            name, ms, 2.0 * M * N * K / ms / 1e9, rel(C, ref)), flush=True)


def stage_c3():
    """BASELINE configs[2] on ONE GPU: 50k x 2k, K = 5..13 x 100 restarts (mixed K in one batch)."""
    from cnmf_b200.synth import make_counts, normalise, restart_table
    from oracle import nmf_ref
    eng = Engine()
    t0 = time.time()
    X, _ = normalise(make_counts(50000, 2000, k_true=12))
    rows = restart_table(list(range(5, 14)), 100)
    print("c3 data %s in %.1fs, %d restarts, sum K = %d" % (X.shape, time.time() - t0, len(rows), sum(r[0] for r in rows)), flush=True)
    kw = dict(solver="mu", tol=1e-4, max_iter=1000)
    ds = eng.dataset(X)
    print("c3 dataset exact=%s f16=%s" % (ds.exact, ds.f16), flush=True)
    for rep in range(2):
        eng.profile(True)
        l0 = eng.launch_count
        t1 = time.time()
        sp, _, n_iter, err = ds.factorize([r[0] for r in rows], [r[2] for r in rows], kw)
        dt = time.time() - t1
        ms, nl, fl = eng.profile_get()
        print("c3 rep %d: factorize %.2fs -> %.1f restarts/s; n_iter mean %.1f max %d; gemm %.0f ms (%d launches, %.1f algo TF/s); %d launches" % (
            rep, dt, len(rows) / dt, n_iter.mean(), n_iter.max(), ms, nl, fl / ms / 1e9 if ms else 0, eng.launch_count - l0), flush=True)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        for r in (0, 450, 899):
            t3 = time.time()
            W, H, it = nmf_ref.nmf(X.astype(np.float64), rows[r][0], rows[r][2], solver="mu")
            print("   oracle restart %d (K=%d): n_iter %d (gpu %d) rel-L2 %.3e  cpu %.1fs" % (
                r, rows[r][0], it, n_iter[r], rel(sp[r], H), time.time() - t3), flush=True)


def stage_consensus_c4():
    """BASELINE configs[3] consensus sizes: R = 4000 stacked spectra (K=20 x 200 restarts) x 2000 genes,
    density_threshold 0.01-style tight clusters + outliers; refits on 68k x 2k.  GPU vs the reference's sklearn path."""
    from cnmf_b200 import consensus as cs
    from cnmf_b200.synth import make_counts, normalise
    from oracle import reference_path, nmf_ref
    eng = Engine()
    rng = np.random.RandomState(11)
    K, R, G = 20, 4000, 2000
    cen = np.abs(rng.gamma(0.3, 1.0, size=(K, G)))
    pts = np.vstack([c * (1 + 0.02 * rng.randn(190, G)) for c in cen] + [np.abs(rng.gamma(0.3, 1.0, size=(200, G)))])
    pts = np.abs(pts)[rng.permutation(R)]
    t0 = time.time()
    dens_r, keep_r, labels_r, med_r = reference_path.consensus_cluster(pts, K, density_threshold=0.1)
    t_ref = time.time() - t0
    for rep in range(2):
        t0 = time.time()
        S = cs.SpectraMatrix(eng, pts).l2_normalize()
        dens, _ = S.local_density(int(0.3 * R / K))
        t1 = time.time()
        keep = dens < 0.1
        S2 = S.take_rows(np.where(keep)[0])
        labels, labels_t, inertia, _ = cs.kmeans(S2, K)
        t2 = time.time()
        med = cs.cluster_medians(S2, labels_t, K)
        t3 = time.time()
        sil = cs.silhouette(S2, labels, labels_t, K)
        t4 = time.time()
    from sklearn.metrics import silhouette_score
    l2 = (pts.T / np.sqrt((pts ** 2).sum(1))).T
    sil_r = silhouette_score(l2[keep_r], labels_r)
    print("consensus_c4: reference (sklearn, %d cores) %.2fs | gpu: l2+density %.3fs kmeans %.3fs median %.3fs silhouette %.3fs" % (
        os.cpu_count(), t_ref, t1 - t0, t2 - t1, t3 - t2, t4 - t3), flush=True)
    print("   density rel %.2e keep equal %s labels equal %s medians rel %.2e silhouette %.6f vs %.6f" % (
        rel(dens, dens_r), np.array_equal(keep, keep_r), np.array_equal(labels, labels_r), rel(med, med_r), sil, sil_r), flush=True)
    # refit on the c4 data matrix
    X, _ = normalise(make_counts(68000, 2000, k_true=20))
    ds = eng.dataset(X)
    H = np.abs(rng.gamma(0.3, 1.0, size=(K, X.shape[1])))
    H /= H.sum(1, keepdims=True)
    for solver in ("cd", "mu"):
        kw = dict(solver=solver, tol=1e-4, max_iter=1000)
        ds.refit(H, kw)
        t0 = time.time()
        W, it, err = ds.refit(H, kw)
        t1 = time.time()
        Wr, itr = nmf_ref.refit(X.astype(np.float64), H, solver)
        t2 = time.time()
        print("   refit %s 68k x 2k K=20: gpu %.3fs (%d its) oracle %.1fs (%d its) rel %.2e exact=%s" % (
            solver, t1 - t0, it, t2 - t1, itr, rel(W, Wr), ds.exact), flush=True)


def stage_consensus_kernels():
    """One pass over the consensus kernels at BASELINE configs[3] size (R = 4000 x 2000, K = 20) -- the launch set
    `ncu --set full -k regex:...` captures for the HBM roofline table in profiles/."""
    from cnmf_b200 import consensus as cs
    eng = Engine()
    rng = np.random.RandomState(11)
    K, R, G = 20, 4000, 2000
    cen = np.abs(rng.gamma(0.3, 1.0, size=(K, G)))
    pts = np.vstack([c * (1 + 0.02 * rng.randn(190, G)) for c in cen] + [np.abs(rng.gamma(0.3, 1.0, size=(200, G)))])
    pts = np.abs(pts)[rng.permutation(R)]
    S = cs.SpectraMatrix(eng, pts).l2_normalize()
    dens, _ = S.local_density(int(0.3 * R / K))
    keep = dens < 0.1
    S2 = S.take_rows(np.where(keep)[0])
    labels, labels_t, inertia, _ = cs.kmeans(S2, K, n_init=1)
    med = cs.cluster_medians(S2, labels_t, K)
    sil = cs.silhouette(S2, labels, labels_t, K)
    print("consensus_kernels: kept %d of %d, inertia %.4f, silhouette %.4f" % (keep.sum(), R, inertia, sil), flush=True)


def stage_big():
    """BASELINE configs[3] and [4] factorize sizes on ONE GPU (capacity / sanity: no oracle at this size):
    c4 68k x 2k, K=20 x 200 restarts; c5 200k x 5k, K=30 x 200 restarts."""
    from cnmf_b200.synth import make_counts, normalise, restart_table
    eng = Engine()
    for name, (n, g, k, nrest) in {"c4": (68000, 2000, 20, 200), "c5": (200000, 5000, 30, 200)}.items():
        t0 = time.time()
        X, _ = normalise(make_counts(n, g, k_true=max(12, k // 2)))
        rows = restart_table([k], nrest)
        t1 = time.time()
        ds = eng.dataset(X)
        eng.profile(True)
        t2 = time.time()
        sp, _, n_iter, err = ds.factorize([r[0] for r in rows], [r[2] for r in rows], dict(solver="mu", tol=1e-4, max_iter=1000))
        t3 = time.time()
        ms, nl, fl = eng.profile_get()
        import torch
        free, tot = torch.cuda.mem_get_info()
        normX = np.sqrt(float((X.astype(np.float64) ** 2).sum()))
        ok = bool(np.isfinite(err).all() and (err < normX).all() and all(np.isfinite(s).all() and (s >= 0).all() for s in sp))
        print("%s %s exact=%s: data %.0fs upload %.1fs factorize %.1fs -> %.1f restarts/s; n_iter mean %.0f max %d; gemm %.0f ms %.0f algo TF/s; "
              "err/||X|| in [%.4f, %.4f]; sane=%s; HBM used %.1f GB" % (
                  name, X.shape, ds.exact, t1 - t0, t2 - t1, t3 - t2, nrest / (t3 - t2), n_iter.mean(), n_iter.max(), ms,
                  fl / ms / 1e9 if ms else 0, err.min() / normX, err.max() / normX, ok, (tot - free) / 2 ** 30), flush=True)
        ds.close()
        del X


def stage_cd():
    """The reference's DEFAULT solver (cd) on the c2 workload."""
    from cnmf_b200.synth import make_counts, normalise, restart_table
    from oracle import reference_path
    eng = Engine()
    X, _ = normalise(make_counts(20000, 2000, k_true=12))
    rows = restart_table([10], 100)
    ds = eng.dataset(X)
    kw = dict(solver="cd", tol=1e-4, max_iter=1000)
    for rep in range(2):
        eng.profile(True)
        t0 = time.time()
        sp, _, n_iter, err = ds.factorize([r[0] for r in rows], [r[2] for r in rows], kw)
        dt = time.time() - t0
        ms, nl, fl = eng.profile_get()
        print("cd c2 rep %d: %.2fs -> %.1f restarts/s; n_iter mean %.1f max %d; gemm %.0f ms (%.1f algo TF/s)" % (
            rep, dt, len(rows) / dt, n_iter.mean(), n_iter.max(), ms, fl / ms / 1e9 if ms else 0), flush=True)
    spr, its, sec = reference_path.factorize(X, [(rows[0][0], rows[0][2]), (rows[1][0], rows[1][2])], "cd")
    print("   reference cd: %.2fs per restart (%d cores); n_iter %s vs gpu %s; rel-L2 %.2e %.2e" % (
        sec / 2, os.cpu_count(), its, n_iter[:2].tolist(), rel(sp[0], spr[0]), rel(sp[1], spr[1])), flush=True)


def stage_kl():
    """--beta-loss kullback-leibler on the c2 workload (streaming kernels, no GEMM)."""
    from cnmf_b200.synth import make_counts, normalise, restart_table
    from oracle import reference_path
    eng = Engine()
    X, _ = normalise(make_counts(20000, 2000, k_true=12))
    rows = restart_table([10], 100)
    ds = eng.dataset(X)
    for max_iter in (20, 1000):
        kw = dict(solver="mu", beta_loss="kullback-leibler", tol=1e-4, max_iter=max_iter)
        n0 = eng.launch_count
        t0 = time.time()
        sp, _, n_iter, err = ds.factorize([r[0] for r in rows], [r[2] for r in rows], kw)
        dt = time.time() - t0
        print("kl c2 max_iter %d: %.2fs -> %.1f restarts/s; n_iter mean %.1f max %d; %.2f ms per batched iteration; %d launches" % (
            max_iter, dt, len(rows) / dt, n_iter.mean(), n_iter.max(), 1e3 * dt / n_iter.max(), eng.launch_count - n0), flush=True)
    spr, its, sec = reference_path.factorize(X, [(rows[0][0], rows[0][2])], "mu", max_iter=50, beta_loss="kullback-leibler")
    kw = dict(solver="mu", beta_loss="kullback-leibler", tol=1e-4, max_iter=50)
    sp50, _, it50, _ = ds.factorize([rows[0][0]], [rows[0][2]], kw)
    print("   reference kl (50 iterations): %.2fs (%d cores) = %.3f s/iteration; n_iter %s vs gpu %s; rel-L2 %.2e" % (
        sec, os.cpu_count(), sec / its[0], its, it50.tolist(), rel(sp50[0], spr[0])), flush=True)


def stage_perf():
    eng = Engine()
    rng = np.random.RandomState(0)
    out = {}
    for name, (M, N, K, sp) in {"XHt_c2": (1000, 20000, 2000, 1), "WtX_c2": (1000, 2000, 20000, 9),
                                "XHt_c3": (8100, 50000, 2000, 1)}.items():
        A = np.abs(rng.randn(M, K)).astype(np.float32)
        B = np.abs(rng.randn(N, K)).astype(np.float32)
        for prec in ("tf32x3", "fp32"):
            if prec == "fp32" and M > 2000:
                continue
            _, ms = eng.gemm_abt(A, B, precision=prec, splits=sp, reps=5)
            tf = 2.0 * M * N * K / (ms * 1e-3) / 1e12
            out["%s_%s" % (name, prec)] = dict(ms=ms, algo_tflops=tf)
            print("perf gemm %s %s: %.3f ms  %.1f algorithmic TFLOP/s" % (name, prec, ms, tf), flush=True)
    from cnmf_b200.synth import make_counts, normalise, restart_table
    counts = make_counts(20000, 2000, k_true=12)
    X, _ = normalise(counts)
    rows = restart_table([10], 100)
    kw = dict(solver="mu", tol=1e-4, max_iter=1000)
    for prec in ("tf32x3", "fp32"):
        t0 = time.time()
        ds = eng.dataset(X, precision=prec)
        t1 = time.time()
        sp, _, n_iter, err = ds.factorize([r[0] for r in rows], [r[2] for r in rows], kw)
        t2 = time.time()
        out["c2_%s" % prec] = dict(upload_s=t1 - t0, factorize_s=t2 - t1, restarts_per_s=len(rows) / (t2 - t1),
                                   n_iter_mean=float(n_iter.mean()), n_iter_max=int(n_iter.max()))
        print("perf c2 %s: upload %.2fs factorize %.2fs -> %.1f restarts/s; n_iter mean %.1f max %d" % (
            prec, t1 - t0, t2 - t1, len(rows) / (t2 - t1), n_iter.mean(), n_iter.max()), flush=True)
        if prec == "tf32x3":
            from oracle import nmf_ref
            with warnings.catch_warnings():
                warnings.simplefilter("ignore")
                for r in (0, 1):
                    t3 = time.time()
                    W, H, it = nmf_ref.nmf(X.astype(np.float64), rows[r][0], rows[r][2], solver="mu")
                    print("   oracle restart %d: n_iter %d (gpu %d) rel-L2 %.3e  cpu %.1fs" % (
                        r, it, n_iter[r], rel(sp[r], H), time.time() - t3), flush=True)
        ds.close()
    os.makedirs(os.path.join(ROOT, "gpurun_out"), exist_ok=True)
    json.dump(out, open(os.path.join(ROOT, "gpurun_out", "probe_perf.json"), "w"), indent=1)


def stage_consensus():
    from cnmf_b200 import consensus as cs
    from oracle import consensus_ref as cr
    eng = Engine()
    for tag in ("sim_mu",):
        g = load_golden(tag)
        for k in g["ks"]:
            k = int(k)
            merged = g["merged_k%d" % k]
            S = cs.SpectraMatrix(eng, merged).l2_normalize()
            l2 = cr.l2_normalize_rows(merged)
            print("consensus k=%d l2 rel %.3e" % (k, rel(S.numpy(), l2)), flush=True)
            n_nb = int(0.3 * merged.shape[0] / k)
            dens, D = S.local_density(n_nb, return_dist=True)
            Dref = cr.euclidean_distances(l2)
            dref = cr.local_density(Dref, n_nb)
            print("   dist maxabs %.3e  density rel %.3e  (golden rel %.3e)" % (
                float(np.abs(D - Dref).max()), rel(dens, dref), rel(dens, g["density_k%d" % k])), flush=True)
            labels, labels_t, inertia, centers = cs.kmeans(S, k)
            lref, iref, cref = cr.kmeans(l2, k)
            print("   kmeans labels equal %s inertia %.6e vs %.6e" % (np.array_equal(labels, lref), inertia, iref), flush=True)
            med = cs.cluster_medians(S, labels_t, k)
            mref = cr.cluster_medians(l2, lref, k)
            print("   medians rel %.3e" % rel(med, mref), flush=True)
    # a bigger random case: R=3000 x G=2000, 12 clusters + outliers
    rng = np.random.RandomState(5)
    cen = np.abs(rng.randn(12, 2000))
    pts = np.vstack([c + 0.05 * np.abs(rng.randn(240, 2000)) for c in cen] + [np.abs(rng.randn(120, 2000))])
    S = cs.SpectraMatrix(eng, pts).l2_normalize()
    l2 = cr.l2_normalize_rows(pts)
    t0 = time.time()
    dens, _ = S.local_density(72)
    t1 = time.time()
    dref = cr.local_density(cr.euclidean_distances(l2), 72)
    print("big: density rel %.3e gpu %.3fs" % (rel(dens, dref), t1 - t0), flush=True)
    keep = dens < 0.5
    S2 = S.take_rows(np.where(keep)[0])
    t0 = time.time()
    labels, labels_t, inertia, _ = cs.kmeans(S2, 12)
    t1 = time.time()
    lref, iref, _ = cr.kmeans(l2[keep], 12)
    t2 = time.time()
    print("big: kmeans equal %s inertia %.6e/%.6e gpu %.2fs oracle %.2fs" % (
        np.array_equal(labels, lref), inertia, iref, t1 - t0, t2 - t1), flush=True)
    med = cs.cluster_medians(S2, labels_t, 12)
    print("big: medians rel %.3e" % rel(med, cr.cluster_medians(l2[keep], lref, 12)), flush=True)


if __name__ == "__main__":
    st = sys.argv[1]
    if st == "gemm_fp32":
        stage_gemm("fp32")
    elif st == "gemm_tf32":
        stage_gemm("tf32x3")
    elif st == "nmf_fp32":
        stage_nmf("fp32")
    elif st == "nmf_tf32":
        stage_nmf("tf32x3")
    elif st == "perf":
        stage_perf()
    elif st == "consensus":
        stage_consensus()
    elif st == "gemmperf":
        stage_gemmperf()
    elif st == "c3":
        stage_c3()
    elif st == "consensus_c4":
        stage_consensus_c4()
    elif st == "kl":
        stage_kl()
    elif st == "cd":
        stage_cd()
    elif st == "big":
        stage_big()
    elif st == "consensus_kernels":
        stage_consensus_kernels()
