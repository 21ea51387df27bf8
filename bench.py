#!/usr/bin/env python
"""bench.py -- restarts/sec of the batched factorize hot path on B200 (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload c3|c2] [--scaling strong|weak]
                    [--dump-outputs DIR]

Workload (default c3 = BASELINE.json configs[2], the north-star target; it fits one B200): synthetic 50 000 cells x
2 000 HVG, K = 5..13 x 100 seeds = 900 restarts, solver 'mu' (Frobenius), tol 1e-4, max_iter 1000 -- the reference's
own restart loop (cnmf.py:735-745) with its own seed rule (cnmf.py:597-610).  `--workload c2` = configs[1]
(20 000 x 2 000, K=10 x 100).  One "step" = factorizing the WHOLE job table to convergence.

With N > 1 ranks (torchrun) every rank holds a replica of X and takes the jobs idx % N == rank of the SAME table
(cnmf.py:52-53; `--scaling strong`, the default: total work fixed) and the step ends with the one collective of the
path, the NCCL all-gather of the spectra slabs (cnmf_allgather_spectra) that replaces `combine`.  `--scaling weak`
gives every rank its own full table instead.  The timed call is cnmf_b200.parallel.factorize_sharded -- the function
the facade's multi-GPU factorize uses -- not a bench-only path.

Printed JSON (rank 0): `value` = restarts/s with X resident in HBM (random init generated on the device, spectra
left in HBM); `e2e` = the same through the public call with HOST buffers (H2D of X and device-side preparation, the
solve, the all-gather, D2H of all spectra inside the timed region); `with_consensus` = factorize + all-gather +
cNMF.consensus numerics for every K (Ks sharded over the ranks) with its HBM roofline; `roofline` = the dominant
kernel (the batched tcgen05 GEMM) from CUDA events inside the timed region (recorded on rank 0); `cpu_baseline` / `cd_default` = the
reference's own scikit-learn call timed on the host cores.
`--dump-outputs DIR` writes what the last timed step returned (see --help); inputs are synthetic and seeded, so two
builds run with the same arguments can be compared output for output.
`--impl reference` times the reference's CPU implementation (oracle/reference_path.py: the reference's call
sequence on scikit-learn, float64): one restart of the job table to convergence per step, K cycling through the
sweep, on the best thread count of a short sweep.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "NMF restarts/sec on NxG counts, K-sweep x100 seeds, 1/2/4/8 B200 vs sklearn CPU"
WORKLOADS = {
    "c3": dict(n_cells=50000, n_genes=2000, ks=list(range(5, 14)), n_iter=100,
               desc="c3 = BASELINE configs[2] (north-star target): synthetic 50000x2000 (Poisson counts / gene std), "
                    "K=5..13 x 100 seeds = 900 restarts"),
    "c2": dict(n_cells=20000, n_genes=2000, ks=[10], n_iter=100,
               desc="c2 = BASELINE configs[1]: synthetic 20000x2000 (Poisson counts / gene std), K=10 x 100 seeds"),
}
NMF_KW = dict(solver="mu", beta_loss=2.0, tol=1e-4, max_iter=1000, init="random", alpha_W=0.0, alpha_H=0.0, l1_ratio=0.0)
CD_KW = dict(NMF_KW, solver="cd", beta_loss="frobenius")


def workload_config(name, world, scaling, n_jobs):
    w = WORKLOADS[name]
    return {"workload": w["desc"] + ", solver=mu (Frobenius), tol=1e-4, max_iter=1000",
            "restarts_total": n_jobs, "scaling": scaling,
            "parallelism": "job table idx %% %d == rank (cnmf.py:52-53), X replicated, one NCCL all-gather of spectra" % world,
            "l2": "inputs larger than L2 (X forms > 1 GB, factors > 1 GB per GPU)"}


def make_data(name, want_tpm=False):
    from cnmf_b200.synth import make_counts, normalise
    w = WORKLOADS[name]
    counts = make_counts(w["n_cells"], w["n_genes"], k_true=12, seed=0)
    X, keep = normalise(counts, np.float32)
    if not want_tpm:
        return X, None, None
    c = counts[:, keep].astype(np.float64)
    tpm = c / c.sum(axis=1, keepdims=True) * 1e6              # cnmf.py:245-251 over the same genes (SURVEY 8d)
    return X, np.ascontiguousarray(tpm, dtype=np.float32), tpm.std(axis=0, ddof=0)


def job_table(name, world, scaling):
    from cnmf_b200.synth import restart_table
    w = WORKLOADS[name]
    n_iter = w["n_iter"] * (world if scaling == "weak" else 1)
    rows = restart_table(w["ks"], n_iter, seed=14)
    return [r[0] for r in rows], [r[2] for r in rows], [r[1] for r in rows]


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.idx = gpu_index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.idx), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm = [float(r[1]) for r in self.rows if len(r) >= 8 and r[1].replace(".", "").isdigit()]
        mx = [float(r[2]) for r in self.rows if len(r) >= 8 and r[2].replace(".", "").isdigit()]
        reasons = set()
        for r in self.rows:
            if len(r) >= 8:
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[4:8]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
        busy = [c for c in sm if c > 0.5 * (max(mx) if mx else 1)] or sm
        return {"sm_mhz": float(np.median(busy)) if busy else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        m = json.load(open(p))
        return m.get("bf16_tflops_sustained", m.get("bf16_tflops")) / 2.0, \
            "MEASURED_PEAKS.json bf16_tflops_sustained/2 (dense TF32 = half the bf16 rate), of measured"
    return 1400.0 / 2.0, "fallback 1.4 PFLOP/s sustained bf16 / 2, of fallback"


def measured_hbm():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return float(json.load(open(p))["hbm_gbs"]), "MEASURED_PEAKS.json hbm_gbs (copy bandwidth), of measured"
    return 6650.0, "fallback 6.65 TB/s copy bandwidth, of fallback"


def host_threads():
    try:
        from threadpoolctl import threadpool_info
        return max([t.get("num_threads", 1) for t in threadpool_info()] + [1])
    except Exception:
        return os.cpu_count()


def best_thread_count(X, job, solver):
    """torchrun exports OMP_NUM_THREADS=1 and 128 BLAS threads oversubscribe a K ~ 10 problem: time 6 iterations of
    the reference call at a few thread counts and keep the fastest (reported in `cores`)."""
    from oracle import reference_path
    try:
        from threadpoolctl import threadpool_limits
    except Exception:
        return os.cpu_count(), {}
    ncpu = os.cpu_count() or 1
    cands = sorted({c for c in (8, 16, 32, 64, ncpu) if c <= ncpu} | {ncpu})
    probe = {}
    for c in cands:
        with threadpool_limits(limits=c):
            t0 = time.perf_counter()
            reference_path.factorize(X, [job], solver, max_iter=6)
            probe[c] = time.perf_counter() - t0
    return min(probe, key=probe.get), probe


def run_reference(args, rank, world):
    if rank != 0:
        return
    from oracle import reference_path
    from threadpoolctl import threadpool_limits
    X, _, _ = make_data(args.workload)
    X = X.astype(np.float64)                                   # cnmf.py:534
    ks, seeds, _ = job_table(args.workload, 1, "strong")
    n_per_k = WORKLOADS[args.workload]["n_iter"]
    n_k = len(WORKLOADS[args.workload]["ks"])
    # step i factorizes restart (K cycling through the sweep, iter i // n_k): the K mix of the table
    pick = [(i % n_k) * n_per_k + (i // n_k) % n_per_k for i in range(args.steps + args.warmup)]
    jobs = [(ks[j], seeds[j]) for j in pick]
    threads, probe = best_thread_count(X, jobs[0], "mu")
    its = []
    with threadpool_limits(limits=threads):
        for i in range(args.warmup):                           # warm-up: a few iterations of the same call
            reference_path.factorize(X, [jobs[i]], "mu", max_iter=3)
        t0 = time.perf_counter()
        for i in range(args.steps):
            sp, it, _ = reference_path.factorize(X, [jobs[args.warmup + i]], "mu")
            its += it
        dt = time.perf_counter() - t0
    if args.dump_outputs:                                      # the last step's restart
        write_outputs(args.dump_outputs, {"spectra": np.asarray(sp[0], np.float64),
                                          "n_iter": np.array(it, np.float64),
                                          "spectra_jobs": np.array([pick[-1]], np.float64)})
    val = args.steps / dt
    sample = ("1 restart of the job table per step to convergence (K cycling %s, reference seeds), sklearn "
              "non_negative_factorization MU float64 as cnmf.py:672 calls it; n_iter=%s; thread sweep (6 iterations): %s"
              % (WORKLOADS[args.workload]["ks"], its, {k: round(v, 2) for k, v in probe.items()}))
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": val, "unit": "restarts/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True,
        "scaling": args.scaling, "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": workload_config(args.workload, 1, args.scaling, len(ks)),
        "cpu_baseline": {"value": val, "unit": "restarts/s", "cores": threads, "kind": "port", "sample": sample},
        "e2e": {"value": val, "unit": "restarts/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }), flush=True)


DUMP_BYTES = 64 * 10 ** 6      # --dump-outputs writes at most this much


def dump_jobs(ks, n_genes, budget):
    """Jobs whose spectra --dump-outputs writes: all of them when they fit in `budget` bytes of fp32, else a fixed
    seeded random subset of whole restarts that does (the same subset for the same job table)."""
    size = [int(k) * n_genes * 4 for k in ks]
    if sum(size) <= budget:
        return list(range(len(ks)))
    pick, used = [], 0
    for j in np.random.RandomState(0).permutation(len(ks)):
        if used + size[j] <= budget:
            pick.append(int(j))
            used += size[j]
    return sorted(pick)


def write_outputs(out_dir, arrays):
    """arrays: name -> float32 / float64 array, written as out_dir/<name>.npy."""
    assert sum(a.nbytes for a in arrays.values()) <= DUMP_BYTES
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        assert a.dtype in (np.float32, np.float64), (name, a.dtype)
        np.save(os.path.join(out_dir, name + ".npy"), a)


def consensus_bytes(R, Rk, G, N, G_all, K, lloyd_iters, refit_iters):
    """Algorithmic bytes of one consensus(K) (SURVEY.md section 8d, fp32): C1 2RG, C2 RG, C3 R^2, C5 lloyd_iters*R'G,
    C6 R'G, C7 per refit NG (X once) + iters*2*N*K, C8 N*G_all."""
    b = 2 * R * G + R * G + R * R + lloyd_iters * Rk * G + Rk * G
    for n_rows, n_cols, it in refit_iters:
        b += n_rows * n_cols + it * 2 * n_rows * K
    b += N * G_all
    return 4.0 * b


def run_ours(args, rank, world, local):
    import torch
    import torch.distributed as dist
    from cnmf_b200 import consensus as cs
    from cnmf_b200.engine import Engine
    from cnmf_b200.parallel import SpectraComm, consensus_ks_of_rank, factorize_sharded, init_process_group
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: cnmf_b200 has no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local)
    init_process_group("nccl")
    dev = torch.device("cuda:%d" % local)
    wl = WORKLOADS[args.workload]

    X, tpm, tpm_std = make_data(args.workload, want_tpm=not args.no_consensus)
    Xpin = torch.from_numpy(X).pin_memory()
    Xnp = Xpin.numpy()
    ks_all, seeds_all, iters_all = job_table(args.workload, world, args.scaling)
    n_jobs = len(ks_all)
    eng = Engine(local)
    comm = SpectraComm(eng) if world > 1 else None
    # Python's cyclic collector walks every object of every imported package (torch, pandas, sklearn: ~10^6) when a
    # generation-2 collection fires -- 60-90 ms at a random point of a timed region (seen in tools/probe_stalls.py).
    # Everything alive now is set-up state: move it out of the collector's reach.
    import gc
    gc.collect()
    gc.freeze()

    def sync_all():
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize(dev)

    def max_over_ranks(v):
        t = torch.tensor([v], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # ---------------- device-resident arm: X already in HBM ----------------
    ds = eng.dataset(Xnp, precision=args.precision)
    passes = 2 if ds.exact else 3
    f16 = bool(ds.f16)
    ld_r, ld_c = ds.ld()

    def step_resident(kw=NMF_KW):
        return factorize_sharded(ds, ks_all, seeds_all, kw, comm)

    for _ in range(args.warmup):
        step_resident()
    clocks = ClockSampler(local)
    sync_all()
    if rank == 0:
        clocks.start()
    launches0 = eng.launch_count
    # per-launch CUDA events (the roofline's kernel times) on the rank that reports them; on the other ranks they would
    # only add their ~3 us per launch to a max-over-ranks time nobody reads them from
    eng.profile(rank == 0)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    sync_all()
    e0.record()
    for _ in range(args.steps):
        sharded, n_iter, my_jobs = step_resident()
    e1.record()
    sync_all()
    ms = max_over_ranks(e0.elapsed_time(e1))
    gemm_ms, gemm_launches, gemm_flops = eng.profile_get(0)
    upd_ms, upd_launches, upd_bytes = eng.profile_get(1)
    eng.profile(False)
    launches = eng.launch_count - launches0
    value = n_jobs * args.steps / (ms * 1e-3)

    dump = None
    if args.dump_outputs:              # what the last timed step returned: spectra of every job, n_iter of every job
        it_all = torch.zeros(n_jobs, dtype=torch.float64, device=dev)
        it_all[torch.as_tensor(my_jobs, dtype=torch.long, device=dev)] = torch.as_tensor(
            np.asarray(n_iter, np.float64), device=dev)
        if world > 1:
            dist.all_reduce(it_all)                            # every job belongs to exactly one rank
        if rank == 0:                                          # the gathered slab is the same on every rank
            jobs = dump_jobs(ks_all, X.shape[1], DUMP_BYTES - 16 * n_jobs)
            spectra = sharded.host()
            dump = {"spectra": np.vstack([spectra[j] for j in jobs]), "n_iter": it_all.cpu().numpy(),
                    "spectra_jobs": np.asarray(jobs, np.float64)}

    # ---------------- factorize + all-gather + consensus for every K (Ks sharded over the ranks) ----------------
    with_consensus = None
    if not args.no_consensus:
        tpm_ds = eng.dataset(tpm, precision=args.precision)
        ks_sorted = sorted(set(ks_all))
        my_ks = consensus_ks_of_rank(ks_sorted, rank, world)
        jobs_of_k = {k: [j for j in sorted(range(n_jobs), key=lambda j: iters_all[j]) if ks_all[j] == k] for k in ks_sorted}
        G = X.shape[1]
        hv_idx = np.arange(G)

        def step_consensus():
            t0 = time.perf_counter()
            sharded, _, _ = factorize_sharded(ds, ks_all, seeds_all, NMF_KW, comm)
            torch.cuda.synchronize(dev)
            t1 = time.perf_counter()
            work, per_k = 0.0, {}
            for k in my_ks:
                tk = time.perf_counter()
                cs.STATS.clear()
                res = cs.consensus_numerics(eng, sharded.matrix(eng, jobs_of_k[k]), k, ds, NMF_KW, density_threshold=0.5,
                                            tpm_ds=tpm_ds, hvg_idx=hv_idx, tpm_std_hvg=tpm_std)
                torch.cuda.synchronize(dev)
                per_k[k] = 1e3 * (time.perf_counter() - tk)
                R = len(jobs_of_k[k]) * k
                work += consensus_bytes(R, len(res["keep"]), G, X.shape[0], G, k, cs.STATS.get("lloyd_iters", 0),
                                        cs.STATS.get("refits", []))
            return t1 - t0, time.perf_counter() - t1, work, per_k

        step_consensus()                                                   # warm-up (allocations, caches)
        sync_all()
        n_c = args.steps
        t_all0 = time.perf_counter()
        acc = [0.0, 0.0, 0.0]
        per_k = {}
        for _ in range(n_c):
            tf, tc, work, per_k = step_consensus()
            acc[0] += tf; acc[1] += tc; acc[2] += work
        sync_all()
        t_total = max_over_ranks(time.perf_counter() - t_all0)
        t_cons = max_over_ranks(acc[1])
        hbm_peak, hbm_src = measured_hbm()
        w = torch.tensor([acc[2]], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(w, op=dist.ReduceOp.SUM)
        cons_gbs = float(w.item()) / (t_cons * world) / 1e9 if t_cons > 0 else 0.0
        with_consensus = {
            "value": n_jobs * n_c / t_total, "unit": "restarts/s", "steps": n_c,
            "ms_per_step": {"factorize_allgather": 1e3 * acc[0] / n_c, "consensus_all_k_max_rank": 1e3 * t_cons / n_c,
                            "total": 1e3 * t_total / n_c},
            "consensus_ks": {"all": ks_sorted, "rank0": my_ks, "rank0_ms_per_k": {str(k): round(v, 2) for k, v in per_k.items()}},
            "roofline": {"bound": "hbm", "achieved": cons_gbs, "peak": hbm_peak, "unit": "GB/s", "frac": cons_gbs / hbm_peak,
                         "traffic": None,
                         "note": "consensus stage only: algorithmic bytes of SURVEY.md 8d (C1 2RG, C2 RG, C3 R^2, C5 "
                                 "lloyd_iters*R'G, C6 R'G, C7 NG + iters*2NK per refit, C8 N*G_all; fp32) summed over all "
                                 "K / (consensus wall time per GPU); the stage is a chain of small dependent launches "
                                 "(latency-bound), not a streaming kernel; peak = " + hbm_src},
            "note": "wall clock, max over ranks; cNMF.consensus numerics (cnmf.py:879-975: l2, distances, density, KMeans, "
                    "medians, 3 refits, OLS) through cnmf_b200.consensus.consensus_numerics, Ks sharded over ranks",
        }
        tpm_ds.close()

    # ---------------- reference's DEFAULT solver (cd, cnmf.py:629-631) on the same table, resident ----------------
    cd_default = None
    if world == 1 and not args.no_cd:
        step_resident(CD_KW)
        torch.cuda.synchronize(dev)
        t0 = time.perf_counter()
        for _ in range(args.steps):
            _, it_cd, _ = step_resident(CD_KW)
        torch.cuda.synchronize(dev)
        cd_default = {"gpu_value": n_jobs * args.steps / (time.perf_counter() - t0), "unit": "restarts/s",
                      "n_iter_mean": float(np.mean(it_cd)), "n_iter_max": int(np.max(it_cd))}

    # ---------------- end-to-end arm: host buffers through the public call ----------------
    ds.close()
    phases = {"dataset_ms": 0.0, "factorize_allgather_ms": 0.0, "d2h_ms": 0.0}

    def step_e2e():
        t0 = time.perf_counter()
        d2 = eng.dataset(Xnp, precision=args.precision)                   # H2D of X + device-side preparation
        t1 = time.perf_counter()
        sharded, _, _ = factorize_sharded(d2, ks_all, seeds_all, NMF_KW, comm)   # device RNG, solve, all-gather
        t2 = time.perf_counter()
        sp = sharded.host() if rank == 0 else None                        # D2H of every restart's spectra
        d2.close()
        phases["dataset_ms"] += 1e3 * (t1 - t0)
        phases["factorize_allgather_ms"] += 1e3 * (t2 - t1)
        phases["d2h_ms"] += 1e3 * (time.perf_counter() - t2)
        return sp

    for _ in range(max(1, args.warmup // 2)):
        step_e2e()
    sync_all()
    for k_ in phases:
        phases[k_] = 0.0
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step_e2e()
    sync_all()
    e2e_value = n_jobs * args.steps / max_over_ranks(time.perf_counter() - t0)
    clk = clocks.stop() if rank == 0 else None      # sampled across the timed regions
    SK_all = int(sum(ks_all))
    h2d = X.shape[0] * X.shape[1] * 4 * world       # every rank uploads its replica of X; nothing else goes up
    d2h = SK_all * X.shape[1] * 4                   # rank 0 reads every restart's spectra back
    if comm is not None:
        comm.close()
    if rank != 0:
        return

    peak, peak_src = measured_peaks()
    if f16:           # kind::f16 runs at the bf16 rate: the denominator is the measured bf16 figure itself
        peak, peak_src = 2.0 * peak, peak_src.replace("/2 (dense TF32 = half the bf16 rate)", " (kind::f16 = the bf16 rate)")
    hbm_peak, hbm_src = measured_hbm()
    upd_gbs = upd_bytes / (upd_ms * 1e-3) / 1e9 if upd_ms > 0 else 0.0
    achieved = gemm_flops / (gemm_ms * 1e-3) / 1e12 if gemm_ms > 0 else 0.0
    traffic = None
    tp = os.path.join(ROOT, "profiles", "gemm_traffic.json")
    if os.path.exists(tp):
        tj = json.load(open(tp))
        traffic = tj.get("dram_bytes_per_launch_f16" if f16 else "dram_bytes_per_launch", tj.get("dram_bytes_per_launch"))
    out = {
        "metric": METRIC, "value": value, "unit": "restarts/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": args.scaling,
        "vs_baseline": None,
        "dtype": ("f32 (2-pass split-fp16 tensor-core products of group-normalised factors x exact integer counts, fp32 "
                  "accumulate)" if f16 else "f32 (%d-pass split-TF32 tensor-core products, fp32 accumulate)" % passes),
        "data": "synthetic",
        "config": workload_config(args.workload, world, args.scaling, n_jobs),
        "clocks": clk,
        "e2e": {"value": e2e_value, "unit": "restarts/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                "ms_per_step": {k_: v_ / args.steps for k_, v_ in phases.items()},
                "note": "public call with host buffers: Engine.dataset(X host) + parallel.factorize_sharded + D2H of all spectra"},
        "gpu_launches": int(launches),
        "roofline": {"bound": "tensor", "kernel": "gemm_tf32x3_kernel<256,%s>" % ("3,exact-B,kind::f16" if f16 else "3,exact-B" if passes == 2 else "2,general"),
                     "achieved": achieved, "peak": peak, "unit": "TFLOP/s", "frac": achieved / peak, "traffic": traffic,
                     "mma_passes": passes, "mma_frac": passes * achieved / peak,
                     "note": "achieved = algorithmic 2*M*N*K per launch (counted once, not %dx for the passes) / "
                             "CUDA-event launch time; %d launches, %.1f ms of %.1f ms timed (rank 0); peak = %s; X %s" % (
                                 passes, gemm_launches, gemm_ms, ms, peak_src,
                                 "recognised as scaled integer counts -> exact B operand, 2 passes" if passes == 2
                                 else "general real matrix -> 3 passes")},
        "roofline_update": {"bound": "hbm", "kernel": "update_kernel<16,mu> (multiplicative update fused with the Gram "
                            "of the factor it writes and the emission of its tensor-core operand pieces)", "achieved": upd_gbs, "peak": hbm_peak, "unit": "GB/s",
                            "frac": upd_gbs / hbm_peak, "traffic": None,
                            "note": "second kernel of the step: achieved = algorithmic bytes per launch (factor read + "
                                    "product slices read + factor and its 2 operand pieces written, x live rows x items) / "
                                    "CUDA-event launch time; %d launches, %.1f ms of %.1f ms timed; peak = %s" % (
                                        upd_launches, upd_ms, ms, hbm_src)},
        "n_iter": {"mean": float(np.mean(n_iter)), "max": int(np.max(n_iter)), "jobs_rank0": len(my_jobs)},
        "with_consensus": with_consensus,
    }
    if world == 1 and not args.no_cpu_baseline:
        from oracle import reference_path
        from threadpoolctl import threadpool_limits
        X64 = X.astype(np.float64)
        mid = n_jobs // 2                                        # a restart of the median K of the sweep
        job = (ks_all[mid], seeds_all[mid])
        threads, probe = best_thread_count(X64, job, "mu")
        with threadpool_limits(limits=threads):
            _, its, sec = reference_path.factorize(X64, [job], "mu")
        out["cpu_baseline"] = {"value": 1.0 / sec, "unit": "restarts/s", "cores": threads, "kind": "port",
                               "sample": "1 of the %d restarts (K=%d, seed %d) to convergence (n_iter=%d), sklearn "
                                         "non_negative_factorization MU float64 as called by cnmf.py:672; best of a thread "
                                         "sweep %s" % (n_jobs, job[0], job[1], its[0], {k: round(v, 2) for k, v in probe.items()})}
        if cd_default is not None:
            with threadpool_limits(limits=threads):
                _, its_cd, sec_cd = reference_path.factorize(X64, [job], "cd")
            cd_default.update(cpu_value=1.0 / sec_cd, cpu_cores=threads,
                              note="the reference's DEFAULT solver for beta_loss='frobenius' (coordinate descent, cnmf.py:629-631): "
                                   "same job table on the GPU (%d steps, resident) vs 1 restart (K=%d, n_iter=%d) of the reference's "
                                   "sklearn call on the host" % (args.steps, job[0], its_cd[0]))
    out["cd_default"] = cd_default
    if dump is not None:
        write_outputs(args.dump_outputs, dump)
    print(json.dumps(out), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", type=str, default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", type=str, default="c3", choices=sorted(WORKLOADS))
    ap.add_argument("--scaling", type=str, default="strong", choices=["strong", "weak"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-consensus", action="store_true")
    ap.add_argument("--no-cd", action="store_true")
    ap.add_argument("--precision", type=str, default="f16x2", choices=["f16x2", "tf32x3", "tf32x3-general", "fp32"],
                    help="f16x2 (default): 2 kind::f16 passes when X is scaled integer counts, else 3 kind::tf32 passes; tf32x3: 2 / 3 kind::tf32 passes")
    ap.add_argument("--dump-outputs", type=str, default=None, metavar="DIR",
                    help="after the timed steps, write what the last timed step returned as DIR/<name>.npy: spectra "
                         "(the stacked k x genes spectra of the jobs in spectra_jobs: every job of the table, or a fixed "
                         "seeded subset when they exceed 64 MB), n_iter (of every job the step solved, in job-table "
                         "order), spectra_jobs")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
    else:
        run_ours(args, rank, world, local)
        if world > 1:
            import torch.distributed as dist
            if dist.is_initialized():
                dist.destroy_process_group()


if __name__ == "__main__":
    main()
