#!/usr/bin/env python
"""Generate tests/golden/*.npz by running the UNMODIFIED reference
(/root/reference/src/cnmf/cnmf.py, loaded through oracle/refshim.py) in the build container.

    python -m oracle.make_golden            # from the repo root; needs /root/reference

Test infrastructure (see oracle/__init__.py).  The reference's own golden tarballs are
network downloads (download_pytest_data.py:38-52) and are not available offline, so these
fixtures -- outputs of the reference itself on deterministic synthetic inputs -- are what
pins the oracle and, through it, the CUDA path.

Fixture ``<tag>.npz`` (one per solver / loss, tags ``sim_mu`` / ``sim_cd`` / ``sim_kl``; ``sim_nndsvd`` = init='nndsvd'
with the default solver; ``c1_mu`` / ``c1_cd`` are
BASELINE.json configs[0] -- 1 000 cells x 500 HVG, K=7, 10 restarts -- in full) holds
  counts          int16 cells x genes_all  (input given to reference prepare())
  hvg_idx         positions of the HVGs chosen by the reference inside genes_all
  ks, n_iter, seed, solver   (+ beta_loss in fixtures generated for a non-Frobenius loss)
  table           (n_components, iter, nmf_seed) rows written by reference prepare()
  merged_k<K>     reference combine() output (R x G, f64) after reference factorize()
  density_k<K>    reference local_density_cache
  cspectra_k<K>, cusages_k<K>, score_k<K>, tpmspec_k<K>   reference consensus() outputs
  stats_k<K>      [k, dt, silhouette, prediction_error] from consensus(skip_density...=True)
  fp32dev_k<K>    per restart: rel-L2 between scikit-learn's OWN float32 path and the reference (float64)
                  spectra for the same seed -- a conditioning yardstick for fp32-class implementations
                  (computed with a direct sklearn call; the reference itself always runs float64)
``path_table.json`` (``python -m oracle.make_golden path_table``) holds the reference's cNMF path table for
output_dir D and name "run", every path relative to D.
Everything derives from RandomState seeds, so the script is reproducible bit for bit on the
same library versions (numpy 2.3.5, scikit-learn 1.9.0, pandas 3.0.2).
"""
import os
import shutil
import sys
import tempfile
import warnings

import numpy as np
import pandas as pd

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from oracle import refshim  # noqa: E402
from cnmf_b200.synth import make_counts  # noqa: E402

GOLDEN_DIR = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden")

CASES = {
    # tag: (n_cells, n_genes_all, k_true, nhvg, ks, n_iter, seed, beta_loss, consensus dt)
    "sim_mu": (400, 260, 5, 200, [4, 5], 8, 14, 2.0, 0.5),      # float beta_loss -> solver 'mu' (SURVEY fact 3)
    "sim_cd": (400, 260, 5, 200, [4, 5], 8, 14, "frobenius", 0.5),  # reference default -> 'cd'
    "sim_kl": (400, 260, 5, 200, [4, 5], 6, 14, "kullback-leibler", 0.5),  # --beta-loss kullback-leibler -> 'mu', beta=1
    # BASELINE.json configs[0] in full: 1 000 cells x 500 HVG, K=7, n_iter=10 (both solvers)
    "c1_mu": (1000, 640, 7, 500, [7], 10, 14, 2.0, 0.5),
    "c1_cd": (1000, 640, 7, 500, [7], 10, 14, "frobenius", 0.5),
    # `--init nndsvd` (cnmf.py:1252) with the reference's default solver: every restart starts from a randomized SVD
    "sim_nndsvd": (400, 260, 5, 200, [4, 5], 4, 14, "frobenius", 0.5),
}
INIT_OF = {"sim_nndsvd": "nndsvd"}          # prepare(init=...) of a case; default 'random' (cnmf.py:335)


def run_case(tag, spec):
    n_cells, n_genes, k_true, nhvg, ks, n_iter, seed, beta_loss, dt = spec
    ref = refshim.load_reference()
    counts = make_counts(n_cells, n_genes, k_true=k_true, seed=0, libsize=800.0)
    genes = np.array(["g%d" % i for i in range(counts.shape[1])], dtype=object)
    cells = np.array(["c%d" % i for i in range(counts.shape[0])], dtype=object)
    tmp = tempfile.mkdtemp(prefix="golden_")
    out = {}
    try:
        df = pd.DataFrame(counts.astype(np.float64), index=cells, columns=genes)
        counts_fn = os.path.join(tmp, "counts.df.npz")
        ref.save_df_to_npz(df, counts_fn)
        obj = ref.cNMF(output_dir=tmp, name="g")
        obj.prepare(counts_fn, components=ks, n_iter=n_iter, densify=True, seed=seed,
                    beta_loss=beta_loss, num_highvar_genes=nhvg, init=INIT_OF.get(tag, "random"))
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            obj.factorize(0, 1)
        obj.combine()
        table = ref.load_df_from_npz(obj.paths["nmf_replicate_parameters"])
        hvgs = open(obj.paths["nmf_genes_list"]).read().split("\n")
        hvg_idx = np.array([int(g[1:]) for g in hvgs], dtype=np.int32)
        import yaml
        run_params = yaml.load(open(obj.paths["nmf_run_parameters"]), Loader=yaml.FullLoader)
        out.update(counts=counts.astype(np.int16), hvg_idx=hvg_idx, ks=np.array(ks), n_iter=n_iter,
                   seed=seed, solver=run_params["solver"], beta_loss=str(run_params["beta_loss"]),
                   init=str(run_params["init"]),
                   table=table[["n_components", "iter", "nmf_seed"]].values.astype(np.int64))
        for k in ks:
            merged = ref.load_df_from_npz(obj.paths["merged_spectra"] % k)
            out["merged_k%d" % k] = merged.values
            from sklearn.decomposition import non_negative_factorization
            norm = refshim._read(obj.paths["normalized_counts"])
            dev = []
            for _, p in table[table.n_components == k].sort_values("iter").iterrows():
                kw = dict(run_params)
                kw.update(n_components=int(k), random_state=int(p["nmf_seed"]))
                with warnings.catch_warnings():
                    warnings.simplefilter("ignore")
                    _, H32, _ = non_negative_factorization(np.asarray(norm.X, dtype=np.float32), **kw)
                ref_H = merged.values[int(p["iter"]) * k:(int(p["iter"]) + 1) * k]
                dev.append(np.linalg.norm(H32 - ref_H) / np.linalg.norm(ref_H))
            out["fp32dev_k%d" % k] = np.array(dev)
            with warnings.catch_warnings():
                warnings.simplefilter("ignore")
                stats = obj.consensus(k, skip_density_and_return_after_stats=True, show_clustering=False)
                out["stats_k%d" % k] = stats.values.astype(np.float64).reshape(-1)
                obj.consensus(k, density_threshold=dt, show_clustering=False, build_ref=True)
            dts = str(dt).replace(".", "_")
            out["density_k%d" % k] = ref.load_df_from_npz(obj.paths["local_density_cache"] % k).values.reshape(-1)
            out["cspectra_k%d" % k] = ref.load_df_from_npz(obj.paths["consensus_spectra"] % (k, dts)).values
            out["cusages_k%d" % k] = ref.load_df_from_npz(obj.paths["consensus_usages"] % (k, dts)).values
            out["score_k%d" % k] = ref.load_df_from_npz(obj.paths["gene_spectra_score"] % (k, dts)).values
            out["tpmspec_k%d" % k] = ref.load_df_from_npz(obj.paths["gene_spectra_tpm"] % (k, dts)).values
            out["starcat_k%d" % k] = ref.load_df_from_npz(obj.paths["starcat_spectra"] % (k, dts)).values
        out["dt"] = dt
    finally:
        shutil.rmtree(tmp, ignore_errors=True)
    os.makedirs(GOLDEN_DIR, exist_ok=True)
    np.savez_compressed(os.path.join(GOLDEN_DIR, tag + ".npz"), **out)
    print(tag, "->", {k: getattr(v, "shape", v) for k, v in out.items()})


def write_path_table():
    """``path_table.json``: the reference's cNMF(output_dir, name="run").paths, relative to output_dir."""
    import json
    ref = refshim.load_reference()
    tmp = tempfile.mkdtemp(prefix="golden_")
    try:
        paths = ref.cNMF(output_dir=tmp, name="run").paths
        table = {key: os.path.relpath(p, tmp) for key, p in paths.items()}
    finally:
        shutil.rmtree(tmp, ignore_errors=True)
    with open(os.path.join(GOLDEN_DIR, "path_table.json"), "w") as f:
        json.dump(table, f, indent=1, sort_keys=True)
        f.write("\n")
    print("path_table ->", len(table), "entries")


if __name__ == "__main__":
    for tag, spec in CASES.items():
        if len(sys.argv) == 1 or tag in sys.argv[1:]:      # `python -m oracle.make_golden sim_kl` regenerates one
            run_case(tag, spec)
    if len(sys.argv) == 1 or "path_table" in sys.argv[1:]:
        write_path_table()
