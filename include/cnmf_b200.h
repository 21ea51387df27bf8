/* cnmf_b200 -- C ABI of the B200-native consensus-NMF hot path.
 *
 * Plain C, plain pointers and sizes, no torch / C++ types.  This is the boundary a reference
 * maintainer binds instead of scikit-learn at the seam
 *
 *     cNMF._nmf(X, nmf_kwargs) -> (spectra, usages)          /root/reference/src/cnmf/cnmf.py:661-674
 *
 * which the reference calls from cNMF.factorize (cnmf.py:735-745, one call per (k, seed)
 * restart) and cNMF.refit_usage (cnmf.py:776-802, update_H=False), plus the numeric steps of
 * cNMF.consensus (cnmf.py:882-975).  INTEGRATION.md shows the ctypes stub.
 *
 * Conventions
 *   - every function returns 0 on success, <0 on error; cnmf_last_error() gives the message
 *     (thread-local).  -1 = invalid argument, -2 = CUDA error, -3 = unsupported.
 *   - "host" pointers are ordinary (ideally pinned) host memory; "dev" pointers are device
 *     memory of the device the handle was created on (e.g. torch.Tensor.data_ptr()).
 *   - matrices are dense row-major fp32; `ld` = row stride in elements.
 *   - `stream` is a cudaStream_t passed as void* (NULL = default stream).  Calls are
 *     synchronous with respect to the host on return unless stated otherwise.
 *   - there is NO CPU fallback: without a CUDA device every compute entry point fails.
 */
#ifndef CNMF_B200_H
#define CNMF_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define CNMF_B200_ABI_VERSION 7
#define CNMF_MAX_COMPONENTS 32          /* largest n_components per restart on the CUDA path */

typedef struct cnmf_handle_s* cnmf_handle_t;
typedef struct cnmf_dataset_s* cnmf_dataset_t;

enum { CNMF_SOLVER_MU = 0, CNMF_SOLVER_CD = 1 };            /* yaml 'solver': cnmf.py:618-631 */
/* FFMA | tcgen05 3xTF32 with exact-count detection (default: 2 passes when X is scaled integers, else 3) |
 * tcgen05 3xTF32 always in the general 3-pass form.  Params for a dataset created with 2 use precision 1. */
enum { CNMF_PRECISION_FP32 = 0, CNMF_PRECISION_TF32X3 = 1, CNMF_PRECISION_TF32X3_GENERAL = 2,
       /* dataset_create only: like TF32X3, but when X is recognised as scaled integer counts the big products run as
        * 2 kind::f16 tensor-core passes (integer operand exact in fp16, factor = two fp16 pieces of its row-normalised
        * values: the same 22 significant bits as the tf32 pair at twice the MMA rate); params.precision stays TF32X3 */
       CNMF_PRECISION_F16X2 = 3 };

/* yaml 'beta_loss' (cnmf.py:622, CLI --beta-loss cnmf.py:1251).  'frobenius' (or 2) runs the tensor-core path with
 * either solver; 'kullback-leibler' (1) and 'itakura-saito' (0) run the multiplicative updates of sklearn
 * _nmf.py:551-608, 637-694 as fused streaming kernels (solver must be CNMF_SOLVER_MU, as in sklearn). */
enum { CNMF_LOSS_FROBENIUS = 0, CNMF_LOSS_KULLBACK_LEIBLER = 1, CNMF_LOSS_ITAKURA_SAITO = 2 };

/* Mirrors the nmf_kwargs dict of cnmf.py:618-627 after sklearn's own scaling of the
 * regularisation (sklearn/decomposition/_nmf.py:1249-1260): l1_reg_W = n_features*alpha_W*l1_ratio ... */
typedef struct cnmf_nmf_params {
  int32_t solver;        /* CNMF_SOLVER_* */
  int32_t precision;     /* CNMF_PRECISION_* */
  int32_t max_iter;      /* 'max_iter' (cnmf.py:625) */
  int32_t reserved;      /* flags: bit 0 = draw the random init on the host (bit-exact numpy stream) instead of the GPU */
  double tol;            /* 'tol' (cnmf.py:624) */
  double l1_reg_W, l2_reg_W, l1_reg_H, l2_reg_H;
  int32_t beta_loss;     /* CNMF_LOSS_* ('beta_loss', cnmf.py:622); 0 = frobenius */
  int32_t reserved2;     /* must be 0 */
} cnmf_nmf_params;

/* ---- library / handle -------------------------------------------------------------- */
int cnmf_abi_version(void);
const char* cnmf_last_error(void);
int cnmf_create(cnmf_handle_t* out, int device);
int cnmf_destroy(cnmf_handle_t h);
/* number of kernels this library has launched through the handle since creation */
long long cnmf_launch_count(cnmf_handle_t h);
/* free / total bytes of the handle's device (cudaMemGetInfo) plus the bytes parked in the handle's own buffer
 * pool and workspace (reusable by the next call): what the facade sizes its restart groups from, so that a
 * K-sweep larger than HBM is factorized in several batched solves instead of failing in cudaMalloc */
int cnmf_mem_info(cnmf_handle_t h, long long* free_bytes, long long* total_bytes, long long* cached_bytes);
/* device bytes one packed factor row (one component of one restart) costs in a batched solve on this dataset:
 * factors, operand pieces, compaction ping-pong and result slabs, product slices */
long long cnmf_solve_bytes_per_row(cnmf_dataset_t d);

/* per-launch CUDA-event timing of the dominant kernel (the batched GEMM) on its launching stream:
 * enable (resets the counters), run, then read total device ms, launches and algorithmic FLOPs
 * (2*M*N*K per launch, counted once -- not 3x for the 3xTF32 passes) */
int cnmf_profile_enable(cnmf_handle_t h, int on);
int cnmf_profile_get(cnmf_handle_t h, double* gemm_ms, long long* gemm_launches, double* gemm_flops);
/* same counters per kernel class: 0 = batched GEMM (work = algorithmic FLOPs), 1 = fused update kernels
 * (work = algorithmic bytes: factor read + product slices read + factor and tf32 pieces written) */
int cnmf_profile_get_class(cnmf_handle_t h, int kernel_class, double* ms, long long* launches, double* work);

/* host wall-clock phases (ms) of the last factorize call on this handle (cnmf_factorize, _seeds_dev, _init or _dev;
 * each resets all four when it starts): host RNG (device RNG: its enqueue time), H2D of the host RNG's factors,
 * batched solve, copy-out of the results.  A phase the call did not run reads 0.  With profiling enabled,
 * cnmf_refit and cnmf_kmeans_fit write their own phases into the same fields. */
int cnmf_last_timing(cnmf_handle_t h, double* rng_ms, double* h2d_ms, double* solve_ms, double* d2h_ms);

/* ---- dataset: a cells x genes matrix made resident on the device ------------------- */
/* Replaces `norm_counts.X` / `tpm.X` handed to _nmf (cnmf.py:726,741,873,919,950-952).
 * Builds the device-side forms both GEMM orientations need (X, X^T, tf32 pieces) and
 * sum(X), sum(X^2).  `src_is_device` = 0: X is host memory (copied H2D inside the call). */
int cnmf_dataset_create(cnmf_handle_t h, const float* X, int n_rows, int n_cols, long long ld,
                        int src_is_device, int precision, void* stream, cnmf_dataset_t* out);
/* new dataset = src[:, cols] * col_scale (cnmf.py:965-969: tpm[:, hvgs] / std) */
int cnmf_dataset_from_columns(cnmf_dataset_t src, const int32_t* cols_host, const float* col_scale_host,
                              int n_cols, void* stream, cnmf_dataset_t* out);
int cnmf_dataset_destroy(cnmf_dataset_t d);
int cnmf_dataset_shape(cnmf_dataset_t d, int* n_rows, int* n_cols);
/* padded row strides of the packed factor layout: W^T rows (ld_rows >= n_rows), H rows (ld_cols >= n_cols) */
int cnmf_dataset_ld(cnmf_dataset_t d, int* ld_rows, int* ld_cols);
int cnmf_dataset_sums(cnmf_dataset_t d, double* sum, double* sum_sq);
/* smallest entry of X (sklearn refuses beta_loss <= 0 when X.min() == 0, _nmf.py:1675-1680; the caller raises) */
int cnmf_dataset_min(cnmf_dataset_t d, float* min_host, void* stream);
/* 1 when the dataset was recognised as (row scale) x (integer counts <= 2048) x (column scale) -- what
 * HVG-normalised counts (cnmf.py:542) and TPM (cnmf.py:245-251) are -- and therefore runs the 2-pass
 * tensor-core products (the integer operand needs no tf32 "lo" piece); 0 = general 3-pass 3xTF32.
 * Returns 2 when, in addition, the dataset was created with CNMF_PRECISION_F16X2 and the 2 passes therefore run on
 * kind::f16 MMAs. */
int cnmf_dataset_is_exact(cnmf_dataset_t d);
/* per-column mean and population variance (StandardScaler(with_mean=False), cnmf.py:131-134) */
int cnmf_dataset_col_stats(cnmf_dataset_t d, double* mean_host, double* var_host, void* stream);

/* ---- device-side `prepare` numerics (cnmf.py:131-251, 487-556) on a resident counts matrix ------------- */
/* per-row (cell) totals, fp64: the TPM denominators of compute_tpm / sc.pp.normalize_total (cnmf.py:245-251) */
int cnmf_dataset_row_sums(cnmf_dataset_t d, double* row_sums_host, void* stream);
/* per-column mean and population variance of diag(row_scale) * X accumulated in fp64 from the stored values:
 * with X = raw counts and row_scale = 1e6 / cell total these are the TPM gene statistics that drive the
 * over-dispersion ranking (get_highvar_genes, cnmf.py:192-242) and `tpm_stats` (cnmf.py:436-445), without
 * materialising TPM */
int cnmf_dataset_scaled_col_stats(cnmf_dataset_t d, const double* row_scale_host, double* mean_host, double* var_host,
                                  void* stream);
/* new dataset = diag(row_scale) * src (TPM from counts, cnmf.py:245-251); the exact-count detection runs again */
int cnmf_dataset_scale_rows(cnmf_dataset_t src, const float* row_scale_host, void* stream, cnmf_dataset_t* out);

/* ---- random init (sklearn _nmf.py:296-307; host RNG, bit-exact numpy legacy stream) -- */
/* Writes |avg*z| as fp32: H (k x n_features, row stride ldH) first, then W stored transposed
 * Wt (k x n_samples, row stride ldW).  Pure host code (no CUDA). */
int cnmf_random_init_host(uint32_t seed, double avg, int n_samples, int n_features, int k,
                          float* Wt, long long ldW, float* H, long long ldH);

/* Same stream generated ON THE DEVICE (one thread block per restart; see csrc/rng_device.cu for the one
 * caveat: log() may differ from glibc in the last fp64 bit, visible in ~1 fp32 value per 10^8) into packed,
 * padded device buffers: Wt_dev (sum ks) x ld_rows, H_dev (sum ks) x ld_cols (cnmf_dataset_ld), avg =
 * sqrt(mean(X) / k) as sklearn.  This is what cnmf_factorize uses unless params.reserved bit 0 is set. */
int cnmf_random_init_dev(cnmf_dataset_t d, int n_restarts, const int32_t* ks, const uint32_t* seeds, float* Wt_dev,
                         float* H_dev, void* stream);

/* ---- batched factorize: replaces the restart loop of cNMF.factorize ---------------- */
/* For r in [0, n_restarts): one NMF of the dataset with n_components = ks[r] and
 * random_state = seeds[r] (cnmf.py:738-741), all restarts advanced together on the GPU.
 *   spectra_host : packed (sum ks) x n_cols, row stride n_cols; restart r owns rows
 *                  [sum ks[0..r), +ks[r])  -- what factorize saves per restart (cnmf.py:742-745)
 *   usages_host  : optional (may be NULL; the reference discards W) packed (sum ks) x n_rows,
 *                  i.e. W^T per restart
 *   n_iter_host  : optional [n_restarts] iterations run;  err_host: optional [n_restarts]
 *                  ||X - WH||_F of the returned factors (every solver and loss) */
int cnmf_factorize(cnmf_dataset_t d, int n_restarts, const int32_t* ks, const uint32_t* seeds,
                   const cnmf_nmf_params* params, float* spectra_host, float* usages_host,
                   int32_t* n_iter_host, double* err_host, void* stream);

/* Same restarts, same seeds, but the spectra stay on the device: spectra_dev is (sum ks) x ld_out (ld_out >= n_cols).
 * This is the per-rank half of the multi-GPU path: the slab goes straight into cnmf_allgather_spectra / an NCCL
 * all-gather without touching the host (cnmf.py:748-773 `combine` meets on disk instead). */
int cnmf_factorize_seeds_dev(cnmf_dataset_t d, int n_restarts, const int32_t* ks, const uint32_t* seeds,
                             const cnmf_nmf_params* params, float* spectra_dev, long long ld_out,
                             int32_t* n_iter_host, double* err_host, void* stream);

/* ---- the one collective of the path: all-gather of the per-rank spectra slabs (SURVEY.md 8b/8e) ---------------- */
/* merged_dev (world x rows_per_rank x ld) <- every rank's local_dev (rows_per_rank x ld; ranks with fewer rows pad),
 * asynchronous on `stream`.  `nccl_comm` is an ncclComm_t -- the host application's own, or one made by
 * cnmf_comm_create.  libnccl.so.2 is bound at run time (no link-time dependency; CNMF_NCCL_LIB overrides the path). */
int cnmf_allgather_spectra(void* nccl_comm, const float* local_dev, long long rows_per_rank, long long ld,
                           float* merged_dev, void* stream);
/* communicator bootstrap for hosts without one: rank 0 calls cnmf_comm_unique_id and ships the 128 bytes to every
 * rank over whatever channel it has (MPI, a TCP store, torch.distributed ...); every rank then calls
 * cnmf_comm_create with its rank (collective: blocks until all ranks arrive) */
int cnmf_comm_unique_id(char* id_out_128);
int cnmf_comm_create(cnmf_handle_t h, const char* id_128, int rank, int world, void** comm_out);
int cnmf_comm_destroy(void* nccl_comm);

/* Same, but initial factors are supplied (host, packed like the outputs) instead of seeds. */
int cnmf_factorize_init(cnmf_dataset_t d, int n_restarts, const int32_t* ks, const float* Wt0_host,
                        const float* H0_host, const cnmf_nmf_params* params, float* spectra_host,
                        float* usages_host, int32_t* n_iter_host, double* err_host, void* stream);

/* Device-resident form: initial factors and the output stay on the GPU (packed, padded strides from
 * cnmf_dataset_ld): Wt0_dev (sum ks) x ld_rows, H0_dev / spectra_dev (sum ks) x ld_cols. */
int cnmf_factorize_dev(cnmf_dataset_t d, int n_restarts, const int32_t* ks, const float* Wt0_dev,
                       const float* H0_dev, const cnmf_nmf_params* params, float* spectra_dev,
                       int32_t* n_iter_host, double* err_host, void* stream);

/* ---- NNLS refit: replaces cNMF.refit_usage / refit_spectra (cnmf.py:776-820) ------- */
/* NMF with one factor fixed (sklearn update_H=False), same solver as factorize (cnmf.py:792).
 * transposed = 0 (refit_usage,  cnmf.py:798):  fixed_host = H   (k x n_cols), out_host = W (n_rows x k)
 * transposed = 1 (refit_spectra, cnmf.py:820): fixed_host = W^T (k x n_rows), out_host = H^T (n_cols x k)
 * W0 follows sklearn _nmf.py:1223-1228 ('mu': sqrt(X.mean()/k) constant, 'cd': zeros).
 * err_host (optional): final ||X - W H||_F (its square is the prediction error of cnmf.py:926-930). */
int cnmf_refit(cnmf_dataset_t d, int transposed, int k, const float* fixed_host, const cnmf_nmf_params* params,
               float* out_host, int32_t* n_iter_host, double* err_host, void* stream);

/* out (k x n_cols) = Ut (k x n_rows) * X : the X^T Y accumulator of efficient_ols_all_cols
 * (cnmf.py:98-119) as one tensor-core GEMM; the caller centres U (see cnmf_b200/consensus.py). */
int cnmf_project_rows(cnmf_dataset_t d, int k, const float* Ut_host, float* out_host, void* stream);

/* test / micro-benchmark hook: C (M x N) = A (M x Kd) * B (N x Kd)^T through the same GEMM kernels the
 * solver uses (precision selects FFMA or tcgen05 3xTF32); reps > 1 reports mean device ms per launch. */
int cnmf_gemm_abt_host(cnmf_handle_t h, int precision, const float* A, const float* B, int M, int N, int Kd,
                       int splits, float* C, int reps, float* ms_out, void* stream);

/* ---- consensus kernels (cnmf.py:882-916) on a stacked-spectra matrix S (R x G, device, row stride ld) -- */
/* rows / ||row||_2 in place (cnmf.py:882) */
int cnmf_l2_normalize_rows(cnmf_handle_t h, float* S_dev, int R, int G, int ld, void* stream);
/* local density (cnmf.py:891-896): density[i] = (sum of the n_neighbors+1 smallest entries of row i of the
 * Euclidean distance matrix, self-distance 0 included) / n_neighbors.  D_dev: optional R x R output
 * (ld = R) for the clustergram; NULL keeps it in the library's workspace. Asynchronous on `stream`. */
int cnmf_local_density(cnmf_handle_t h, const float* S_dev, int R, int G, int ld, int n_neighbors,
                       float* density_dev, float* D_dev, void* stream);
/* per-column mean and population variance of a device matrix (KMeans tolerance, sklearn _kmeans.py:285-293) */
int cnmf_col_stats_dev(cnmf_handle_t h, const float* S_dev, int R, int G, int ld, double* mean_host,
                       double* var_host, void* stream);
/* dst row i = src row idx[i] (density filter compaction, cnmf.py:903-904) */
int cnmf_gather_rows(cnmf_handle_t h, const float* src_dev, int ld_src, const int32_t* idx_host, int n, int G,
                     float* dst_dev, int ld_dst, void* stream);
/* squared Euclidean distances from rows idx[0..n_c) of S to every row of S -> out_host (n_c x R):
 * candidate scoring of k-means++ (sklearn _kmeans.py:231-262; the random draws stay on the host) */
int cnmf_sq_dists_to_rows(cnmf_handle_t h, const float* S_dev, int R, int G, int ld, const int32_t* idx_host,
                          int n_c, float* out_host, void* stream);
/* one Lloyd E+M step (sklearn _k_means_lloyd.pyx:168-219): labels_dev updated in place (first minimum wins),
 * mind_dev[i] = squared distance to the assigned centre; optional host outputs: per-cluster fp64 column
 * sums (K x G) + counts, number of labels that changed, inertia = sum(mind). */
int cnmf_kmeans_assign(cnmf_handle_t h, const float* S_dev, int R, int G, int ld, const float* centers_host, int K,
                       int32_t* labels_dev, double* sums_host, int32_t* counts_host, float* mind_dev,
                       int32_t* n_changed_host, double* inertia_host, void* stream);
/* one full Lloyd iteration with the centres resident on the device (the loop of sklearn _kmeans.py:630-758 without a
 * K x G round trip per iteration): E step against C32_cur (labels_dev / mind_dev updated), fp64 per-cluster sums and
 * counts (sums_dev K x G, counts_dev K), new centres = sums / count into C64_new (fp64) and C32_new (their fp32 copy
 * for the next E step).  Host outputs: labels that changed, whether a cluster came out empty (then C*_new are not
 * valid for it: the caller applies the relocation rule of _k_means_common.pyx:167-211 from sums_dev / counts_dev and
 * the current centres, which this call leaves untouched), and sum((C64_new - C64_cur)^2) over the non-empty clusters. */
int cnmf_kmeans_step(cnmf_handle_t h, const float* S_dev, int R, int G, int ld, int K, const float* C32_cur_dev,
                     const double* C64_cur_dev, double* C64_new_dev, float* C32_new_dev, int32_t* labels_dev,
                     float* mind_dev, double* sums_dev, int32_t* counts_dev, int32_t* n_changed_host,
                     int32_t* any_empty_host, double* shift_host, void* stream);
/* The whole KMeans(n_clusters=K, n_init, random_state) fit of the consensus step (cnmf.py:908-910) with every
 * initialisation resident and advancing together on the device: k-means++ for all runs (2 launches per centre, no
 * host round trip), Lloyd for all runs (one small flag read per iteration), final E step + inertia.  The random
 * draws are data-independent in count and order, so the caller draws them from numpy's legacy RandomState exactly
 * as sklearn would and passes them in: first_idx_host[n_init] (rng.choice per run) and uniforms_host
 * [n_init][K-1][n_trials] (rng.uniform(size=n_trials) per further centre, n_trials = 2 + int(log(K))), in sklearn's
 * order of consumption (run by run).  tol_abs = mean feature variance * tol (sklearn _kmeans.py:285-293).
 * Outputs per run: labels (n_init x R), inertia, iterations; the caller applies sklearn's best-run rule
 * (_kmeans.py:1534-1541).  *needs_host_path = 1 when a cluster came out empty (sklearn's relocation rule,
 * _k_means_common.pyx:167-211): outputs are then undefined and the caller falls back to cnmf_kmeans_step. */
int cnmf_kmeans_fit(cnmf_handle_t h, const float* S_dev, int R, int G, int ld, int K, int n_init, int max_iter,
                    double tol_abs, const int32_t* first_idx_host, const double* uniforms_host, int n_trials,
                    int32_t* labels_host, double* inertia_host, int32_t* n_iter_host, int32_t* needs_host_path,
                    void* stream);
/* sums_host[i*K + c] = sum over rows j with label c of ||S_i - S_j||_2 : the per-sample cluster distance sums
 * from which sklearn.metrics.silhouette_score(metric='euclidean') is formed (cnmf.py:923, k_selection) */
int cnmf_cluster_dist_sums(cnmf_handle_t h, const float* S_dev, int R, int G, int ld, const int32_t* labels_dev,
                           int K, double* sums_host, void* stream);
/* per-cluster per-gene median (pandas groupby().median(), cnmf.py:913), rows then divided by their sum
 * (cnmf.py:916) -> M_dev (K x ldm). Asynchronous on `stream`. */
int cnmf_cluster_median(cnmf_handle_t h, const float* S_dev, int R, int G, int ld, const int32_t* labels_dev, int K,
                        float* M_dev, int ldm, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* CNMF_B200_H */
