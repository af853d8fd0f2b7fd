/* lz.h — C ABI of the B200-native Lanczos e^A·x library (liblzb200.so).
 *
 * This is the drop-in boundary. The reference (hdelan/MSc-HPC-Final-Project) has no FFI layer: its boundary is the
 * C++ object API of parallel-final/lib (adjMatrix -> lanczosDecomp<T> -> eigenDecomp<T> -> multOut). The host-side
 * mirror of that API lives in msc-hpc-final-project_b200/lib/ and is implemented *entirely* on the entry points below;
 * each entry point cites the reference interface it replaces. Plain pointers and sizes only; every call returns an
 * int status (LZ_OK == 0, negative on error; text via lz_last_error()). There is no CPU fallback anywhere: a call
 * that needs the GPU fails with LZ_ERR_CUDA when no device is present.
 *
 * Threading: one lz_ctx <-> one host thread <-> one GPU. Multi-GPU = one ctx per rank (process or thread), tied
 * together by an NCCL communicator created from lz_nccl_unique_id() (rank 0) + lz_create_dist() (all ranks).
 * All device work is enqueued on the ctx's own stream; nothing inside lz_lanczos_run / lz_tridiag_expv / lz_multout
 * synchronises with the host, except that the first lz_lanczos_run with a larger k than any before grows the basis (one
 * allocation + stream sync before the loop; never inside it).
 *
 * Vertex order: callers always see the ORIGINAL vertex numbering (the one of the CSR / generator). Internally the
 * library relabels vertices (degree-descending, dealt cyclically over ranks); that permutation never leaks.
 *
 * Environment knobs (read at lz_create / graph load; all optional, for tuning and tests): LZ_SPMV_VARIANT, LZ_SPMV_CTAS,
 * LZ_SPMV_WINDOW_MB, LZ_SPMV_COLBLOCKS, LZ_ORDER (d|n), LZ_LAGGED_NORM, LZ_BASIS (f32), LZ_PUSH_CTAS, LZ_PEER_PUSH,
 * LZ_PEER_SCALARS, LZ_FUSED_PUSH, LZ_SPARSE_PUSH, LZ_COMM_OVERLAP, LZ_PEER_TIMEOUT_S, LZ_KEEP_CSR, LZ_SHARDED_INGEST, LZ_CUDA_GRAPH.
 */
#ifndef LZ_H_B200
#define LZ_H_B200

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define LZ_OK 0
#define LZ_ERR_ARG (-1)     /* bad argument / call order */
#define LZ_ERR_CUDA (-2)    /* CUDA runtime error (including "no device") */
#define LZ_ERR_NCCL (-3)    /* NCCL error */
#define LZ_ERR_ALLOC (-4)   /* host or device allocation failed */
#define LZ_ERR_IO (-5)      /* file problem */
#define LZ_ERR_NUMERIC (-6) /* breakdown (beta == 0), non-finite Ritz value, eigensolver did not converge */

#define LZ_NCCL_UID_BYTES 128

typedef struct lz_ctx lz_ctx;

/* ---- graph generators (deterministic, counter-based; identical output on host and device) ------------------ */
#define LZ_GRAPH_ER 1     /* G(n,m)-style: m candidate edges drawn uniformly, loops + duplicates dropped          */
#define LZ_GRAPH_RMAT 2   /* R-MAT, n = 2^scale, m = param_a * n candidate edges, (a,b,c,d)=(.45,.15,.15,.25) unless
                             overridden, bijective random vertex relabel, loops + duplicates dropped                  */
#define LZ_GRAPH_BAND 3   /* irregular banded: (i,i+1),(i,i+b) b=ceil(sqrt n) kept w.p. 0.98, + n/64 random chords */

typedef struct lz_graph_spec {
  uint32_t kind;      /* LZ_GRAPH_*                                                                */
  uint32_t scale;     /* RMAT: log2(n). otherwise ignored                                           */
  uint64_t n;         /* ER / BAND: number of vertices. RMAT: ignored (n = 1<<scale)                */
  uint64_t param_a;   /* ER: m candidate edges. RMAT: edge factor (candidates per vertex). BAND: 0 */
  uint64_t seed;
  double rmat_a, rmat_b, rmat_c; /* RMAT quadrant probabilities; all 0 -> (.45,.15,.15), d = 1-a-b-c */
} lz_graph_spec;

typedef struct lz_graph_info {
  uint64_t n;           /* vertices                                                   */
  uint64_t nnz;         /* stored directed entries (= 2 * undirected edges)           */
  uint64_t n_local;     /* rows owned by this rank                                    */
  uint64_t nnz_local;   /* entries owned by this rank                                 */
  uint32_t max_degree;  /* global                                                     */
  uint32_t pad_;
  uint64_t empty_rows;  /* global number of isolated vertices                         */
} lz_graph_info;

/* Host generator: returns malloc'ed CSR (original vertex order, columns ascending within a row); free with lz_free_host.
 * Replaces adjMatrix::random_adj / barabasi (parallel-final/lib/make_graph.cc:21-113), which are seeded from
 * std::random_device and therefore cannot be replayed. Needs no GPU. */
int lz_graph_generate_host(const lz_graph_spec* spec, uint64_t* n_out, uint64_t* nnz_out,
                           uint32_t** row_offset_out, uint32_t** col_idx_out);
void lz_free_host(void* p);

/* Edge list (0-based endpoints, any order, duplicates / both orientations / self loops allowed) -> symmetric simple CSR.
 * What adjMatrix::populate_sparse_matrix does after parsing (adjMatrix.cc:36-44), without the std::set. */
int lz_csr_from_edges(uint64_t n, uint64_t n_edges, const uint32_t* u, const uint32_t* v, uint64_t* nnz_out,
                      uint32_t** row_offset_out, uint32_t** col_idx_out);

/* Reference text format ("n n E" header, then E lines "col row", 1-based, upper-triangle entries once):
 * adjMatrix::populate_sparse_matrix (parallel-final/lib/adjMatrix.cc:21-46) and write_matrix_to_file (:53-69). That format is a
 * MatrixMarket coordinate file with its banner stripped (serial/README.md:9); the reader also accepts the unstripped file:
 * '%' comment lines are skipped and a value column is ignored (the matrix is pattern-only either way). */
int lz_csr_read_text(const char* path, uint64_t* n_out, uint64_t* nnz_out, uint32_t** row_offset_out, uint32_t** col_idx_out);
int lz_csr_write_text(const char* path, uint64_t n, const uint32_t* row_offset, const uint32_t* col_idx);
/* Binary CSR cache ("LZCSR1\0\0", u64 n, u64 nnz, u32 row_offset[n+1], u32 col_idx[nnz]); also what oracle/_ref/ref_final --csr reads. */
int lz_csr_read_bin(const char* path, uint64_t* n_out, uint64_t* nnz_out, uint32_t** row_offset_out, uint32_t** col_idx_out);
int lz_csr_write_bin(const char* path, uint64_t n, const uint32_t* row_offset, const uint32_t* col_idx);

/* ---- context -------------------------------------------------------------------------------------------------- */
const char* lz_last_error(void);
int lz_version(void);
int lz_device_count(int* count_out);

/* One GPU. Replaces the implicit device-0 context of lanczosDecomp<T>::cu_decompose (parallel-final/lib/cu_lanczos.cu:20-94). */
int lz_create(int device, lz_ctx** ctx_out);
/* Rank `rank` of `world` ranks, one GPU each, NCCL over NVLink. Generalises parallel-two-cards/lib/cu_lanczos.cu:39-69. */
int lz_nccl_unique_id(void* uid_out /* LZ_NCCL_UID_BYTES */);
int lz_create_dist(int device, int rank, int world, const void* uid, lz_ctx** ctx_out);
int lz_destroy(lz_ctx* ctx);
int lz_sync(lz_ctx* ctx);

/* ---- adjacency matrix -> device shard --------------------------------------------------------------------------- */
/* Host CSR -> device. Every rank passes the same full CSR and keeps its own rows. Replaces the three cudaMemcpyAsync
 * of cu_lanczos.cu:88-90 (and the racy change_IA_for_device1, parallel-two-cards/lib/cu_lanczos.cu:21-27). */
int lz_csr_upload(lz_ctx* ctx, uint64_t n, const uint32_t* row_offset, const uint32_t* col_idx);
/* Build the graph on the device (same bits as lz_graph_generate_host) and ingest it. */
int lz_graph_generate(lz_ctx* ctx, const lz_graph_spec* spec);
int lz_graph_info_get(lz_ctx* ctx, lz_graph_info* info_out);
/* Full CSR in original order back to the host (buffers sized n+1 and nnz from lz_graph_info_get). Test / oracle hook: a one-GPU
 * context keeps that copy, a multi-GPU context drops it after sharding (9 GB per GPU at 2^27) unless LZ_KEEP_CSR=1 is set. */
int lz_csr_download(lz_ctx* ctx, uint32_t* row_offset_out, uint32_t* col_idx_out);

/* ---- hot path ---------------------------------------------------------------------------------------------------- */
#define LZ_REORTH_NONE 0  /* plain three-term recurrence == reference (cu_lanczos.cu:97-128)                 */
#define LZ_REORTH_FULL 1  /* every step, against all stored basis vectors: classical Gram-Schmidt, repeated when the first
                             pass removed more than half of ||w||^2 ("twice is enough", decided on the device)        */

/* Storage precision of the Krylov basis V (call before lz_set_start_vector; changing it drops the start vector and any result).
 *   LZ_BASIS_F64 (default): V in fp64, the graded precision (1e-9 parity with the reference's double path).
 *   LZ_BASIS_F32: V in fp32 — half the bytes of every pass over the basis (multOut, full reorthogonalisation) and half its HBM
 *     footprint. All arithmetic stays fp64 and the three-term recurrence runs on fp64 copies of the last vectors, so alpha/beta of a
 *     plain run are those of the fp64 run; only the consumers of V see rounded vectors (error ~1e-8 relative, inside the 1e-6 the
 *     reference's own float build agrees with its double build to). This is what lanczosDecomp<float> (cu_lanczos.cu:144) maps to.
 *     With world > 1 every rank must select the same precision. */
#define LZ_BASIS_F64 0
#define LZ_BASIS_F32 1
int lz_set_basis_precision(lz_ctx* ctx, int precision);
/* x (n doubles, original order; NULL = all ones as in main.cu:79) -> device, computes ||x|| (cu_lanczos.h:18-24,63). ||x|| is taken
 * as 2^e ||2^-e x|| with e the exponent of max|x_i|, so it neither underflows nor overflows for any finite x: f(A)(2^p x) is
 * 2^p f(A) x to the bit while the values stay normal, and for every x whose squares are normal the bits are those of the plain sum
 * of squares. A host vector costs one read-back of max|x_i| (synchronises). LZ_ERR_ARG for a zero or non-finite x. */
int lz_set_start_vector(lz_ctx* ctx, const double* x_host);
/* Multi-GPU: only rank `root` reads x_host (one PCIe upload); the other ranks receive the vector over NVLink. Collective. */
int lz_set_start_vector_root(lz_ctx* ctx, const double* x_host, int root);
/* k Lanczos steps, basis V kept resident on the device (parallel-mult-on-card/lib/cu_lanczos.cu:39,57), alpha/beta in
 * device memory. Enqueue only. Replaces lanczosDecomp<T>::cu_decompose (parallel-final/lib/cu_lanczos.cu:97-128). */
int lz_lanczos_run(lz_ctx* ctx, uint32_t k, int reorth);
/* alpha[k], beta[k-1] to the host (cu_lanczos.cu:129-130). Synchronises. Either pointer may be NULL. */
int lz_get_tridiag(lz_ctx* ctx, double* alpha_out, double* beta_out);
/* On-device eigendecomposition of T = tridiag(beta, alpha, beta) and coefficient vector
 *   c = ||x|| * Z * (f(lambda) .* Z^T e1),   f = exp by default (see lz_set_matfun)
 * Replaces eigenDecomp<T> (LAPACKE_dstevd, parallel-final/lib/eigen.cu:17-21) + multiplyOut.cu:30-40. Enqueue only. */
int lz_tridiag_expv(lz_ctx* ctx);
/* Matrix function applied by the coefficient solve, so that lz_multout yields f(A) x. Ritz values theta_j, parameter p:
 *   LZ_MATFUN_EXP        exp(p*theta)            e^{pA} x: total communicability at inverse temperature p. (EXP, 1.0) is the
 *                                                default and gives the same bits as a context that never calls this.
 *   LZ_MATFUN_EXP_SCALED exp(p*theta - ls)       e^{p(A - sI)} x with s the Ritz value maximising p*theta and ls = p*s, so
 *                                                e^{pA} x = ans * e^ls. Never overflows (plain EXP fails with LZ_ERR_NUMERIC once
 *                                                p*theta_max passes ~709); ls is on the device, read it with lz_get_matfun_scale.
 *   LZ_MATFUN_RESOLVENT  1 / (1 - p*theta)       (I - pA)^{-1} x; with x = ones this is Katz centrality (up to subtracting x,
 *                                                which leaves the ranking unchanged). LZ_ERR_NUMERIC with its own message when
 *                                                1 - p*theta_j <= 0 for some Ritz value. That check sees theta_max <= lambda_max
 *                                                only: passing it does not prove p < 1/lambda_max. The Ritz values of any graph
 *                                                (theta_max among them) come from EXP_SCALED followed by lz_get_eigen.
 * Followed by lz_tridiag_expv, lz_get_eigen (coefficients), lz_estimate_change, lz_choose_k, lz_expv_host(_root); lz_multout,
 * lz_get_ans and lz_top_k consume the coefficients as before. Drops the coefficients and the answer but keeps the tridiagonal and
 * the basis, so one lz_lanczos_run serves any number of functions. Kept across start vectors and runs. LZ_ERR_ARG for an unknown
 * kind or a non-finite parameter. With world > 1 every rank must pass the same values (every rank then computes the same c). */
#define LZ_MATFUN_EXP 0
#define LZ_MATFUN_EXP_SCALED 1
#define LZ_MATFUN_RESOLVENT 2
int lz_set_matfun(lz_ctx* ctx, int kind, double param);
/* log of the factor the last lz_tridiag_expv left out: ls = p*s under LZ_MATFUN_EXP_SCALED, 0 otherwise. Synchronises.
 * LZ_ERR_ARG before lz_tridiag_expv. */
int lz_get_matfun_scale(lz_ctx* ctx, double* log_scale_out);
/* Optional read-back: eigenvalues ascending [k], eigenvectors row-major [k*k] with eigvecs[i*k+j] = component i of
 * vector j (the LAPACK_ROW_MAJOR layout eigen.cu:20 produces), coeff [k]. Synchronises. Any pointer may be NULL. */
int lz_get_eigen(lz_ctx* ctx, double* eigvals_out, double* eigvecs_out, double* coeff_out);
/* Convergence estimate: relative 2-norm change of e^A x (f(A) x, lz_set_matfun) between Krylov dimensions k_prev < k (k = the last run), from the
 * tridiagonal alone (no pass over the basis). The reference has no such check; its author recommends one (writeup sec. 11). */
int lz_estimate_change(lz_ctx* ctx, uint32_t k_prev, double* rel_out);
/* The smallest Krylov dimension k' <= k (k = the last run) such that every dimension in [k', k] reproduces the k-step answer to
 * within `tol` (relative 2-norm, by the estimate above). *k_out == k: not even k-1 steps do, convergence at k is not demonstrated;
 * *est_out (optional) is the estimate at *k_out, or at k-1 in that case. The reference fixes k by hand (main.cu:28, -k). */
int lz_choose_k(lz_ctx* ctx, double tol, uint32_t* k_out, double* est_out);
/* ans = V * c as a tall-skinny GEMV on the device. Replaces multOut's cblas_dgemv (multiplyOut.cu:43-47) and
 * cu_multOut's cublasDgemv (parallel-mult-on-card/lib/cu_multiplyOut.cu:66-72). Enqueue only. */
int lz_multout(lz_ctx* ctx);
/* ans (n doubles, original order) to the host (cublasGetVector, cu_multiplyOut.cu:77). Synchronises. With world > 1 the call
 * is collective; a rank that does not need the vector may pass NULL (it still takes part in the gather). */
int lz_get_ans(lz_ctx* ctx, double* ans_host);
/* Centrality ranking: the m (<= 1024) largest entries of the last lz_multout result, descending, ties towards the lower
 * vertex id (argsort(-y) with a stable index tie-break, SURVEY.md section 0) — ORIGINAL vertex ids and their values. Selected
 * on the device (radix select + one small sort), so the caller downloads m pairs instead of n doubles. The reference only
 * prints the vector (parallel-final/lib/write_ans.h:10-16); BASELINE.json names the top-100 ranking as an output of the path.
 * *count_out (optional) = min(m, n) valid pairs. Synchronises. With world > 1 the call is collective and every rank receives the
 * same result (idx_out / val_out may be NULL on ranks that do not need it). */
int lz_top_k(lz_ctx* ctx, uint32_t m, uint32_t* idx_out, double* val_out, uint32_t* count_out);
/* ---- top Ritz pairs: eigenvector centrality and a certified spectral-radius bracket ----------------------------------------------
 * After lz_lanczos_run(k) let T = Z Theta Z^T (Theta ascending). For j = 0..m-1: theta_j is the j-th largest Ritz value and
 * y_j = V z_j / ||V z_j|| its Ritz vector, unit 2-norm, sign chosen so that sum_i y_j(i) >= 0. Then, with a real SpMV,
 *   rho_j = y_j^T A y_j             the Rayleigh quotient (computed),
 *   r_j   = ||A y_j - rho_j y_j||_2 the true residual (not the Lanczos estimate beta_k |e_k^T z_j|, which needs the beta_k the run does not
 *                                   compute and is not valid once orthogonality is lost), computed and then enlarged by the fp64
 *                                   rounding allowance r_j (2n + 24) 2^-52 + (max_degree + 8) 2^-52 hi. It covers the SpMV's row
 *                                   sums, the dot product, the residual's sum of squares and ||y_j|| != 1 in fp64 (DESIGN.md).
 * A is symmetric, so [rho_j - r_j, rho_j + r_j] contains an eigenvalue of A (Krylov-Bogoliubov) for plain and reorthogonalised runs,
 * fp64 or fp32 basis, lagged or not; so does that interval with its ends rounded to fp64. A plain run can return two copies of a converged eigenvalue when m > 1 ("ghosts"); each interval
 * is still correct. Use LZ_REORTH_FULL and a random start vector when the pairs beyond the first matter.
 * Spectral-radius bracket lo <= lambda_max <= hi, for every graph (connected or not): lo = rho_0 (1 - (2n + max_degree + 24) 2^-52)
 * (lo = rho_0 when rho_0 <= 0), which covers the rounding of rho_0 as above; hi = max_i (A z)_i / z_i over the
 * vertices (Collatz-Wielandt, A >= 0, z > 0) with z_i = max(|y_0(i)|, LZ_CW_FLOOR * max|y_0|), inflated by the fp64 rounding
 * allowance (max_degree + 2) * 2^-52 (relative). Tight when y_0 has converged on a connected graph. hi certifies a Katz parameter:
 * alpha = f / hi with f < 1 gives alpha < 1 / lambda_max.
 *
 * lz_ritz: 1 <= m <= min(LZ_RITZ_MAX, k). Collective when world > 1; synchronises once at the end. Leaves y_0 as the answer, so
 * lz_get_ans / lz_top_k return eigenvector centrality (lz_multout brings f(A) x back). Does not touch the coefficients, the
 * tridiagonal or the basis. Works after a coefficient solve that overflowed (only the eigensolver's convergence is checked).
 * LZ_ERR_ARG: bad m or no run. LZ_ERR_NUMERIC: eigensolver failure, a zero Ritz vector or non-finite results.
 * A new run, start vector, graph or basis precision drops the pairs; lz_set_matfun keeps them. */
#define LZ_RITZ_MAX 16
#define LZ_CW_FLOOR 1e-6
int lz_ritz(lz_ctx* ctx, uint32_t m);
/* m values each, largest first. Any pointer may be NULL. LZ_ERR_ARG before lz_ritz. */
int lz_get_ritz(lz_ctx* ctx, double* theta_out, double* rayleigh_out, double* resid_out);
/* y_j (n doubles, original vertex order), j < m. Collective when world > 1; NULL on ranks that do not need the vector. */
int lz_get_ritz_vector(lz_ctx* ctx, uint32_t j, double* y_host);
/* lo <= lambda_max <= hi (see above); identical on every rank. LZ_ERR_ARG before lz_ritz. */
int lz_spectral_radius_bounds(lz_ctx* ctx, double* lo_out, double* hi_out);

/* Whole pipeline with HOST buffers, what lanczosDecomp<double>(A,k,x,true) + eigenDecomp + multOut do in main.cu:115-127:
 * H2D x, k steps, eigensolve, multOut, D2H ans. */
int lz_expv_host(lz_ctx* ctx, const double* x_host, uint32_t k, int reorth, double* ans_host);
/* Same with one caller: only rank `root` passes x_host and receives ans_host (ignored on the other ranks). Collective. */
int lz_expv_host_root(lz_ctx* ctx, const double* x_host, uint32_t k, int reorth, double* ans_host, int root);

/* ---- test hooks / measurement --------------------------------------------------------------------------------------- */
/* y = A x with host vectors in original order (all ranks get the full y). Parity hook against spMV, SPMV.cc:19-28. */
int lz_spmv_host(lz_ctx* ctx, const double* x_host, double* y_host);
/* Basis vector q_j (original order, full length) to the host. */
int lz_get_basis(lz_ctx* ctx, uint32_t j, double* q_host);
/* Selects the SpMV kernel variant. */
#define LZ_SPMV_AUTO 0     /* default: by row length — warp per row for long rows, sliced (32 rows per warp, one lane
                              per row, index stream transposed so it is read as whole lines) for the rest            */
#define LZ_SPMV_VECTOR 1   /* CSR, sub-warp (1..32 lanes) per row, lanes chosen per degree bin                        */
#define LZ_SPMV_WARP 2     /* CSR, one warp per row for every row                                                     */
int lz_set_spmv_variant(lz_ctx* ctx, int variant);

/* How the Krylov vector travels between the ranks of a multi-GPU context (valid once a start vector has been set):
 * in full through ncclAllGather, in full by peer stores over NVLink, or — when each rank's rows reference only a small part
 * of the other ranks' entries (band-like graphs: a halo plus chords) — only the referenced entries by peer stores.
 * need_frac = referenced remote entries / entries a full exchange would send, over all ranks. Generalises the whole-half-
 * vector cudaMemcpyPeer of parallel-two-cards/lib/cu_lanczos.cu:116-165. */
#define LZ_EXCHANGE_NONE 0         /* one GPU */
#define LZ_EXCHANGE_NCCL 1
#define LZ_EXCHANGE_PEER_DENSE 2
#define LZ_EXCHANGE_PEER_SPARSE 3
int lz_exchange_info(lz_ctx* ctx, int* mode_out, double* need_frac_out);

typedef struct lz_timings {
  float lanczos_ms;     /* device time of the last lz_lanczos_run (cudaEvent pair on the ctx stream) */
  float tridiag_ms;     /* last lz_tridiag_expv                                                      */
  float multout_ms;     /* last lz_multout                                                           */
  float spmv_ms_avg;    /* mean device time of one SpMV launch inside the last lz_lanczos_run (profiling on) */
  float update_ms_avg;  /* mean device time of the fused vector-update launches of one step (profiling on)   */
  float comm_ms_avg;    /* mean device time of the NCCL calls of one step (profiling on)                     */
  float reorth_ms_total;/* total device time spent in reorthogonalisation kernels (profiling on)             */
  uint32_t spmv_launches;
  uint32_t kernel_launches; /* kernels of this library launched on this ctx since lz_create (cumulative)           */
  uint32_t reorth_second_passes; /* steps of the last run whose Gram-Schmidt pass had to be repeated (LZ_REORTH_FULL)  */
} lz_timings;
/* profiling on => event pairs around the per-step launches (adds ~2 us per event). Off by default. */
int lz_set_profiling(lz_ctx* ctx, int on);
int lz_timings_get(lz_ctx* ctx, lz_timings* out);
/* cudaEvent stopwatch on the ctx stream, for callers that time several calls as one region (bench.py). */
int lz_timer_start(lz_ctx* ctx);
int lz_timer_stop(lz_ctx* ctx, float* ms_out); /* synchronises on the stop event */
/* Device-side timeline of the kernels' internal phases (start, wait for the peers over, push done, end): tells waiting for peers
 * apart from work inside the fused kernels, which stream events cannot. cap_events > 0: switch on and clear. cap_events == 0: read
 * back into out ((tag, globaltimer ns) pairs; tag = kernel << 8 | phase, see lz_kernels.cu) and switch off. Measurement only. */
int lz_debug_trace(lz_ctx* ctx, uint32_t cap_events, uint64_t* out, uint32_t out_cap_events, uint32_t* count_out);
/* Writes >= bytes of device memory (L2 flush between timed repetitions). */
int lz_flush_l2(lz_ctx* ctx);

#ifdef __cplusplus
}
#endif
#endif
