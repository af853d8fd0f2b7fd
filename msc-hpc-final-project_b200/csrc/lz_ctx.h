// lz_ctx.h — the per-GPU context behind the C ABI (include/lz.h) and the launch interfaces between translation units.
#pragma once
#include <cuda_runtime.h>
#include <nccl.h>
#include <stdint.h>
#include <vector>
#include "lz_internal.h"

#define LZ_CUDA(call)                                                                                   \
  do {                                                                                                  \
    cudaError_t e_ = (call);                                                                            \
    if (e_ != cudaSuccess)                                                                              \
      return lz_fail(LZ_ERR_CUDA, "%s:%d %s -> %s", __FILE__, __LINE__, #call, cudaGetErrorString(e_)); \
  } while (0)
// NCCL is bound at run time (dlopen) so that (a) single-GPU use needs no NCCL at all and (b) inside a process that
// already loaded a libnccl.so.2 (e.g. PyTorch's bundled one) we share that copy instead of clashing with it.
struct lz_nccl_api {
  ncclResult_t (*GetUniqueId)(ncclUniqueId*);
  ncclResult_t (*CommInitRank)(ncclComm_t*, int, ncclUniqueId, int);
  ncclResult_t (*CommDestroy)(ncclComm_t);
  ncclResult_t (*CommAbort)(ncclComm_t);
  ncclResult_t (*CommSplit)(ncclComm_t, int, int, ncclComm_t*, void*);   // may be null (NCCL < 2.18)
  ncclResult_t (*AllReduce)(const void*, void*, size_t, ncclDataType_t, ncclRedOp_t, ncclComm_t, cudaStream_t);
  ncclResult_t (*AllGather)(const void*, void*, size_t, ncclDataType_t, ncclComm_t, cudaStream_t);
  ncclResult_t (*Broadcast)(const void*, void*, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t);
  const char* (*GetErrorString)(ncclResult_t);
  ncclResult_t (*GetVersion)(int*);
};
const lz_nccl_api* lz_nccl();   // nullptr (with lz_last_error set) when no libnccl.so.2 can be loaded
#define LZ_NCCL(call)                                                                                   \
  do {                                                                                                  \
    ncclResult_t r_ = (call);                                                                           \
    if (r_ != ncclSuccess)                                                                              \
      return lz_fail(LZ_ERR_NCCL, "%s:%d %s -> %s", __FILE__, __LINE__, #call, lz_nccl()->GetErrorString(r_)); \
  } while (0)
#define LZ_TRY(call)            \
  do {                          \
    int rc_ = (call);           \
    if (rc_ != LZ_OK) return rc_; \
  } while (0)

// SpMV launch plan: local rows are sorted by length (non-increasing), so each bin is a contiguous row range that one
// kernel variant (lanes-per-row = 1 << log2_lanes) serves.
#define LZ_MAX_BINS 8
#define LZ_MAX_COLBLK 32
#define LZ_MAX_WORLD 16
#define LZ_SELL_LONG 128          // rows longer than this are served warp-per-row
#define LZ_SPMV_BLOCK 256         // threads per CTA of the SpMV kernel
#define LZ_SPMV_ROWS_PER_GROUP 4  // rows handled concurrently by one lane group (memory-level parallelism)
struct lz_spmv_bin {
  uint32_t row_begin, row_end;   // local rows [begin, end)
  uint16_t log2_lanes;           // lanes cooperating on one row
  uint16_t per_lane;             // entries each lane fetches per chunk (2 or 8); longer segments take further chunks
  uint32_t item_begin;           // first work item of this bin; one item = (BLOCK >> log2_lanes) * ROWS_PER_GROUP rows
};
struct lz_spmv_plan {
  lz_spmv_bin bin[LZ_MAX_BINS];
  uint32_t nbins;
  uint32_t nitems;
};

struct lz_ctx {
  int device = 0, rank = 0, world = 1;
  int sm_count = 148;
  ncclComm_t comm = nullptr;       // scalar / coefficient all-reduces, on `stream`
  ncclComm_t comm_ag = nullptr;    // chunked all-gather of the Krylov vector, on `comm_stream` (overlaps the SpMV passes)
  cudaStream_t stream = nullptr, comm_stream = nullptr;
  cudaEvent_t ev_scaled = nullptr, ev_chunk[LZ_MAX_COLBLK] = {};
  bool comm_overlap = true;
  bool chunks_in_flight = false;
  // Peer exchange (default for world > 1): k_scale stores q_{j+1} straight into every rank's gathered vector over NVLink
  // and raises per-chunk arrival counters there; SpMV pass b spins on chunk b's counters. No collective, no extra pass.
  bool peer_push = false;
  double* peer_xfull[LZ_MAX_WORLD] = {};              // every rank's xfull as seen from this GPU (own included)
  unsigned long long* peer_flags[LZ_MAX_WORLD] = {};  // every rank's arrival counters
  bool peer_ipc[LZ_MAX_WORLD] = {};                   // mapping came from cudaIpcOpenMemHandle (must be closed)
  unsigned long long* flags = nullptr;                // device, [LZ_MAX_COLBLK][LZ_MAX_WORLD], written by the peers
  unsigned int* push_ticket = nullptr;                // device, [LZ_MAX_COLBLK]
  unsigned long long push_seq = 0;                    // sequence number of the last push (same on every rank)
  unsigned long long red_seq = 0;                     // sequence number of the last peer scalar reduction
  double* gfull = nullptr;                            // device, [n_loc * world], scratch for the host-facing gathers
  // Needed-columns exchange: per peer, the ascending list of this rank's rows that the peer's rows reference. Used instead of
  // the dense push when the lists are short (lz_build_push_lists, lz_graph.cu).
  bool sparse_push = false;
  uint32_t* push_list = nullptr;                      // device, lists of all peers back to back
  uint32_t push_off[LZ_MAX_WORLD + 1] = {};           // list of peer r = push_list[push_off[r] .. push_off[r + 1])
  uint64_t graph_id = 0, push_graph_id = 0;           // graph the lists were built for (rebuilt when a new graph has the same shape)
  double push_need_frac = 1.0;                        // referenced remote entries / dense exchange volume (global)
  cudaEvent_t ev_a = nullptr, ev_b = nullptr;      // lz_lanczos_run
  cudaEvent_t ev_e0 = nullptr, ev_e1 = nullptr;    // lz_tridiag_expv
  cudaEvent_t ev_m0 = nullptr, ev_m1 = nullptr;    // lz_multout
  cudaEvent_t ev_t0 = nullptr, ev_t1 = nullptr;    // lz_timer_start / lz_timer_stop

  // ---- graph ------------------------------------------------------------------------------------------------------
  uint64_t n = 0, nnz = 0;         // global
  uint64_t n_loc = 0;              // rows per rank (>= ceil(n / world), multiple of chunk_rows); padded length = n_loc * world
  uint64_t nnz_loc = 0;
  uint64_t chunk_rows = 0;         // cl: rows of each rank per column block; n_loc = ncolblk * cl
  uint64_t ldv = 0;                // leading dimension of V (n_loc rounded up to 32 doubles => 256-byte aligned rows)
  uint32_t max_degree = 0;
  bool natural_order = false;      // vertex order kept (band-like, unskewed graphs) instead of degree-sorted
  uint64_t empty_rows = 0;
  uint32_t* orig_ro = nullptr;     // device, original-order full CSR (kept for lz_csr_download)
  uint32_t* orig_ci = nullptr;
  uint32_t* row_ptr = nullptr;     // device, local rows, [n_loc + 1]
  uint32_t* col = nullptr;         // device, [nnz_loc], NEW global column ids, ascending within a row
  uint32_t* new2old = nullptr;     // device, [n_loc * world]; 0xFFFFFFFF for padding slots
  // Column blocking: the gathered vector is cut into ncolblk windows small enough to stay L2-resident; pass b of the
  // SpMV handles the entries of every row whose column lies in window b. col[] is stored column-block-major, and
  // seg[b] is the row pointer of block b ([n_loc + 1] entries, absolute positions into col[]).
  uint32_t ncolblk = 1;
  uint32_t* seg[LZ_MAX_COLBLK + 1] = {};
  uint32_t* seg_store = nullptr;   // device, [ncolblk][n_loc + 1]
  // Sliced layout used by the default SpMV (LZ_SPMV_AUTO): per column block, work items of 32 lanes.
  //   item <  n_long : one long row (total length > LZ_SELL_LONG); its block slice is padded to a multiple of 32, lane l
  //                    reads entries l, l+32, ... (warp per row, coalesced along the row)
  //   item >= n_long : 32 consecutive rows, lane l owns row n_long + 32*(item - n_long) + l; entry j of the 32 rows is
  //                    stored contiguously (sliced ELLPACK, slice height 32; rows are length-sorted so padding is small)
  // sell_sp[b * n_items + item] = offset of the item in sell_col in units of 32 entries; padding = 0xFFFFFFFF.
  uint32_t n_long = 0, n_items = 0;
  uint32_t* sell_sp = nullptr;     // device, [ncolblk * n_items + 1]
  uint32_t* sell_col = nullptr;    // device
  uint64_t sell_entries = 0;       // padded entries stored (all blocks)
  bool sell_narrow[LZ_MAX_COLBLK] = {};   // block b (natural order only): mean width of the 32-row slices <= 6 -> batched-quad instantiation of the kernel
  lz_spmv_plan plan_auto[LZ_MAX_COLBLK] = {}, plan_warp{};
  int spmv_variant = LZ_SPMV_AUTO;
  uint32_t spmv_ctas_per_sm = 6;   // persistent SpMV grid = sm_count * this
  uint32_t push_ctas = 0;          // sender CTAs fused into an SpMV pass (0 = sm_count / 4; LZ_PUSH_CTAS)
  uint32_t sell_group_force = 0;   // 0 = automatic; 1 or 4 = items per work unit of the sliced kernel (LZ_SELL_GROUP, tests)

  // ---- vectors ----------------------------------------------------------------------------------------------------
  uint64_t vec_n = 0, vec_nloc = 0; // graph size the vectors below were allocated for
  uint32_t k_cap = 0;              // rows allocated in V
  uint32_t k_done = 0;             // steps of the last run
  int reorth_done = 0;
  double* V = nullptr;             // device, [k_cap][ldv] basis, vector-contiguous (parallel-mult-on-card layout); null in fp32-basis mode
  // fp32-basis mode (LZ_BASIS_F32): the basis is stored as floats; the recurrence itself runs on a ring of three fp64 vectors
  // (u_{j-1}, u_j, u_{j+1}) plus the fp64 start vector, so alpha/beta are those of the fp64 run and only the consumers of V
  // (full reorthogonalisation, multOut, lz_get_basis) see rounded vectors.
  bool basis_f32 = false;
  float* V32 = nullptr;            // device, [k_cap][ldv]
  double* ring[3] = {};            // device, [ldv] each
  double* q0_64 = nullptr;         // device, [ldv] normalised start vector
  double* w = nullptr;             // device, [n_loc]
  double* xfull = nullptr;         // device, [n_loc * world] gathered Krylov vector (world > 1), else unused
  double* xstage = nullptr;        // device, [n] staging for host vectors in original order
  double* ans = nullptr;           // device, [n_loc]
  double* alpha = nullptr;         // device, [k_cap]
  double* beta = nullptr;          // device, [k_cap]
  double* norm2v = nullptr;        // device, [k_cap + 1]: ||V[j]||^2 of the last run when the basis is stored unnormalised (lagged_done)
  bool lagged = true;              // use the lagged normalisation where it applies (one GPU, no reorthogonalisation); LZ_LAGGED_NORM=0 disables
  bool lagged_done = false;        // the last run left rows 1.. of V unnormalised
  bool lagged_run = false;         // set by the step loop that is being enqueued
  double* scal = nullptr;          // device scalars: [0]=alpha acc, [1]=norm2 acc, [2]=||2^-x_exp x||^2, [5]=log scale of the last
                                   // coefficient solve (lz_get_matfun_scale), [6]=max|x| (bits), others: scratch of the step loop and set-up
  int x_exp = 0;                   // exponent of max|x|: x is scaled by 2^-x_exp before squaring, so ||x|| neither overflows nor underflows
  double* partials = nullptr;      // device, per-CTA partial sums
  uint32_t partials_cap = 0;
  unsigned int* ticket = nullptr;  // device, last-block counters
  double* hcoef = nullptr;         // device, [k_cap] reorth coefficients / multOut coefficients
  double* eigvals = nullptr;       // device, [k_cap]
  double* eigvecs = nullptr;       // device, [k_cap * k_cap] (row-major, dstevd layout), + scratch of same size
  double* eigwork = nullptr;
  double* coef = nullptr;          // device, [k_cap]
  int* status = nullptr;           // device: [0] eigensolver status, [1] reorth skip flag, [2] second-pass counter
  int matfun_kind = LZ_MATFUN_EXP; // function the coefficient solve applies (lz_set_matfun); kept across runs and start vectors
  double matfun_param = 1.0;
  bool have_x = false, have_tridiag = false, have_coef = false, have_ans = false;
  // top Ritz pairs of the run numbered ritz_run (lz_ritz): valid while have_tridiag && ritz_run == run_serial, so anything that drops
  // the run (new run, start vector, graph, basis precision) drops them too
  uint64_t run_serial = 0, ritz_run = 0;
  uint32_t ritz_m = 0, ritz_rows = 0;   // pairs held; rows allocated in R
  double* ritz_R = nullptr;             // device, [ritz_rows][ldv]: y_j, this rank's rows
  double ritz_theta[16] = {}, ritz_rho[16] = {}, ritz_res[16] = {}, ritz_lo = 0.0, ritz_hi = 0.0;
  void* flush_buf = nullptr;
  size_t flush_bytes = 0;

  // ---- CUDA graph of the k-step loop (single GPU, small problems) ----------------------------------------------
  cudaGraphExec_t graph_exec = nullptr;
  uint32_t graph_k = 0, graph_launches = 0;
  int graph_reorth = 0, graph_variant = 0;
  double* graph_V = nullptr;
  uint64_t graph_epoch = 0, epoch = 0;   // epoch: bumped whenever the graph data or the vectors are re-created

  // ---- ranking (lz_rank.cu) -------------------------------------------------------------------------------------------
  void* rank_state = nullptr;              // device, radix-select state
  unsigned long long* rank_key = nullptr;  // device, [rank_cap] candidate keys (m per rank)
  uint32_t* rank_idx = nullptr;            // device, [rank_cap] candidate original vertex ids
  uint32_t* rank_out_idx = nullptr;        // device, sorted result
  double* rank_out_val = nullptr;
  uint32_t rank_cap = 0;

  // ---- measurement ------------------------------------------------------------------------------------------------
  bool profiling = false;
  std::vector<cudaEvent_t> ev_pool;
  size_t ev_used = 0;
  lz_timings tm{};
  unsigned long long* trace_buf = nullptr;   // device, lz_debug_trace
  uint32_t trace_cap = 0;
  uint32_t launches = 0;
};

// lz_graph.cu
int lz_ingest_device_csr(lz_ctx* c, uint64_t n, uint64_t nnz, uint32_t* ro_d, uint32_t* ci_d);  // takes ownership of ro_d / ci_d
void lz_free_graph(lz_ctx* c);
int lz_build_push_lists(lz_ctx* c);   // collective; call after the peers are mapped
// lz_rank.cu
void lz_free_rank(lz_ctx* c);

// lz_kernels.cu — all launches are asynchronous on c->stream
int lz_k_spmv_dot(lz_ctx* c, const double* x_gather, const double* q_local, double* w_out, double* alpha_out /* device scalar or null */,
                  unsigned long long wait_seq = 0 /* > 0: pass b first waits until chunk b of x_gather has arrived from every rank */,
                  const double* push_src = nullptr /* sliced variant only: pass b also sends chunk b + 1 of this local vector */,
                  unsigned long long red_seq = 0 /* > 0 (sliced variant): alpha partial is published to all ranks instead of stored */,
                  const double* alpha_div = nullptr /* device scalar: alpha_out = (w . q) / *alpha_div (lagged normalisation) */);
// lagged normalisation (one GPU, plain recurrence): see k_update_lagged
int lz_k_update_lagged(lz_ctx* c, const double* t, const double* uj, const double* uprev, const double* alpha, const double* norm2_j,
                       const double* norm2_prev, double* u_next, double* norm2_out, double* beta_out, float* u32_next = nullptr);
// dst32 != null: dst32 = (float)src64 ; else dst64 = (double)src32
int lz_k_convert(lz_ctx* c, const double* src64, float* dst32, const float* src32, double* dst64, uint64_t n);
// lagged normalisation on several GPUs (peer exchange + peer scalars): see k_update_lagged_push
int lz_k_update_lagged_push(lz_ctx* c, const double* t, const double* uj, const double* uprev, double* u_next, uint32_t j,
                            unsigned long long push_seq, uint32_t push_chunks, unsigned long long red_seq, float* u32_next = nullptr);
int lz_k_lagged_finish(lz_ctx* c, uint32_t j, unsigned long long red_seq);
int lz_k_set_trace(lz_ctx* c, unsigned long long* buf_device);   // device timeline on (buffer) / off (null)
int lz_k_set_peer_timeout(lz_ctx* c, double seconds);   // watchdog of the in-kernel peer waits; <= 0 disables it
int lz_k_coef_scale(lz_ctx* c, const double* coef, const double* norm2, uint32_t k, double* out);
int lz_k_div_sqrt(lz_ctx* c, double* v, uint64_t n, const double* norm2);
int lz_k_update_norm(lz_ctx* c, double* w, const double* qj, const double* qprev, double* alpha, const double* beta_prev,
                     double* norm2_out /* device scalar or null */, unsigned long long red_seq = 0 /* > 0: scalars go through the peer exchange */);
// q_next = w / sqrt(*norm2); when xfull != null also stores it into this rank's slots of the chunk-major gathered vector
int lz_k_scale(lz_ctx* c, const double* w, const double* norm2, double* q_next, double* xfull, double* beta_out, float* q32_next = nullptr);
// peer exchange: q_next = w / sqrt(*norm2) (norm2 == null: plain copy of w) stored locally and into every rank's gathered vector; raises seq
int lz_k_scale_push(lz_ctx* c, const double* w, const double* norm2, double* q_next, double* beta_out, unsigned long long seq,
                    uint32_t push_chunks /* chunks [0, push_chunks) are sent here; the rest by the SpMV passes */,
                    unsigned long long red_seq = 0);
// q0_local[l] = 2^-x_exp x_orig[new2old[slot(l)]] / sqrt(*norm2)
int lz_k_permute_in_local(lz_ctx* c, const double* x_orig, const double* norm2, double* q0_local);
// local vector <-> this rank's slots of the chunk-major gathered vector
int lz_k_spread(lz_ctx* c, const double* local, double* xfull);
int lz_k_collect(lz_ctx* c, const double* xfull, double* local);
// *out = ||2^-e v||^2
int lz_k_norm2(lz_ctx* c, const double* v, uint64_t len, int e, double* out);
// *out = max(*out, bits of max_i |v[i]|) (NaN > inf > finite as integers)
int lz_k_absmax_bits(lz_ctx* c, const double* v, uint64_t len, unsigned long long* out);
// V: the basis, [nvec][ldv] doubles, or floats when f32 (LZ_BASIS_F32)
int lz_k_multidot(lz_ctx* c, const void* V, bool f32, uint32_t nvec, const double* w, double* h_out /* device [nvec] */, const int* skip = nullptr,
                  const double* h_div = nullptr /* h[t] /= h_div[t]: unnormalised basis rows */);
int lz_k_combine(lz_ctx* c, const void* V, bool f32, uint32_t nvec, const double* coef, double coef_sign, const double* base, double* out,
                 double* norm2_out /* device scalar or null */, const int* skip = nullptr, float* out32 = nullptr /* fp32 copy of out */);
int lz_k_reorth_decide(lz_ctx* c, const double* norm2_before, const double* norm2_after, int* skip, unsigned int* second_passes);
int lz_k_reorth_select(lz_ctx* c, const int* skip, const double* norm2_second, double* norm2, double* norm2_copy = nullptr, double* beta_out = nullptr);
// eigensolver status word: bits 0-29 = 1 + index of an eigenvalue that did not converge, bit 30 = coefficients not finite,
// bit 31 = resolvent denominator 1 - alpha*theta <= 0 for some Ritz value theta
constexpr int kStatusIndefinite = (int)0x80000000u;
int lz_k_tridiag_expv(lz_ctx* c, uint32_t k);   // the ctx's result; log scale -> scal[5]
// ls_in: shift to use for LZ_MATFUN_EXP_SCALED instead of the block's own (null: own); ls_out (may be null) receives the one used
int lz_k_tridiag_expv_into(lz_ctx* c, uint32_t k, double* eigvals, double* eigvecs, double* work, double* coef, int* status,
                           const double* ls_in, double* ls_out);
// dst[i] = x_orig[new2old[first + i]] (times 2^-x_exp / sqrt(*norm2) when norm2 != null), i < count; padding slots -> 0
int lz_k_permute_in(lz_ctx* c, const double* x_orig, const double* norm2, uint64_t first, uint64_t count, double* dst);
int lz_k_permute_out(lz_ctx* c, const double* y_new_full, double* y_orig);
int lz_k_fill(lz_ctx* c, double* p, uint64_t n, double value);
int lz_k_reserve_partials(lz_ctx* c, uint64_t count);
// top Ritz pairs (lz_ritz). partials: caller scratch of 2 * 16 * 8 * sm_count doubles (the loop's c->partials is baked into its CUDA
// graph and must not be regrown here).
// theta[j] = eigvals[k-1-j], W[t*M + j] = eigvecs[t*k + k-1-j] / (norm2 ? sqrt(norm2[t]) : 1) for j < m, 0 for m <= j < M
int lz_k_ritz_select(lz_ctx* c, uint32_t k, uint32_t m, uint32_t M, const double* eigvals, const double* eigvecs, const double* norm2, double* W,
                     double* theta);
// Y[j][0..n_loc) = sum_t W[t*M + j] V[t] for j < M (M = 2, 4, 8, 16), rows of Y ldv apart; ||y_j||^2 -> nrm2[j], sum_i y_j(i) -> vsum[j]
int lz_k_ritz_combine(lz_ctx* c, const void* V, bool f32, uint32_t k, uint32_t M, const double* W, double* Y, double* partials, double* nrm2,
                      double* vsum);
int lz_k_vsum(lz_ctx* c, const double* v, uint64_t n, double* partials, double* out);
// y_j *= sgn(vsum[j]) / sqrt(nrm2[j]), j < m; max |y_0| -> *absmax0 (bit pattern of a double; zero it first)
int lz_k_ritz_scale(lz_ctx* c, double* Y, uint32_t m, const double* nrm2, const double* vsum, unsigned long long* absmax0);
// z[i] = max(|y[i]|, delta * *absmax), i < n
int lz_k_cw_z(lz_ctx* c, const double* y, double* z, uint64_t n, const double* absmax, double delta);
// *out = max(*out, max over this rank's vertices of az[l] / zfull[slot(l)]) (bit pattern of a non-negative double)
int lz_k_cw_bound(lz_ctx* c, const double* az, const double* zfull, unsigned long long* out);
