// lz_kernels.cu — hand-written sm_100a kernels of the Lanczos e^A·x hot path. Every kernel is HBM/L2-bandwidth bound
// fp64 streaming or gather work (<= 0.25 flop/byte): no tensor-core shapes anywhere.
//
//   k_spmv_sell / k_spmv_dot   w = A x  (value-less gather-sum; sliced-ELLPACK default, CSR variants) fused with the partial of
//                   alpha = w . q_j; on several GPUs also the consumer (acquire-spin on chunk arrival) and, through a few sender
//                   CTAs, the producer of the NVLink exchange. Replaces cu_spMV1 + cu_dot_prod + cu_reduce (reference
//                   parallel-final/lib/cu_SPMV.cu:31-41, cu_linalg.cu:67-131; launches at cu_lanczos.cu:101-105)
//   k_update_lagged            one GPU: u_{j+1} = (t - alpha u_j)/||u_j|| - (||u_j||/||u_{j-1}||) u_{j-1}, partial of ||u_{j+1}||^2 — ONE pass;
//                   the normalisation is lagged into the consumers. Replaces cu_dpax x2 + cu_norm_sq + cu_reduce_sqrt + cu_dvexda
//                   (cu_linalg.cu:223-226,184-208,146-170,241-244; cu_lanczos.cu:108-123) and the per-step D2H of q_j (:126)
//   k_update_lagged_push       several GPUs: the same pass fused with both cross-GPU scalar reductions (peer memory) and with the
//                   peer stores of u_{j+1} into every rank's gathered vector (whole chunks, or entry-wise for band-like graphs).
//                   Generalises parallel-two-cards/lib/cu_lanczos.cu:116-165
//   k_update_norm, k_scale, k_scale_push[_sparse]   the reference-shaped two-kernel step (fallback paths, multi-GPU reorthogonalisation)
//   k_multidot      h = V_j^T w   (tall-skinny GEMV-T) for full reorthogonalisation (precedent: serial/lib/lanczos.cc:85-91)
//   k_combine       out = base + s * V^T-combination: reorth update  w -= V h  and  multOut  ans = V c; fp64 or fp32 basis rows
//                   replaces cblas_dgemv / cublasDgemv (multiplyOut.cu:43-47, parallel-mult-on-card/lib/cu_multiplyOut.cu:66-72)
//   k_tridiag_expv  eigen-decomposition of the k x k tridiagonal (implicit-shift QL) + c = ||x|| Z (e^lambda . Z^T e1)
//                   replaces LAPACKE_dstevd (eigen.cu:17-21) and multiplyOut.cu:30-40
// (the ranking kernels are in lz_rank.cu, graph construction in lz_graph.cu)
//
// All grid-wide reductions are deterministic: per-CTA partials in a fixed slot, summed in a fixed order by the last CTA
// to finish (ticket counter), result left in device memory so the next kernel reads it without a host round-trip —
// the same "scalars never visit the host" property as the reference (cu_linalg.cu:223-226 take T* device scalars).
#include "lz_ctx.h"

#include <math.h>
#include <stdlib.h>
#include <string.h>

namespace {

constexpr int kBlock = LZ_SPMV_BLOCK;
constexpr int kWarps = kBlock / 32;

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// Sum over the CTA; result valid in thread 0. `sm` has kWarps doubles.
__device__ __forceinline__ double block_sum(double v, double* sm) {
  v = warp_sum(v);
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  __syncthreads();   // protect sm from a previous use
  if (lane == 0) sm[wid] = v;
  __syncthreads();
  if (wid == 0) {
    v = (lane < kWarps) ? sm[lane] : 0.0;
    v = warp_sum(v);
  }
  return v;
}

// ---- scalar all-reduce over peer memory (multi-GPU, plain Lanczos) ------------------------------------------------
// Each rank's reduction kernel publishes its partial (value, then sequence number with release semantics) in slot
// [kind][seq & 1][rank] of EVERY rank's exchange area; the consuming kernel spins until all `world` slots carry `seq`
// and adds them in rank order, so all ranks obtain the bit-identical sum without a collective launch in between.
// Two parities suffice: a rank can be at most one reduction of a kind ahead of its slowest peer (the vector exchange
// of the step in between needs every rank's contribution).
// Watchdog of the in-kernel spins (wait_chunk, red_consume): nanoseconds after which a peer that never arrives turns into a
// launch failure (__trap: the CUDA context is then unusable and must be destroyed) instead of a silent hang. 0 = wait for ever,
// which is what NCCL would do. Set per device from LZ_PEER_TIMEOUT_S (default 20 s) by lz_k_set_peer_timeout.
__device__ unsigned long long g_peer_timeout_ns = 20000000000ull;

// Optional device-side timeline (lz_debug_trace): (tag, globaltimer) pairs appended by a few designated threads, so the waits on
// peers inside the kernels can be told apart from their work. Off (null) unless the measurement hook switches it on.
__device__ unsigned long long* g_trace = nullptr;      // [0] = number of events so far, [1] = capacity, events from [2]
__device__ __forceinline__ void trace_mark(unsigned long long tag) {
  unsigned long long* tr = g_trace;
  if (!tr) return;
  const unsigned long long i = atomicAdd(tr, 1ull);
  if (i < tr[1]) {
    unsigned long long now;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(now));
    tr[2 + 2 * i] = tag;
    tr[3 + 2 * i] = now;
  }
}
// tags: kernel << 8 | phase.  kernel: 0x10 + column block = SpMV pass, 0x01 = update/push, 0x02 = scale/push (unlagged)
#define LZ_TR(kernel, phase) (((unsigned)(kernel) << 8) | (unsigned)(phase))
enum { TR_START = 1, TR_WAITED = 2, TR_PUSHED = 3, TR_END = 4, TR_SEND_START = 5, TR_SEND_END = 6 };

struct lz_red_slot { double val; unsigned long long seq; };
struct lz_red {
  lz_red_slot* area[LZ_MAX_WORLD];   // exchange area of every rank as seen from this GPU: [2 kinds][2][LZ_MAX_WORLD]
  unsigned long long seq;           // 0 = disabled (single GPU / NCCL path): plain device scalars are used
  uint32_t world, rank;
};
__device__ __forceinline__ void red_publish(const lz_red& red, int kind, double v) {
  const size_t idx = ((size_t)kind * 2 + (red.seq & 1)) * LZ_MAX_WORLD + red.rank;
  for (uint32_t r = 0; r < red.world; r++) red.area[r][idx].val = v;      // all values first ...
  __threadfence_system();                                                 // ... one fence ...
  for (uint32_t r = 0; r < red.world; r++)                                // ... then the sequence numbers (relaxed: the fence is the release)
    asm volatile("st.relaxed.sys.global.u64 [%0], %1;" ::"l"(&red.area[r][idx].seq), "l"(red.seq) : "memory");
}
// All threads of the CTA call this; returns the total of reduction `seq` of `kind` in every thread.
__device__ __forceinline__ double red_consume_seq(const lz_red& red, int kind, unsigned long long seq, double* sm_bcast) {
  __syncthreads();   // sm_bcast may still be read from a previous call
  if (threadIdx.x == 0) {
    const lz_red_slot* base = red.area[red.rank] + ((size_t)kind * 2 + (seq & 1)) * LZ_MAX_WORLD;
    const unsigned long long limit = g_peer_timeout_ns;
    double tot = 0.0;
    for (uint32_t r = 0; r < red.world; r++) {
      unsigned long long got, t0 = 0;
      unsigned int spins = 0;
      for (;;) {
        asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(got) : "l"(&base[r].seq) : "memory");
        if (got >= seq) break;
        __nanosleep(32);
        if (limit && (++spins & 0xFFFFu) == 0) {
          unsigned long long now;
          asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(now));
          if (t0 == 0) t0 = now;
          else if (now - t0 > limit) __trap();
        }
      }
      tot += *reinterpret_cast<const volatile double*>(&base[r].val);
    }
    *sm_bcast = tot;
  }
  __syncthreads();
  return *sm_bcast;
}
__device__ __forceinline__ double red_consume(const lz_red& red, int kind, double* sm_bcast) {
  return red_consume_seq(red, kind, red.seq, sm_bcast);
}

// Basis storage: fp64, or fp32 (LZ_BASIS_F32: half the bytes of every pass over V; all arithmetic stays fp64). Every thread
// moves 16 bytes per load either way: a group of kEpt<TV> consecutive entries (2 doubles or 4 floats).
template <class TV> struct ept { static constexpr int value = 16 / sizeof(TV); };
template <class TV> __device__ __forceinline__ void ld_group(const TV* base, uint64_t g, double (&v)[ept<TV>::value]);
template <> __device__ __forceinline__ void ld_group<double>(const double* base, uint64_t g, double (&v)[2]) {
  const double2 d = __ldcs(reinterpret_cast<const double2*>(base) + g);
  v[0] = d.x; v[1] = d.y;
}
template <> __device__ __forceinline__ void ld_group<float>(const float* base, uint64_t g, double (&v)[4]) {
  const float4 f = __ldcs(reinterpret_cast<const float4*>(base) + g);
  v[0] = (double)f.x; v[1] = (double)f.y; v[2] = (double)f.z; v[3] = (double)f.w;
}

// Deterministic grid reduction tail. Thread 0 of every CTA passes its CTA value; the last CTA to arrive sums all
// `gridDim.x` partials in index order (strided per thread, then a fixed tree) and stores op(sum) to *out.
__device__ __forceinline__ void grid_sum_finish(double cta_val, double* partials, unsigned int* ticket, double* out, double* sm,
                                                bool* s_last, unsigned int cta = 0xFFFFFFFFu, unsigned int nctas = 0,
                                                const lz_red* red = nullptr, int kind = 0, const double* out_div = nullptr) {
  if (cta == 0xFFFFFFFFu) { cta = blockIdx.x; nctas = gridDim.x; }   // default: every CTA of the grid takes part
  if (threadIdx.x == 0) {
    partials[cta] = cta_val;
    __threadfence();
    unsigned int t = atomicAdd(ticket, 1u);
    *s_last = (t == nctas - 1);
  }
  __syncthreads();
  if (*s_last) {
    __threadfence();
    double acc = 0.0;
    for (unsigned int i = threadIdx.x; i < nctas; i += kBlock) acc += __ldcg(partials + i);
    acc = block_sum(acc, sm);
    if (threadIdx.x == 0) {
      if (red && red->seq) red_publish(*red, kind, acc);   // multi-GPU: the partial goes to every rank's exchange area
      else *out = out_div ? acc / *out_div : acc;   // lagged normalisation: alpha = (A u . u) / ||u||^2
      *ticket = 0u;
    }
  }
}

// ---- peer exchange over NVLink ---------------------------------------------------------------------------------------
struct lz_peers {
  double* x[LZ_MAX_WORLD];
  unsigned long long* f[LZ_MAX_WORLD];
};

struct lz_push_job {     // work of the sender CTAs fused into an SpMV pass (nctas == 0: none)
  lz_peers peers;
  const double* src;
  unsigned int* ticket;
  unsigned long long seq;
  uint64_t cl;
  uint32_t chunk, rank, nctas;
};

__device__ __forceinline__ unsigned long long ld_acquire_sys(const unsigned long long* p) {
  unsigned long long v;
  asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
  return v;
}
// Flag / sequence-number store of the release pattern "fence.acq_rel.sys ; st.relaxed.sys": every caller issues ONE
// __threadfence_system() after its data stores and then publishes to all ranks with relaxed system-scope stores. A
// st.release.sys per destination would repeat the fence (SASS: MEMBAR.ALL.SYS before every STG.STRONG.SYS — 8 serialised
// system-wide barriers by one thread on the critical path of every chunk arrival at 8 GPUs).
__device__ __forceinline__ void st_relaxed_sys(unsigned long long* p, unsigned long long v) {
  asm volatile("st.relaxed.sys.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}

// Consumer side: block until chunk `blk` of the gathered vector has been written by every rank (counter >= seq).
// The producers are kernels on OTHER GPUs that never wait for this GPU's SpMV (see DESIGN.md section 4), so this cannot deadlock.
__device__ __forceinline__ void wait_chunk(const unsigned long long* flags, uint32_t blk, uint32_t world, unsigned long long seq) {
  if (seq == 0) return;
  if (threadIdx.x < world) {
    const unsigned long long* f = flags + (uint64_t)blk * LZ_MAX_WORLD + threadIdx.x;
    const unsigned long long limit = g_peer_timeout_ns;
    unsigned long long t0 = 0;
    unsigned int spins = 0;
    while (ld_acquire_sys(f) < seq) {
      __nanosleep(64);
      if (limit && (++spins & 0xFFFFu) == 0) {             // watchdog: a lost peer becomes a launch failure, not a hang
        unsigned long long now;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(now));
        if (t0 == 0) t0 = now;
        else if (now - t0 > limit) __trap();
      }
    }
  }
  __syncthreads();
}

// Producer side: copy chunk `c` of this rank's local vector `src` (already normalised) into the chunk-major gathered vector
// of every rank (16-byte peer stores over NVLink), then — once all `nctas` participating CTAs are done — publish `seq` in
// every rank's arrival counter for (chunk c, this rank). `cta` is this CTA's index among the participants.
__device__ __forceinline__ void push_chunk(const double* __restrict__ src, const lz_peers& peers, uint32_t c, uint64_t cl, uint32_t world,
                                           uint32_t rank, unsigned long long seq, unsigned int* ticket, uint32_t cta, uint32_t nctas,
                                           bool* s_flag) {
  const uint64_t cl2 = cl >> 1;
  const uint64_t slot2 = ((uint64_t)c * world * cl + (uint64_t)rank * cl) >> 1;
  const double2* s2 = reinterpret_cast<const double2*>(src) + (uint64_t)c * cl2;
  for (uint64_t i = (uint64_t)cta * kBlock + threadIdx.x; i < cl2; i += (uint64_t)nctas * kBlock) {
    const double2 v = s2[i];
    for (uint32_t r = 0; r < world; r++) reinterpret_cast<double2*>(peers.x[r])[slot2 + i] = v;
  }
  __threadfence_system();          // this thread's peer stores are visible system-wide before the CTA reports in
  __syncthreads();
  if (threadIdx.x == 0) {
    const unsigned int t = atomicAdd(ticket + c, 1u);
    *s_flag = (t == nctas - 1);
    if (*s_flag) {
      ticket[c] = 0u;
      __threadfence_system();
      for (uint32_t r = 0; r < world; r++) st_relaxed_sys(peers.f[r] + (uint64_t)c * LZ_MAX_WORLD + rank, seq);
    }
  }
  __syncthreads();
}

// ------------------------------------------------------------------------------------------------------------- SpMV
// Value-less CSR gather-sum. One row is served by L = 2^LG cooperating lanes ("vector per row"; L = 32 is warp per row).
// Local rows are sorted by length, so every row of a bin has len in (L, 2L] (L = 1: len <= 2; L = 32: len > 32): all
// lanes of a warp run the same trip count, and the rows a warp touches are adjacent in col[], so the index stream is
// read in contiguous 128-byte pieces with streaming (evict-first) loads.
//
// The kernel is bound by the rate at which an SM's L1 can look up distinct 128-byte lines (one per clock: 275 G random
// 8-byte gathers/s chip-wide, profiles/microbench/gather_bench_r01.txt), not by DRAM; what matters is keeping ~10^3
// gathers in flight per SM. Each lane group therefore works on R rows at once: all 2R index loads are issued, then all
// 2R gathers, then the sums — and CTAs are persistent (static item-stride loop), so the reduction tail is paid once.
constexpr int kSpmvR = LZ_SPMV_ROWS_PER_GROUP;

// The gathered vector. One GPU: read-only for the whole kernel -> ld.global.nc. Several GPUs: the peers write it while this
// kernel is resident (it starts, acquires the chunk's arrival counters, then reads), so the non-coherent path is not allowed
// there: plain ld.global, which the acquire + bar.sync of wait_chunk orders after the peers' released stores.
template <bool PEER>
__device__ __forceinline__ double ldx(const double* x, uint32_t c) {
  if constexpr (PEER) {
    double v;
    asm volatile("ld.global.f64 %0, [%1];" : "=d"(v) : "l"(x + c));
    return v;
  } else {
    return __ldg(x + c);
  }
}

template <int LG, int PER, bool PEER>
__device__ __forceinline__ double spmv_item(const lz_spmv_bin& bin, uint32_t item, const uint32_t* __restrict__ seg_lo,
                                            const uint32_t* __restrict__ seg_hi, const uint32_t* __restrict__ col,
                                            const double* x, const double* q, double* __restrict__ w,
                                            bool accumulate, bool final_pass) {
  constexpr uint32_t L = 1u << LG;
  constexpr uint32_t GROUPS = kBlock >> LG;
  const uint32_t g = threadIdx.x >> LG, sub = threadIdx.x & (L - 1);
  const uint32_t base = bin.row_begin + item * (GROUPS * kSpmvR) + g;
  uint32_t b[kSpmvR], e[kSpmvR];
  bool valid[kSpmvR];
#pragma unroll
  for (int r = 0; r < kSpmvR; r++) {
    const uint32_t row = base + r * GROUPS;
    valid[r] = row < bin.row_end;
    b[r] = valid[r] ? __ldg(seg_lo + row) : 0u;
    e[r] = valid[r] ? __ldg(seg_hi + row) : 0u;
  }
  double sum[kSpmvR];
  constexpr bool kJoint = (PER * kSpmvR <= 8);   // short slices: first chunk of all R rows at once (PER*R loads in flight)
  if constexpr (kJoint) {
    uint32_t c[kSpmvR][PER];
    bool p[kSpmvR][PER];
#pragma unroll
    for (int r = 0; r < kSpmvR; r++)
#pragma unroll
      for (int u = 0; u < PER; u++) {
        const uint32_t j = b[r] + sub + u * L;
        p[r][u] = j < e[r];
        c[r][u] = p[r][u] ? __ldcs(col + j) : 0u;
      }
    double v[kSpmvR][PER];
#pragma unroll
    for (int r = 0; r < kSpmvR; r++)
#pragma unroll
      for (int u = 0; u < PER; u++) v[r][u] = p[r][u] ? ldx<PEER>(x, c[r][u]) : 0.0;
#pragma unroll
    for (int r = 0; r < kSpmvR; r++) {
      double s = v[r][0];
#pragma unroll
      for (int u = 1; u < PER; u++) s += v[r][u];
      sum[r] = s;
    }
  } else {
#pragma unroll
    for (int r = 0; r < kSpmvR; r++) sum[r] = 0.0;
  }
  // remaining chunks (all chunks for the long-slice variants), row by row, PER loads in flight
#pragma unroll
  for (int r = 0; r < kSpmvR; r++) {
    for (uint32_t j0 = b[r] + sub + (kJoint ? PER * L : 0u); j0 < e[r]; j0 += PER * L) {
      uint32_t cc[PER];
#pragma unroll
      for (int u = 0; u < PER; u++) cc[u] = (j0 + u * L < e[r]) ? __ldcs(col + j0 + u * L) : 0xFFFFFFFFu;
      double vv[PER];
#pragma unroll
      for (int u = 0; u < PER; u++) vv[u] = (cc[u] != 0xFFFFFFFFu) ? ldx<PEER>(x, cc[u]) : 0.0;
      double s = 0.0;
#pragma unroll
      for (int u = 0; u < PER; u++) s += vv[u];
      sum[r] += s;
    }
  }
  double d = 0.0;
#pragma unroll
  for (int r = 0; r < kSpmvR; r++) {
    double s = sum[r];
#pragma unroll
    for (int o = L / 2; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    if (valid[r] && sub == 0) {
      const uint32_t row = base + r * GROUPS;
      if (accumulate) {
        if (final_pass || e[r] > b[r]) {
          s += w[row];
          w[row] = s;
        }
      } else {
        w[row] = s;
      }
      if (final_pass) d += s * q[row];
    }
  }
  return d;
}

// One pass = one column block. accumulate: w += (pass > 0). final_pass: also alpha partial = w . q and the grid reduction.
template <bool PEER>
__global__ void __launch_bounds__(kBlock) k_spmv_dot(const __grid_constant__ lz_spmv_plan plan, const uint32_t* __restrict__ seg_lo,
                                                     const uint32_t* __restrict__ seg_hi, const uint32_t* __restrict__ col,
                                                     const double* x, const double* q, double* __restrict__ w,
                                                     double* partials, unsigned int* ticket, double* alpha_out, int accumulate,
                                                     int final_pass, const unsigned long long* flags, uint32_t blk, uint32_t world,
                                                     unsigned long long wait_seq, const double* alpha_div) {
  __shared__ double sm[kWarps];
  __shared__ bool s_last;
  wait_chunk(flags, blk, world, wait_seq);
  double d = 0.0;
  const bool acc = accumulate != 0, fin = final_pass != 0;
  for (uint32_t item = blockIdx.x; item < plan.nitems; item += gridDim.x) {
    uint32_t bi = 0;
#pragma unroll
    for (uint32_t i = 1; i < LZ_MAX_BINS; i++)
      if (i < plan.nbins && item >= plan.bin[i].item_begin) bi = i;
    const lz_spmv_bin& bin = plan.bin[bi];
    const uint32_t it = item - bin.item_begin;
#define LZ_SPMV_CASE(LG, PER) d += spmv_item<LG, PER, PEER>(bin, it, seg_lo, seg_hi, col, x, q, w, acc, fin)
    switch (bin.log2_lanes) {
      case 5:
        if (bin.per_lane == 2) LZ_SPMV_CASE(5, 2);
        else LZ_SPMV_CASE(5, 8);
        break;
      case 4: LZ_SPMV_CASE(4, 2); break;
      case 3: LZ_SPMV_CASE(3, 2); break;
      case 2: LZ_SPMV_CASE(2, 2); break;
      case 1: LZ_SPMV_CASE(1, 2); break;
      default: LZ_SPMV_CASE(0, 2); break;
    }
#undef LZ_SPMV_CASE
  }
  if (fin) {
    d = block_sum(d, sm);
    grid_sum_finish(d, partials, ticket, alpha_out, sm, &s_last, 0xFFFFFFFFu, 0, nullptr, 0, alpha_div);
  }
}

// ---------------------------------------------------------------------------------------- SpMV, sliced layout (default)
// One warp per work item (lz_ctx.h): a long row read along the row, or 32 consecutive short rows read "one entry of every
// row" at a time. Either way the index stream is consumed as whole 128-byte lines (one L1 wavefront per 32 gathers),
// there are no per-row pointer loads and — for the short-row items, i.e. almost all of the matrix — no shuffles: the
// gathers themselves are all that is left on the SM's load path, which is what bounds this kernel (1 line/clk/SM).
// NARROW (column blocks whose slices are only a few entries wide: band-like graphs in natural order, the cold column block
// of a degree-sorted graph): a quad of up to 8-wide slices is processed 4 chunks x 4 items at a time, 16 gathers per lane
// in flight instead of one slice's 3-6 — such a block is latency-bound otherwise. Costs registers (3 CTAs/SM instead of
// 6), so it is a separate instantiation chosen per column block at ingest. Summation order per row is unchanged.
constexpr int kSellU = 8;   // chunks (gathers per lane) in flight
template <bool NARROW, bool PEER>
__global__ void __launch_bounds__(kBlock, NARROW ? 4 : 6) k_spmv_sell(const uint32_t* __restrict__ sp, const uint32_t* __restrict__ scol, uint32_t n_long,
                                                      uint32_t n_items, uint32_t n_loc, const double* x,
                                                      const double* q, double* __restrict__ w, double* partials,
                                                      unsigned int* ticket, double* alpha_out, int accumulate, int final_pass,
                                                      const unsigned long long* flags, uint32_t blk, uint32_t world,
                                                      unsigned long long wait_seq, const __grid_constant__ lz_push_job job,
                                                      uint32_t group, const __grid_constant__ lz_red red, const double* alpha_div) {
  __shared__ double sm[kWarps];
  __shared__ bool s_last;
  // Fused exchange: the first job.nctas CTAs of pass `blk` send chunk job.chunk (= blk + 1) of the new Krylov vector to
  // every rank while the remaining CTAs gather from chunk blk. Senders never wait, gatherers wait only for data sent by
  // strictly earlier launches on every rank, so the scheme cannot deadlock whatever the CTA placement.
  if (blockIdx.x < job.nctas) {
    if (blockIdx.x == 0 && threadIdx.x == 0) trace_mark(LZ_TR(0x10 + blk, TR_SEND_START));
    push_chunk(job.src, job.peers, job.chunk, job.cl, world, job.rank, job.seq, job.ticket, blockIdx.x, job.nctas, &s_last);
    if (s_last && threadIdx.x == 0) trace_mark(LZ_TR(0x10 + blk, TR_SEND_END));
    if (threadIdx.x == 0 && g_trace && g_trace[1] >= 65536) {   // detailed mode: every sender CTA's end, with its SM id
      unsigned smid;
      asm volatile("mov.u32 %0, %%smid;" : "=r"(smid));
      trace_mark(LZ_TR(0x10 + blk, 8) | (smid << 16) | (blockIdx.x << 24));
    }
    return;
  }
  const uint32_t cta = blockIdx.x - job.nctas, nctas = gridDim.x - job.nctas;
  if (cta == 0 && threadIdx.x == 0) trace_mark(LZ_TR(0x10 + blk, TR_START));
  wait_chunk(flags, blk, world, wait_seq);
  if (cta == 0 && threadIdx.x == 0) trace_mark(LZ_TR(0x10 + blk, TR_WAITED));
  const uint32_t lane = threadIdx.x & 31;
  const uint32_t nwarps = nctas * kWarps;
  double d = 0.0;
  // Work is handed out in quads of consecutive items. Consecutive slices have similar widths (rows are length-sorted), and
  // most slices of a sparse column block are only one or two entries wide: such a quad is processed as one batch (all
  // index loads, then all gathers) so a warp keeps ~8 gathers per lane in flight instead of 1-2.
  // (group = 4 on large inputs; 1 when there are too few items to keep every warp busy with quads.)
  const uint32_t n_units = (n_items + group - 1) / group;
  for (uint32_t unit = cta * kWarps + (threadIdx.x >> 5); unit < n_units; unit += nwarps) {
    const uint32_t first = unit * group;
    uint32_t off[5];
#pragma unroll
    for (int t = 0; t < 5; t++) off[t] = (group == 4) ? __ldg(sp + min(first + t, n_items)) : 0u;
    const uint32_t wmax = max(max(off[1] - off[0], off[2] - off[1]), max(off[3] - off[2], off[4] - off[3]));
    if (NARROW && group == 4 && wmax <= 8 && first >= n_long) {
      // one base pointer and one width per slice; the two rounds are unrolled so every index load is base + immediate
      const uint32_t* pt[4];
      uint32_t wd[4];
#pragma unroll
      for (int t = 0; t < 4; t++) { wd[t] = off[t + 1] - off[t]; pt[t] = scol + (uint64_t)off[t] * 32 + lane; }
      double acc[4] = {0.0, 0.0, 0.0, 0.0};
#pragma unroll
      for (int round = 0; round < 2; round++) {
        if (round == 1 && wmax <= 4) break;
        uint32_t cc[4][4];
#pragma unroll
        for (int t = 0; t < 4; t++)
#pragma unroll
          for (int u = 0; u < 4; u++) cc[t][u] = ((uint32_t)(round * 4 + u) < wd[t]) ? __ldcs(pt[t] + (round * 4 + u) * 32) : 0xFFFFFFFFu;
        double vv[4][4];
#pragma unroll
        for (int t = 0; t < 4; t++)
#pragma unroll
          for (int u = 0; u < 4; u++) vv[t][u] = (cc[t][u] != 0xFFFFFFFFu) ? ldx<PEER>(x, cc[t][u]) : 0.0;
#pragma unroll
        for (int t = 0; t < 4; t++)
#pragma unroll
          for (int u = 0; u < 4; u++) acc[t] += vv[t][u];
      }
#pragma unroll
      for (int t = 0; t < 4; t++) {
        const uint32_t item = first + t;
        const uint32_t row = n_long + (item - n_long) * 32 + lane;
        if (item < n_items && row < n_loc) {
          double a = acc[t];
          if (accumulate) {
            if (final_pass || off[t + 1] > off[t]) {
              a += w[row];
              w[row] = a;
            }
          } else {
            w[row] = a;
          }
          if (final_pass) d += a * q[row];
        }
      }
      continue;
    }
    if (group == 4 && wmax <= 2 && first >= n_long) {
      uint32_t cc[4][2];
#pragma unroll
      for (int t = 0; t < 4; t++)
#pragma unroll
        for (int u = 0; u < 2; u++)
          cc[t][u] = (off[t] + u < off[t + 1]) ? __ldcs(scol + (uint64_t)(off[t] + u) * 32 + lane) : 0xFFFFFFFFu;
      double vv[4][2];
#pragma unroll
      for (int t = 0; t < 4; t++)
#pragma unroll
        for (int u = 0; u < 2; u++) vv[t][u] = (cc[t][u] != 0xFFFFFFFFu) ? ldx<PEER>(x, cc[t][u]) : 0.0;
#pragma unroll
      for (int t = 0; t < 4; t++) {
        const uint32_t item = first + t;
        const uint32_t row = n_long + (item - n_long) * 32 + lane;
        if (item < n_items && row < n_loc) {
          double acc = vv[t][0] + vv[t][1];
          if (accumulate) {
            if (final_pass || off[t + 1] > off[t]) {
              acc += w[row];
              w[row] = acc;
            }
          } else {
            w[row] = acc;
          }
          if (final_pass) d += acc * q[row];
        }
      }
      continue;
    }
    if (!NARROW && group == 4 && wmax <= 4 && first >= n_long) {
      // slices 3-4 entries wide (most of a cold column block): two slices at a time, 8 gathers per lane in flight instead of the
      // 3-4 of a single slice; same summation order per row (entry 0, 1, 2, 3)
#pragma unroll
      for (int half = 0; half < 2; half++) {
        uint32_t cc[2][4];
#pragma unroll
        for (int t = 0; t < 2; t++)
#pragma unroll
          for (int u = 0; u < 4; u++)
            cc[t][u] = (off[2 * half + t] + u < off[2 * half + t + 1]) ? __ldcs(scol + (uint64_t)(off[2 * half + t] + u) * 32 + lane) : 0xFFFFFFFFu;
        double vv[2][4];
#pragma unroll
        for (int t = 0; t < 2; t++)
#pragma unroll
          for (int u = 0; u < 4; u++) vv[t][u] = (cc[t][u] != 0xFFFFFFFFu) ? ldx<PEER>(x, cc[t][u]) : 0.0;
#pragma unroll
        for (int t = 0; t < 2; t++) {
          const int tt = 2 * half + t;
          const uint32_t item = first + tt;
          const uint32_t row = n_long + (item - n_long) * 32 + lane;
          if (item < n_items && row < n_loc) {
            double acc = 0.0;
#pragma unroll
            for (int u = 0; u < 4; u++) acc += vv[t][u];
            if (accumulate) {
              if (final_pass || off[tt + 1] > off[tt]) {
                acc += w[row];
                w[row] = acc;
              }
            } else {
              w[row] = acc;
            }
            if (final_pass) d += acc * q[row];
          }
        }
      }
      continue;
    }
    for (uint32_t item = first; item < min(first + group, n_items); item++) {
      const uint32_t c0 = __ldg(sp + item), nchunk = __ldg(sp + item + 1) - c0;
      const uint32_t* p = scol + (uint64_t)c0 * 32 + lane;
      double acc = 0.0;
      uint32_t j = 0;
      for (; j + kSellU <= nchunk; j += kSellU) {
        uint32_t cc[kSellU];
#pragma unroll
        for (int u = 0; u < kSellU; u++) cc[u] = __ldcs(p + (uint64_t)(j + u) * 32);
        double vv[kSellU];
#pragma unroll
        for (int u = 0; u < kSellU; u++) vv[u] = (cc[u] != 0xFFFFFFFFu) ? ldx<PEER>(x, cc[u]) : 0.0;
#pragma unroll
        for (int u = 0; u < kSellU; u++) acc += vv[u];
      }
      if (j < nchunk) {
        const uint32_t rem = nchunk - j;
        uint32_t cc[kSellU];
#pragma unroll
        for (int u = 0; u < kSellU - 1; u++) cc[u] = (u < (int)rem) ? __ldcs(p + (uint64_t)(j + u) * 32) : 0xFFFFFFFFu;
        double vv[kSellU];
#pragma unroll
        for (int u = 0; u < kSellU - 1; u++) vv[u] = (cc[u] != 0xFFFFFFFFu) ? ldx<PEER>(x, cc[u]) : 0.0;
#pragma unroll
        for (int u = 0; u < kSellU - 1; u++) acc += vv[u];
      }
      uint32_t row;
      bool writer;
      if (item < n_long) {
        acc = warp_sum(acc);
        row = item;
        writer = lane == 0;
      } else {
        row = n_long + (item - n_long) * 32 + lane;
        writer = row < n_loc;
      }
      if (writer) {
        if (accumulate) {
          if (final_pass || nchunk) {
            acc += w[row];
            w[row] = acc;
          }
        } else {
          w[row] = acc;
        }
        if (final_pass) d += acc * q[row];
      }
    }
  }
  if (final_pass) {
    d = block_sum(d, sm);
    grid_sum_finish(d, partials, ticket, alpha_out, sm, &s_last, cta, nctas, &red, 0, alpha_div);
    if (s_last && threadIdx.x == 0) trace_mark(LZ_TR(0x10 + blk, TR_END));
  } else if (cta == 0 && threadIdx.x == 0) {
    trace_mark(LZ_TR(0x10 + blk, TR_END));   // CTA 0 only: indicative
  }
  if (threadIdx.x == 0 && g_trace && g_trace[1] >= 65536) {     // detailed mode: every gatherer CTA's end, with its SM id
    unsigned smid;
    asm volatile("mov.u32 %0, %%smid;" : "=r"(smid));
    trace_mark(LZ_TR(0x10 + blk, 7) | (smid << 16) | ((unsigned long long)cta << 24));
  }
}


// --------------------------------------------------------------------------------------------- fused vector update
// w <- (w - alpha q_j) - beta_prev q_prev, partial of ||w||^2. Same operation order as lanczos.cu:36-43.
__global__ void __launch_bounds__(kBlock) k_update_norm(double* __restrict__ w, const double* __restrict__ qj, const double* __restrict__ qp,
                                                        const double* __restrict__ alpha_p, const double* __restrict__ beta_p,
                                                        uint64_t n, double* partials, unsigned int* ticket, double* norm2_out,
                                                        const __grid_constant__ lz_red red, double* alpha_store) {
  __shared__ double sm[kWarps];
  __shared__ bool s_last;
  __shared__ double s_bcast;
  double a;
  if (red.seq) {                       // alpha_j = sum over ranks of the SpMV kernels' partials (peer exchange)
    a = red_consume(red, 0, &s_bcast);
    if (blockIdx.x == 0 && threadIdx.x == 0) *alpha_store = a;
  } else {
    a = *alpha_p;
  }
  const double b = qp ? *beta_p : 0.0;
  const uint64_t n2 = n >> 1;
  double acc = 0.0;
  double2* w2 = reinterpret_cast<double2*>(w);
  const double2* q2 = reinterpret_cast<const double2*>(qj);
  const double2* p2 = reinterpret_cast<const double2*>(qp);
  for (uint64_t i = (uint64_t)blockIdx.x * kBlock + threadIdx.x; i < n2; i += (uint64_t)gridDim.x * kBlock) {
    double2 wv = w2[i];
    const double2 qv = q2[i];
    wv.x -= a * qv.x;
    wv.y -= a * qv.y;
    if (qp) {
      const double2 pv = p2[i];
      wv.x -= b * pv.x;
      wv.y -= b * pv.y;
    }
    w2[i] = wv;
    acc += wv.x * wv.x;
    acc += wv.y * wv.y;
  }
  if ((n & 1) && blockIdx.x == 0 && threadIdx.x == 0) {
    double t = w[n - 1] - a * qj[n - 1];
    if (qp) t -= b * qp[n - 1];
    w[n - 1] = t;
    acc += t * t;
  }
  acc = block_sum(acc, sm);
  if (norm2_out) grid_sum_finish(acc, partials, ticket, norm2_out, sm, &s_last, 0xFFFFFFFFu, 0, &red, 1);
}

// Lagged normalisation (one GPU, plain recurrence): the basis row j >= 1 holds the UNNORMALISED vector u_j = w' of step
// j-1 and norm2[j] = ||u_j||^2, so q_j = u_j / ||u_j|| is formed on the fly and the separate normalisation pass (read w,
// write q: 16 bytes per row and one launch per step) disappears. With t = A u_j and alpha_j = (t . u_j) / ||u_j||^2:
//   u_{j+1} = t/||u_j|| - alpha_j q_j - beta_{j-1} q_{j-1},   beta_{j-1} = ||u_j||,   beta_j = ||u_{j+1}||
// which is the reference's recurrence (lanczos.cu:32-50) with the division by beta moved to the consumers (as a multiplication
// by the reciprocal: results differ from the divide-first order in the last bit only).
// One entry of the lagged update, u' = (t - alpha u_j) / ||u_j|| - (||u_j|| / ||u_{j-1}||) u_{j-1}, with the operation order pinned by
// explicit fma so that every kernel that forms it (one GPU, dense push, entry-wise push) produces the same bits.
__device__ __forceinline__ double lagged_entry(double t, double q, double p, double a, double rj, double cp, bool has_p) {
  double v = fma(-a, q, t) * rj;
  if (has_p) v = fma(-cp, p, v);
  return v;
}
__global__ void __launch_bounds__(kBlock) k_update_lagged(const double* __restrict__ t, const double* __restrict__ uj, const double* __restrict__ up,
                                                          const double* __restrict__ alpha_p, const double* __restrict__ norm2_j,
                                                          const double* __restrict__ norm2_p, uint64_t n, double* __restrict__ u_next,
                                                          double* partials, unsigned int* ticket, double* norm2_out, double* beta_out,
                                                          float* __restrict__ u32_next /* fp32 basis row, or null */) {
  __shared__ double sm[kWarps];
  __shared__ bool s_last;
  // u_{j+1} = (t - alpha u_j) / ||u_j|| - (||u_j|| / ||u_{j-1}||) u_{j-1}: the two scalars are formed once per thread, so the
  // pass costs three multiply-adds per entry and stays HBM-bound (per-entry fp64 divisions made it compute-bound: measured).
  const double a = *alpha_p;
  const double nj = sqrt(*norm2_j);
  const double rj = 1.0 / nj;
  const double cp = up ? nj / sqrt(*norm2_p) : 0.0;   // beta_{j-1} / ||u_{j-1}||,  beta_{j-1} = ||u_j||
  const uint64_t n2 = n >> 1;
  double acc = 0.0;
  const double2* t2 = reinterpret_cast<const double2*>(t);
  const double2* q2 = reinterpret_cast<const double2*>(uj);
  const double2* p2 = reinterpret_cast<const double2*>(up);
  double2* o2 = reinterpret_cast<double2*>(u_next);
  for (uint64_t i = (uint64_t)blockIdx.x * kBlock + threadIdx.x; i < n2; i += (uint64_t)gridDim.x * kBlock) {
    const double2 tv = t2[i], qv = q2[i];
    const double2 pv = up ? p2[i] : make_double2(0.0, 0.0);
    double2 v;
    v.x = lagged_entry(tv.x, qv.x, pv.x, a, rj, cp, up != nullptr);
    v.y = lagged_entry(tv.y, qv.y, pv.y, a, rj, cp, up != nullptr);
    o2[i] = v;
    if (u32_next) reinterpret_cast<float2*>(u32_next)[i] = make_float2((float)v.x, (float)v.y);
    acc = fma(v.x, v.x, acc);
    acc = fma(v.y, v.y, acc);
  }
  if ((n & 1) && blockIdx.x == 0 && threadIdx.x == 0) {
    const double v = lagged_entry(t[n - 1], uj[n - 1], up ? up[n - 1] : 0.0, a, rj, cp, up != nullptr);
    u_next[n - 1] = v;
    if (u32_next) u32_next[n - 1] = (float)v;
    acc = fma(v, v, acc);
  }
  acc = block_sum(acc, sm);
  if (threadIdx.x == 0) {
    partials[blockIdx.x] = acc;
    __threadfence();
    s_last = (atomicAdd(ticket, 1u) == gridDim.x - 1);
  }
  __syncthreads();
  if (s_last) {
    __threadfence();
    double tot = 0.0;
    for (unsigned int i = threadIdx.x; i < gridDim.x; i += kBlock) tot += __ldcg(partials + i);
    tot = block_sum(tot, sm);
    if (threadIdx.x == 0) {
      *norm2_out = tot;
      *beta_out = sqrt(tot);
      *ticket = 0u;
    }
  }
}
// Lagged normalisation on several GPUs (plain recurrence, peer exchange): the same update as k_update_lagged, fused with the
// two cross-GPU reductions it depends on and with the producer side of the vector exchange, so one step is the SpMV passes plus
// THIS kernel — the separate normalisation kernel (k_scale_push) and its cross-GPU wait are gone:
//   * alpha_j = (sum over ranks of the SpMV kernels' partials of A u_j . u_j) / ||u_j||^2  — consumed from the peer scalar slots;
//   * ||u_j||^2 was published by the previous step's instance of this kernel (long arrived: not on the critical path);
//   * u_{j+1} is written to the local basis AND — unnormalised — straight into every rank's gathered vector (chunks
//     [0, push_chunks); the SpMV passes send the rest), or entry-wise to the peers that reference it (needed-columns exchange);
//   * the partial of ||u_{j+1}||^2 is published for the next step. Nobody waits for it inside this step.
// The peers' SpMV gathers from the unnormalised vector; every consumer of V folds 1/||u_j|| in (multOut, lz_get_basis).
struct lz_push_lists {
  const uint32_t* list;
  uint32_t off[LZ_MAX_WORLD + 1];
};
template <bool SPARSE>
__global__ void __launch_bounds__(kBlock) k_update_lagged_push(const double* __restrict__ t, const double* __restrict__ uj, const double* __restrict__ up,
                                                               uint64_t n, double* __restrict__ u_next, double* __restrict__ norm2v /* [j] is written here */,
                                                               uint32_t j, double* __restrict__ alpha_out, double* __restrict__ beta_out,
                                                               const __grid_constant__ lz_peers peers, uint64_t cl, uint32_t nchunks, uint32_t push_chunks,
                                                               uint32_t world, uint32_t rank, unsigned long long push_seq, unsigned int* push_ticket,
                                                               double* partials, unsigned int* ticket, const __grid_constant__ lz_red red,
                                                               const __grid_constant__ lz_push_lists lists, float* __restrict__ u32_next) {
  __shared__ double sm[kWarps];
  __shared__ bool s_last;
  __shared__ double s_bcast;
  // ||u_j||^2 first (published one step ago), then alpha (the reduction this step waits for)
  if (blockIdx.x == 0 && threadIdx.x == 0) trace_mark(LZ_TR(0x01, TR_START));
  const double n2j = j ? red_consume_seq(red, 1, red.seq - 1, &s_bcast) : 1.0;
  const double a = red_consume_seq(red, 0, red.seq, &s_bcast) / n2j;
  if (blockIdx.x == 0 && threadIdx.x == 0) trace_mark(LZ_TR(0x01, TR_WAITED));
  const double nj = sqrt(n2j);
  const double rj = 1.0 / nj;
  const double cp = up ? nj / sqrt(norm2v[j - 1]) : 0.0;      // norm2v[j-1]: written by the previous launch of this kernel
  if (blockIdx.x == 0 && threadIdx.x == 0) {
    alpha_out[j] = a;
    if (j) { norm2v[j] = n2j; beta_out[j - 1] = nj; }
  }
  const double2* t2 = reinterpret_cast<const double2*>(t);
  const double2* q2 = reinterpret_cast<const double2*>(uj);
  const double2* p2 = reinterpret_cast<const double2*>(up);
  double2* o2 = reinterpret_cast<double2*>(u_next);
  const uint64_t cl2 = cl >> 1;
  double acc = 0.0;
  double* own = peers.x[rank];
  for (uint32_t c = 0; c < nchunks; c++) {
    const bool send = !SPARSE && c < push_chunks;
    const uint64_t slot2 = ((uint64_t)c * world * cl + (uint64_t)rank * cl) >> 1;
    for (uint64_t i = (uint64_t)blockIdx.x * kBlock + threadIdx.x; i < cl2; i += (uint64_t)gridDim.x * kBlock) {
      const uint64_t li = (uint64_t)c * cl2 + i;
      const double2 tv = t2[li], qv = q2[li];
      const double2 pv = up ? p2[li] : make_double2(0.0, 0.0);
      double2 v;
      v.x = lagged_entry(tv.x, qv.x, pv.x, a, rj, cp, up != nullptr);
      v.y = lagged_entry(tv.y, qv.y, pv.y, a, rj, cp, up != nullptr);
      o2[li] = v;
      if (u32_next) reinterpret_cast<float2*>(u32_next)[li] = make_float2((float)v.x, (float)v.y);   // fp32 basis row
      acc = fma(v.x, v.x, acc);
      acc = fma(v.y, v.y, acc);
      if (SPARSE) reinterpret_cast<double2*>(own)[slot2 + i] = v;
      else if (send)
        for (uint32_t r = 0; r < world; r++) reinterpret_cast<double2*>(peers.x[r])[slot2 + i] = v;
    }
    if (!send) continue;
    __threadfence_system();          // this thread's peer stores are visible system-wide before the CTA reports in
    __syncthreads();
    if (threadIdx.x == 0) {
      const unsigned int tk = atomicAdd(push_ticket + c, 1u);
      s_last = (tk == gridDim.x - 1);
      if (s_last) {
        push_ticket[c] = 0u;
        __threadfence_system();
        for (uint32_t r = 0; r < world; r++) st_relaxed_sys(peers.f[r] + (uint64_t)c * LZ_MAX_WORLD + rank, push_seq);
        trace_mark(LZ_TR(0x01, TR_PUSHED));
      }
    }
    __syncthreads();
  }
  if (SPARSE) {
    // every peer receives only the entries its rows reference; the values are recomputed from the inputs (same operations =>
    // same bits as the local copy), because the entry may have been produced by another CTA of this launch
    for (uint32_t r = 0; r < world; r++) {
      if (r == rank) continue;
      double* dst = peers.x[r];
      const uint32_t e = lists.off[r + 1];
      for (uint64_t s = (uint64_t)lists.off[r] + (uint64_t)blockIdx.x * kBlock + threadIdx.x; s < e; s += (uint64_t)gridDim.x * kBlock) {
        const uint32_t l = __ldg(lists.list + s);
        const double v = lagged_entry(t[l], uj[l], up ? up[l] : 0.0, a, rj, cp, up != nullptr);
        const uint64_t c = l / cl;
        dst[c * (world * cl) + (uint64_t)rank * cl + (l - c * cl)] = v;
      }
    }
    __threadfence_system();
    __syncthreads();
    if (threadIdx.x == 0) {
      const unsigned int tk = atomicAdd(push_ticket, 1u);
      s_last = (tk == gridDim.x - 1);
      if (s_last) {
        *push_ticket = 0u;
        __threadfence_system();
        for (uint32_t c = 0; c < nchunks; c++)
          for (uint32_t r = 0; r < world; r++) st_relaxed_sys(peers.f[r] + (uint64_t)c * LZ_MAX_WORLD + rank, push_seq);
      }
    }
    __syncthreads();
  }
  acc = block_sum(acc, sm);
  grid_sum_finish(acc, partials, ticket, nullptr, sm, &s_last, 0xFFFFFFFFu, 0, &red, 1);   // publishes the partial of ||u_{j+1}||^2
  if (s_last && threadIdx.x == 0) trace_mark(LZ_TR(0x01, TR_END));
}
// Closes a lagged multi-GPU run: the last step has no update kernel, so its alpha and the last ||u||^2 are finished here.
__global__ void k_lagged_finish(uint32_t j, double* __restrict__ norm2v, double* __restrict__ alpha_out, double* __restrict__ beta_out,
                                const __grid_constant__ lz_red red) {
  __shared__ double s_bcast;
  const double n2j = j ? red_consume_seq(red, 1, red.seq - 1, &s_bcast) : 1.0;
  const double a = red_consume_seq(red, 0, red.seq, &s_bcast) / n2j;
  if (threadIdx.x == 0) {
    alpha_out[j] = a;
    if (j) { norm2v[j] = n2j; beta_out[j - 1] = sqrt(n2j); }
  }
}

// out[j] = coef[j] / sqrt(norm2[j]): multOut coefficients for an unnormalised basis
__global__ void k_coef_scale(const double* __restrict__ coef, const double* __restrict__ norm2, uint32_t k, double* __restrict__ out) {
  const uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j < k) out[j] = coef[j] / sqrt(norm2[j]);
}
__global__ void k_div_sqrt(double* __restrict__ v, uint64_t n, const double* __restrict__ norm2) {
  const double d = sqrt(*norm2);
  for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) v[i] /= d;
}

// Index of local row l in the chunk-major gathered vector (see k_relabel in lz_graph.cu).
__device__ __forceinline__ uint64_t xfull_index(uint64_t l, uint64_t cl, uint32_t world, uint32_t rank) {
  const uint64_t c = l / cl;
  return c * (world * cl) + rank * cl + (l - c * cl);
}

// q_next = w / sqrt(norm2)  (true division, as cu_dvexda); optional second copy into this rank's slots of the gathered
// vector; beta_out = sqrt(norm2). n and cl are even, so a double2 never straddles a chunk.
__global__ void __launch_bounds__(kBlock) k_scale(const double* __restrict__ w, const double* __restrict__ norm2_p, uint64_t n,
                                                  double* __restrict__ q_next, double* __restrict__ xfull, uint64_t cl, uint32_t world,
                                                  uint32_t rank, double* beta_out, float* __restrict__ q32_next) {
  const double beta = sqrt(*norm2_p);
  if (blockIdx.x == 0 && threadIdx.x == 0 && beta_out) *beta_out = beta;
  const uint64_t n2 = n >> 1;
  const double2* w2 = reinterpret_cast<const double2*>(w);
  double2* q2 = reinterpret_cast<double2*>(q_next);
  for (uint64_t i = (uint64_t)blockIdx.x * kBlock + threadIdx.x; i < n2; i += (uint64_t)gridDim.x * kBlock) {
    double2 v = w2[i];
    v.x /= beta;
    v.y /= beta;
    q2[i] = v;
    if (q32_next) reinterpret_cast<float2*>(q32_next)[i] = make_float2((float)v.x, (float)v.y);
    if (xfull) *reinterpret_cast<double2*>(xfull + xfull_index(2 * i, cl, world, rank)) = v;
  }
  if ((n & 1) && blockIdx.x == 0 && threadIdx.x == 0) {      // odd tail (n_loc is a multiple of 32 in practice)
    const double v = w[n - 1] / beta;
    q_next[n - 1] = v;
    if (q32_next) q32_next[n - 1] = (float)v;
  }
}
// dst32[i] = (float)src[i]
__global__ void __launch_bounds__(kBlock) k_to_f32(const double* __restrict__ src, float* __restrict__ dst, uint64_t n) {
  for (uint64_t i = (uint64_t)blockIdx.x * kBlock + threadIdx.x; i < n; i += (uint64_t)gridDim.x * kBlock) dst[i] = (float)src[i];
}
__global__ void __launch_bounds__(kBlock) k_to_f64(const float* __restrict__ src, double* __restrict__ dst, uint64_t n) {
  for (uint64_t i = (uint64_t)blockIdx.x * kBlock + threadIdx.x; i < n; i += (uint64_t)gridDim.x * kBlock) dst[i] = (double)src[i];
}

// Producer side of the peer exchange, fused into the normalisation: q_next = w / beta is stored locally and, 16 bytes at a
// time, into the chunk-major gathered vector of EVERY rank (peer stores over NVLink; own rank included). Rows are
// processed chunk by chunk; when the last CTA has finished a chunk it publishes `seq` in every rank's arrival counter for
// (chunk, this rank), so remote SpMV passes over early (hot) chunks start while later chunks are still being sent.
__global__ void __launch_bounds__(kBlock) k_scale_push(const double* __restrict__ w, const double* __restrict__ norm2_p, uint64_t n,
                                                       double* __restrict__ q_next, const __grid_constant__ lz_peers peers, uint64_t cl,
                                                       uint32_t nchunks, uint32_t push_chunks, uint32_t world, uint32_t rank,
                                                       unsigned long long seq, unsigned int* ticket, double* beta_out,
                                                       const __grid_constant__ lz_red red) {
  __shared__ double s_bcast;
  const double beta = norm2_p ? sqrt(red.seq ? red_consume(red, 1, &s_bcast) : *norm2_p) : 1.0;
  if (blockIdx.x == 0 && threadIdx.x == 0 && beta_out) *beta_out = beta;
  const double2* w2 = reinterpret_cast<const double2*>(w);
  double2* q2 = reinterpret_cast<double2*>(q_next);
  const uint64_t cl2 = cl >> 1;
  __shared__ bool s_last;
  for (uint32_t c = 0; c < nchunks; c++) {
    const bool send = c < push_chunks;
    const uint64_t slot2 = ((uint64_t)c * world * cl + (uint64_t)rank * cl) >> 1;
    for (uint64_t i = (uint64_t)blockIdx.x * kBlock + threadIdx.x; i < cl2; i += (uint64_t)gridDim.x * kBlock) {
      const uint64_t li = (uint64_t)c * cl2 + i;
      double2 v = w2[li];
      if (norm2_p) { v.x /= beta; v.y /= beta; }
      if (q_next != w) q2[li] = v;
      if (send)
        for (uint32_t r = 0; r < world; r++) reinterpret_cast<double2*>(peers.x[r])[slot2 + i] = v;
    }
    if (!send) continue;
    __threadfence_system();          // this thread's peer stores are visible system-wide before the CTA reports in
    __syncthreads();
    if (threadIdx.x == 0) {
      const unsigned int t = atomicAdd(ticket + c, 1u);
      s_last = (t == gridDim.x - 1);
      if (s_last) {
        ticket[c] = 0u;
        __threadfence_system();
        for (uint32_t r = 0; r < world; r++) st_relaxed_sys(peers.f[r] + (uint64_t)c * LZ_MAX_WORLD + rank, seq);
      }
    }
    __syncthreads();
  }
}


// Producer side of the needed-columns exchange (lz_build_push_lists): q_next = w / beta is stored locally and into this
// rank's own slots of the gathered vector in full; every peer receives only the entries its rows reference (8-byte peer
// stores over NVLink, ascending addresses). One arrival counter per chunk is raised at the end, as in k_scale_push, so the
// consuming SpMV passes are unchanged. Remote values are recomputed from w (same division => same bits as the local copy).
__global__ void __launch_bounds__(kBlock) k_scale_push_sparse(const double* __restrict__ w, const double* __restrict__ norm2_p, uint64_t n,
                                                              double* __restrict__ q_next, const __grid_constant__ lz_peers peers, uint64_t cl,
                                                              uint32_t nchunks, uint32_t world, uint32_t rank, unsigned long long seq,
                                                              unsigned int* ticket, double* beta_out, const __grid_constant__ lz_red red,
                                                              const __grid_constant__ lz_push_lists lists) {
  __shared__ double s_bcast;
  __shared__ bool s_last;
  const double beta = norm2_p ? sqrt(red.seq ? red_consume(red, 1, &s_bcast) : *norm2_p) : 1.0;
  if (blockIdx.x == 0 && threadIdx.x == 0 && beta_out) *beta_out = beta;
  const double2* w2 = reinterpret_cast<const double2*>(w);
  double2* q2 = reinterpret_cast<double2*>(q_next);
  double* own = peers.x[rank];
  const uint64_t n2 = n >> 1;
  for (uint64_t i = (uint64_t)blockIdx.x * kBlock + threadIdx.x; i < n2; i += (uint64_t)gridDim.x * kBlock) {
    double2 v = w2[i];
    if (norm2_p) { v.x /= beta; v.y /= beta; }
    if (q_next != w) q2[i] = v;
    *reinterpret_cast<double2*>(own + xfull_index(2 * i, cl, world, rank)) = v;
  }
  for (uint32_t r = 0; r < world; r++) {
    if (r == rank) continue;
    double* dst = peers.x[r];
    const uint32_t e = lists.off[r + 1];
    for (uint64_t t = (uint64_t)lists.off[r] + (uint64_t)blockIdx.x * kBlock + threadIdx.x; t < e; t += (uint64_t)gridDim.x * kBlock) {
      const uint32_t l = __ldg(lists.list + t);
      double v = w[l];
      if (norm2_p) v /= beta;
      dst[xfull_index(l, cl, world, rank)] = v;
    }
  }
  __threadfence_system();          // this thread's peer stores are visible system-wide before the CTA reports in
  __syncthreads();
  if (threadIdx.x == 0) {
    const unsigned int t = atomicAdd(ticket, 1u);
    s_last = (t == gridDim.x - 1);
    if (s_last) {
      *ticket = 0u;
      __threadfence_system();
      for (uint32_t c = 0; c < nchunks; c++)
        for (uint32_t r = 0; r < world; r++) st_relaxed_sys(peers.f[r] + (uint64_t)c * LZ_MAX_WORLD + rank, seq);
    }
  }
}

// q0_local[l] = 2^-xexp x_orig[new2old[slot(l)]] / sqrt(norm2)
__global__ void k_permute_in_local(const double* __restrict__ x_orig, const uint32_t* __restrict__ new2old, uint64_t n, uint64_t cl,
                                   uint32_t world, uint32_t rank, const double* __restrict__ norm2_p, int xexp, double* __restrict__ dst) {
  const double nrm = sqrt(*norm2_p);
  for (uint64_t l = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; l < n; l += (uint64_t)gridDim.x * blockDim.x) {
    const uint32_t o = new2old[xfull_index(l, cl, world, rank)];
    dst[l] = (o == 0xFFFFFFFFu) ? 0.0 : ldexp(x_orig[o], -xexp) / nrm;
  }
}

// dir 0: xfull[slot(l)] = local[l]   dir 1: local[l] = xfull[slot(l)]
__global__ void __launch_bounds__(kBlock) k_spread_collect(double* __restrict__ local, double* __restrict__ xfull, uint64_t n, uint64_t cl,
                                                           uint32_t world, uint32_t rank, int dir) {
  const uint64_t n2 = n >> 1;
  for (uint64_t i = (uint64_t)blockIdx.x * kBlock + threadIdx.x; i < n2; i += (uint64_t)gridDim.x * kBlock) {
    double2* a = reinterpret_cast<double2*>(local) + i;
    double2* b = reinterpret_cast<double2*>(xfull + xfull_index(2 * i, cl, world, rank));
    if (dir == 0) *b = *a; else *a = *b;
  }
}

// ||2^-e v||^2. Scaling by a power of two is exact, so for an e that keeps the squares normal the result is 2^-2e ||v||^2 to the bit.
__global__ void __launch_bounds__(kBlock) k_norm2(const double* __restrict__ v, uint64_t n, int e, double* partials, unsigned int* ticket,
                                                  double* out) {
  __shared__ double sm[kWarps];
  __shared__ bool s_last;
  double acc = 0.0;
  for (uint64_t i = (uint64_t)blockIdx.x * kBlock + threadIdx.x; i < n; i += (uint64_t)gridDim.x * kBlock) {
    const double a = ldexp(v[i], -e);
    acc += a * a;
  }
  acc = block_sum(acc, sm);
  grid_sum_finish(acc, partials, ticket, out, sm, &s_last);
}

// max_i |v[i]| as the bit pattern of a non-negative double, ordered like the values with NaN above inf: *out must be zeroed first
__global__ void __launch_bounds__(kBlock) k_absmax_bits(const double* __restrict__ v, uint64_t n, unsigned long long* out) {
  __shared__ unsigned long long sm[kWarps];
  unsigned long long mx = 0ull;
  for (uint64_t i = (uint64_t)blockIdx.x * kBlock + threadIdx.x; i < n; i += (uint64_t)gridDim.x * kBlock)
    mx = max(mx, (unsigned long long)__double_as_longlong(v[i]) & 0x7FFFFFFFFFFFFFFFull);
  for (int o = 16; o > 0; o >>= 1) mx = max(mx, __shfl_xor_sync(0xffffffffu, mx, o));
  if ((threadIdx.x & 31) == 0) sm[threadIdx.x >> 5] = mx;
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int w = 1; w < kWarps; w++) mx = max(mx, sm[w]);
    atomicMax(out, mx);
  }
}

// dst[i] = 2^-xexp x_orig[new2old[first + i]] / sqrt(norm2) for i < count (0 for padding slots)
__global__ void k_permute_in(const double* __restrict__ x_orig, const uint32_t* __restrict__ new2old, uint64_t first, uint64_t count,
                             const double* __restrict__ norm2_p, int xexp, double* __restrict__ dst) {
  const double nrm = sqrt(*norm2_p);
  for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < count; i += (uint64_t)gridDim.x * blockDim.x) {
    const uint32_t o = new2old[first + i];
    dst[i] = (o == 0xFFFFFFFFu) ? 0.0 : ldexp(x_orig[o], -xexp) / nrm;
  }
}
// same without scaling
__global__ void k_permute_in_raw(const double* __restrict__ x_orig, const uint32_t* __restrict__ new2old, uint64_t first, uint64_t count,
                                 double* __restrict__ dst) {
  for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < count; i += (uint64_t)gridDim.x * blockDim.x) {
    const uint32_t o = new2old[first + i];
    dst[i] = (o == 0xFFFFFFFFu) ? 0.0 : x_orig[o];
  }
}
__global__ void k_fill(double* __restrict__ p, uint64_t n, double v) {
  for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) p[i] = v;
}
// y_orig[new2old[i]] = y_new[i]
__global__ void k_permute_out(const double* __restrict__ y_new, const uint32_t* __restrict__ new2old, uint64_t count,
                              double* __restrict__ y_orig) {
  for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < count; i += (uint64_t)gridDim.x * blockDim.x) {
    const uint32_t o = new2old[i];
    if (o != 0xFFFFFFFFu) y_orig[o] = y_new[i];
  }
}

// ------------------------------------------------------------------------------------- tall-skinny GEMV-T (reorth dots)
// h[t] = sum_i V[t][i] w[i], t < nvec. Vectors are processed in register tiles of TILE so w is re-read nvec/TILE times
// (+1/TILE traffic) while TILE independent 16-byte loads per thread are in flight.
constexpr int kDotTile = 8;
template <class TV>
__global__ void __launch_bounds__(kBlock) k_multidot(const TV* __restrict__ V, uint64_t ldv, uint32_t nvec, const double* __restrict__ w,
                                                     uint64_t n, double* partials /* [nvec][grid] */, unsigned int* ticket, double* h_out,
                                                     const int* __restrict__ skip, const double* __restrict__ h_div /* h[t] /= h_div[t], or null */) {
  constexpr int E = ept<TV>::value;
  __shared__ double sm[kWarps];
  __shared__ bool s_last;
  if (skip && *skip) return;   // second Gram-Schmidt pass not needed (decided on the device, see k_reorth_decide)
  const uint64_t ng = n / E, ldg = ldv / E;         // whole 16-byte groups; the tail (n % E entries) is handled by thread 0 below
  // w is re-read once per tile of T vectors (fp64 basis: +1/8 of the traffic, fp32 basis: +1/4). A 16-vector tile for the fp32
  // basis was measured slower (80 registers: C3 full reorth 487 vs 499 it/s), so both use 8.
  constexpr int T = kDotTile;
  for (uint32_t t0 = 0; t0 < nvec; t0 += T) {
    double acc[T];
#pragma unroll
    for (int u = 0; u < T; u++) acc[u] = 0.0;
    const uint32_t nt = min((uint32_t)T, nvec - t0);
    const TV* vb = V + (uint64_t)t0 * ldv;
    for (uint64_t i = (uint64_t)blockIdx.x * kBlock + threadIdx.x; i < ng; i += (uint64_t)gridDim.x * kBlock) {
      double wv[E];
      ld_group<double>(w, i * (E / 2), *reinterpret_cast<double(*)[2]>(&wv[0]));
      if constexpr (E == 4) ld_group<double>(w, i * 2 + 1, *reinterpret_cast<double(*)[2]>(&wv[2]));
#pragma unroll
      for (int sub = 0; sub < T / kDotTile; sub++) {
        if ((uint32_t)(sub * kDotTile) >= nt) break;
        double vv[kDotTile][E];
        if (nt >= (uint32_t)((sub + 1) * kDotTile)) {
#pragma unroll
          for (int u = 0; u < kDotTile; u++) ld_group<TV>(vb, (uint64_t)(sub * kDotTile + u) * ldg + i, vv[u]);
#pragma unroll
          for (int u = 0; u < kDotTile; u++)
#pragma unroll
            for (int e = 0; e < E; e++) acc[sub * kDotTile + u] += vv[u][e] * wv[e];
        } else {
#pragma unroll
          for (int u = 0; u < kDotTile; u++)
            if ((uint32_t)(sub * kDotTile + u) < nt) {
              ld_group<TV>(vb, (uint64_t)(sub * kDotTile + u) * ldg + i, vv[u]);
#pragma unroll
              for (int e = 0; e < E; e++) acc[sub * kDotTile + u] += vv[u][e] * wv[e];
            }
        }
      }
    }
    if (blockIdx.x == 0 && threadIdx.x == 0)
      for (uint64_t r = ng * E; r < n; r++)
#pragma unroll
        for (int u = 0; u < T; u++)
          if (u < (int)nt) acc[u] += (double)V[(uint64_t)(t0 + u) * ldv + r] * w[r];
#pragma unroll
    for (int u = 0; u < T; u++) {
      if (u < (int)nt) {
        double s = block_sum(acc[u], sm);
        if (threadIdx.x == 0) partials[(uint64_t)(t0 + u) * gridDim.x + blockIdx.x] = s;
      }
    }
  }
  // last CTA: one warp per vector, lanes stride the CTA partials in index order
  if (threadIdx.x == 0) {
    __threadfence();
    unsigned int t = atomicAdd(ticket, 1u);
    s_last = (t == gridDim.x - 1);
  }
  __syncthreads();
  if (s_last) {
    __threadfence();
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    for (uint32_t t = wid; t < nvec; t += kWarps) {
      double acc = 0.0;
      for (unsigned int i = lane; i < gridDim.x; i += 32) acc += __ldcg(partials + (uint64_t)t * gridDim.x + i);
      acc = warp_sum(acc);
      if (lane == 0) h_out[t] = h_div ? acc / h_div[t] : acc;   // unnormalised basis rows: (u_t . w) / ||u_t||^2
    }
    if (threadIdx.x == 0) *ticket = 0u;
  }
}

// ---------------------------------------------------------------------------- tall-skinny GEMV-N (reorth update, multOut)
// out[i] = (base ? base[i] : 0) + sign * sum_t coef[t] V[t][i], accumulated in t order (the order of the reference's
// row-major Trans dgemv, multiplyOut.cu:44). Optional partial of ||out||^2.
template <class TV>
__global__ void __launch_bounds__(kBlock) k_combine(const TV* __restrict__ V, uint64_t ldv, uint32_t nvec, const double* __restrict__ coef,
                                                    double sign, const double* base, double* out, uint64_t n, double* partials,
                                                    unsigned int* ticket, double* norm2_out, const int* __restrict__ skip,
                                                    float* __restrict__ out32 /* fp32 copy of out, or null */) {
  constexpr int E = ept<TV>::value;
  extern __shared__ double s_coef[];
  __shared__ double sm[kWarps];
  __shared__ bool s_last;
  if (skip && *skip) return;
  for (uint32_t t = threadIdx.x; t < nvec; t += kBlock) s_coef[t] = sign * coef[t];
  __syncthreads();
  const uint64_t ng = n / E, ldg = ldv / E;
  const double2* b2 = reinterpret_cast<const double2*>(base);
  double2* o2 = reinterpret_cast<double2*>(out);
  double nacc = 0.0;
  for (uint64_t i = (uint64_t)blockIdx.x * kBlock + threadIdx.x; i < ng; i += (uint64_t)gridDim.x * kBlock) {
    double acc[E];
#pragma unroll
    for (int h = 0; h < E / 2; h++) {
      const double2 bv = base ? b2[i * (E / 2) + h] : make_double2(0.0, 0.0);
      acc[2 * h] = bv.x; acc[2 * h + 1] = bv.y;
    }
    uint32_t t = 0;
    for (; t + 8 <= nvec; t += 8) {
      double vv[8][E];
#pragma unroll
      for (int u = 0; u < 8; u++) ld_group<TV>(V, (uint64_t)(t + u) * ldg + i, vv[u]);
#pragma unroll
      for (int u = 0; u < 8; u++)
#pragma unroll
        for (int e = 0; e < E; e++) acc[e] += s_coef[t + u] * vv[u][e];
    }
    for (; t < nvec; t++) {
      double vv[E];
      ld_group<TV>(V, (uint64_t)t * ldg + i, vv);
#pragma unroll
      for (int e = 0; e < E; e++) acc[e] += s_coef[t] * vv[e];
    }
#pragma unroll
    for (int h = 0; h < E / 2; h++) o2[i * (E / 2) + h] = make_double2(acc[2 * h], acc[2 * h + 1]);
    if (out32) {
#pragma unroll
      for (int h = 0; h < E / 2; h++) reinterpret_cast<float2*>(out32)[i * (E / 2) + h] = make_float2((float)acc[2 * h], (float)acc[2 * h + 1]);
    }
#pragma unroll
    for (int e = 0; e < E; e++) nacc += acc[e] * acc[e];
  }
  if (blockIdx.x == 0 && threadIdx.x == 0)
    for (uint64_t r = ng * E; r < n; r++) {
      double acc = base ? base[r] : 0.0;
      for (uint32_t t = 0; t < nvec; t++) acc += s_coef[t] * (double)V[(uint64_t)t * ldv + r];
      out[r] = acc;
      if (out32) out32[r] = (float)acc;
      nacc += acc * acc;
    }
  if (norm2_out) {
    nacc = block_sum(nacc, sm);
    grid_sum_finish(nacc, partials, ticket, norm2_out, sm, &s_last);
  }
}

// ------------------------------------------------------------------------------------ tridiagonal eigenproblem + coefficients
// One CTA. Thread 0 runs the scalar implicit-shift QL recurrences and publishes each sweep's rotations; all threads apply
// them to the eigenvector matrix, kept transposed (zt[i*k + q] = component q of vector i) so the update is coalesced.
// Output in the layout LAPACKE_dstevd(LAPACK_ROW_MAJOR,'V') gives the reference (eigen.cu:20): eigenvalues ascending,
// eigvecs[q*k + j] = component q of eigenvector j. Then f_j = f(lambda_j) * x_norm * eigvecs[0*k + j] (multiplyOut.cu:30-33)
// and coef = eigvecs * f (multiplyOut.cu:40), with f selected by fkind (LZ_MATFUN_*):
//   EXP        exp(p*lambda - 0)   (p = 1: exactly the reference's exp(lambda))
//   EXP_SCALED exp(p*lambda - ls), ls = max_j p*lambda_j, or *ls_in when given (leading blocks reuse the full solve's shift);
//              every argument is <= 0, so nothing overflows for any graph
//   RESOLVENT  1 / (1 - p*lambda); a non-positive denominator sets kStatusIndefinite
// ls goes to *ls_out (when given) so that e^{pA} x = ans * e^ls.
constexpr int kEigMax = 1024;
__global__ void __launch_bounds__(kBlock) k_tridiag_expv(uint32_t k, const double* __restrict__ alpha, const double* __restrict__ beta,
                                                         const double* __restrict__ xnorm2_p, int xexp, double* __restrict__ eigvals,
                                                         double* __restrict__ eigvecs, double* __restrict__ zt_global, double* __restrict__ coef,
                                                         int* __restrict__ status, int zt_in_smem, int fkind, double fparam,
                                                         const double* __restrict__ ls_in, double* __restrict__ ls_out) {
  extern __shared__ double zt_smem[];
  double* zt = zt_in_smem ? zt_smem : zt_global;   // k*k doubles: shared memory when it fits (k <= ~150), else global scratch
  __shared__ double d[kEigMax], e[kEigMax], cs[kEigMax], sn[kEigMax];
  __shared__ int perm[kEigMax];
  __shared__ int s_m, s_sweep, s_cont, s_fail;
  __shared__ double s_ls;
  const int n = (int)k, tid = threadIdx.x;
  for (int i = tid; i < n; i += kBlock) {
    d[i] = alpha[i];
    e[i] = (i + 1 < n) ? beta[i] : 0.0;
  }
  for (int i = tid; i < n * n; i += kBlock) zt[i] = ((i / n) == (i % n)) ? 1.0 : 0.0;
  if (tid == 0) s_fail = 0;
  __syncthreads();
  const double eps = 2.220446049250313e-16;
  double f = 0.0, tst1 = 0.0;   // live in thread 0 only
  for (int l = 0; l < n; l++) {
    int iter = 0;
    if (tid == 0) {
      tst1 = fmax(tst1, fabs(d[l]) + fabs(e[l]));
      int m = l;
      while (m < n - 1 && fabs(e[m]) > eps * tst1) m++;   // e[n-1] == 0; written so a NaN input cannot run past the end
      s_m = m;
    }
    __syncthreads();
    const int m = s_m;
    if (m > l) {
      for (;;) {
        if (tid == 0) {
          s_sweep = 1;
          if (++iter > 60) { s_fail = l + 1; s_sweep = 0; s_cont = 0; }
          else {
            double g = d[l];
            double p = (d[l + 1] - g) / (2.0 * e[l]);
            double r = sqrt(fma(p, p, 1.0));
            if (p < 0) r = -r;
            d[l] = e[l] / (p + r);
            d[l + 1] = e[l] * (p + r);
            const double dl1 = d[l + 1];
            double h = g - d[l];
            for (int i = l + 2; i < n; i++) d[i] -= h;
            f += h;
            p = d[m];
            double c = 1.0, c2 = c, c3 = c, s = 0.0, s2 = 0.0;
            const double el1 = e[l + 1];
            double ei = e[m - 1], di = d[m - 1];       // operands of the next rotation are fetched one rotation ahead so
            for (int i = m - 1; i >= l; i--) {          // the shared-memory latency stays off the serial dependency chain
              const double ei_next = (i > l) ? e[i - 1] : 0.0, di_next = (i > l) ? d[i - 1] : 0.0;
              c3 = c2; c2 = c; s2 = s;
              g = c * ei;
              h = c * p;
              // |p|, |e_i| are bounded by ||T|| (graph spectra: << 1e150), so the unscaled form cannot overflow
              const double rr = fma(p, p, ei * ei);
              const double rinv = (rr > 0.0) ? rsqrt(rr) : 0.0;
              r = rr * rinv;
              e[i + 1] = s * r;
              s = ei * rinv;
              c = (rr > 0.0) ? p * rinv : 1.0;
              p = c * di - s * g;
              d[i + 1] = h + s * (c * g + s * di);
              cs[i] = c; sn[i] = s;
              ei = ei_next; di = di_next;
            }
            p = -s * s2 * c3 * el1 * e[l] / dl1;
            e[l] = s * p;
            d[l] = c * p;
            s_cont = fabs(e[l]) > eps * tst1;
          }
        }
        __syncthreads();
        if (s_sweep) {
          for (int q = tid; q < n; q += kBlock) {
            double h = zt[m * n + q];                 // carried in a register from one rotation to the next
            for (int i = m - 1; i >= l; i--) {
              const double c = cs[i], s = sn[i];
              const double z = zt[i * n + q];
              zt[(i + 1) * n + q] = s * z + c * h;
              h = c * z - s * h;
            }
            zt[l * n + q] = h;
          }
        }
        const int cont = s_cont;
        __syncthreads();
        if (!cont) break;
      }
    }
    if (tid == 0) { d[l] += f; e[l] = 0.0; }
    __syncthreads();
    if (s_fail) break;
  }
  // ascending order (rank by counting; ties by index)
  // NaNs (Lanczos breakdown upstream) are ordered last so perm stays a permutation and nothing indexes out of range
  for (int i = tid; i < n; i += kBlock) {
    int r = 0;
    const double di = d[i];
    const bool ni = isnan(di);
    for (int j = 0; j < n; j++) {
      const double dj = d[j];
      const bool nj = isnan(dj);
      const bool less = ni ? (!nj) : (!nj && dj < di);
      const bool same = ni ? nj : (!nj && dj == di);
      r += less || (same && j < i);
    }
    perm[r] = i;
  }
  __syncthreads();
  for (int j = tid; j < n; j += kBlock) eigvals[j] = d[perm[j]];
  for (int i = tid; i < n * n; i += kBlock) {
    const int q = i / n, j = i % n;
    eigvecs[i] = zt[perm[j] * n + q];
  }
  if (tid == 0) {
    double ls = 0.0;
    if (fkind == LZ_MATFUN_EXP_SCALED) {
      if (ls_in) ls = *ls_in;
      else {
        ls = -INFINITY;
        for (int j = 0; j < n; j++) ls = fmax(ls, fparam * d[j]);   // NaNs (breakdown) are skipped here and poison f below
      }
    }
    s_ls = ls;
    if (ls_out) *ls_out = ls;
  }
  __syncthreads();
  const double xn = ldexp(sqrt(*xnorm2_p), xexp), ls = s_ls;   // ||x|| = 2^xexp ||2^-xexp x||
  bool indefinite = false;
  for (int j = tid; j < n; j += kBlock) {   // f_j ; row 0 of eigvecs
    const double lam = d[perm[j]];
    double fj;
    if (fkind == LZ_MATFUN_RESOLVENT) {
      const double den = 1.0 - fparam * lam;
      indefinite |= den <= 0.0;
      fj = 1.0 / den;
    } else {
      fj = exp(fparam * lam - ls);
    }
    cs[j] = fj * xn * eigvecs[j];
  }
  __syncthreads();
  bool bad = false;
  for (int i = tid; i < n; i += kBlock) {
    double s = 0.0;
    for (int j = 0; j < n; j++) s += eigvecs[(size_t)i * n + j] * cs[j];
    coef[i] = s;
    bad |= !isfinite(s);
  }
  if (tid == 0) *status = s_fail;
  __syncthreads();
  if (bad) atomicOr(status, 0x40000000);
  if (indefinite) atomicOr(status, kStatusIndefinite);
}

// "Twice is enough" (Daniel-Gragg-Kaufman-Stewart): after one classical Gram-Schmidt pass the second is needed only if the
// projection removed a substantial part of the vector, ||w_after||^2 < 1/2 ||w_before||^2. Decided on the device so the
// host never waits; the second pass's kernels exit at once when *skip != 0.
__global__ void k_reorth_decide(const double* __restrict__ norm2_before, const double* __restrict__ norm2_after, int* __restrict__ skip,
                                unsigned int* __restrict__ second_passes, int always) {
  const bool need = always || !(*norm2_after >= 0.5 * *norm2_before);   // also true for NaN
  *skip = need ? 0 : 1;
  if (need) atomicAdd(second_passes, 1u);
}
// norm2 = (second pass ran) ? norm2_second : unchanged
__global__ void k_reorth_select(const int* __restrict__ skip, const double* __restrict__ norm2_second, double* __restrict__ norm2,
                                double* __restrict__ norm2_copy, double* __restrict__ beta_out) {
  if (!*skip) *norm2 = *norm2_second;
  if (norm2_copy) *norm2_copy = *norm2;       // lagged normalisation: ||u_{j+1}||^2 and beta_j = ||u_{j+1}||
  if (beta_out) *beta_out = sqrt(*norm2);
}

// ------------------------------------------------------------------------------------------------- top Ritz pairs (lz_ritz)
// One CTA. From the ascending solve of T: theta[j] = eigvals[k-1-j] and W[t*M + j] = s_t * eigvecs[t*k + k-1-j] for j < m, 0 for
// m <= j < M, with s_t = 1/||u_t|| when the basis rows are unnormalised (norm2 != null: the fold k_coef_scale does), else 1.
__global__ void k_ritz_select(uint32_t k, uint32_t m, uint32_t M, const double* __restrict__ eigvals, const double* __restrict__ eigvecs,
                              const double* __restrict__ norm2, double* __restrict__ W, double* __restrict__ theta) {
  for (uint32_t i = threadIdx.x; i < k * M; i += blockDim.x) {
    const uint32_t t = i / M, j = i % M;
    double w = 0.0;
    if (j < m) {
      w = eigvecs[(uint64_t)t * k + (k - 1 - j)];
      if (norm2) w /= sqrt(norm2[t]);
    }
    W[i] = w;
  }
  for (uint32_t j = threadIdx.x; j < m; j += blockDim.x) theta[j] = eigvals[k - 1 - j];
}

// Y[j][i] = sum_t W[t][j] V[t][i] for j < M: every basis row is read once for all M Ritz vectors. Same 16-byte groups and the same
// t-ordered fma chain per output as k_combine (so column j equals k_combine(coef = W[:, j]) bit for bit). Shared memory holds W
// (k*M doubles, at most kEigMax * 16 * 8 = 128 KB) and each thread's running ||y_j||^2 and sum_i y_j(i) in a private column
// (2*M*kBlock doubles; in registers they would cost 4*M of them and spill the fp32 M = 16 instance). Per-vector partials in a fixed
// slot per CTA, summed in index order by the last CTA -> nrm2[j], vsum[j].
template <class TV, int M>
__global__ void __launch_bounds__(kBlock) k_ritz_combine(const TV* __restrict__ V, uint64_t ldv, uint32_t k, const double* __restrict__ W,
                                                         double* __restrict__ Y, uint64_t n, double* partials /* [2M][grid] */,
                                                         unsigned int* ticket, double* nrm2, double* vsum) {
  constexpr int E = ept<TV>::value;
  constexpr int U = M <= 4 ? 8 : (M == 8 ? 4 : 2);   // basis loads in flight per thread, traded against M*E accumulators
  extern __shared__ double s_dyn[];
  double* s_acc = s_dyn;                              // [2M][kBlock]: ||y_j||^2 at 2j, sum y_j at 2j + 1
  double* s_w = s_dyn + 2 * M * kBlock;               // [k][M]
  __shared__ bool s_last;
  const int tid = threadIdx.x;
  for (uint32_t i = tid; i < k * M; i += kBlock) s_w[i] = W[i];
#pragma unroll
  for (int v = 0; v < 2 * M; v++) s_acc[v * kBlock + tid] = 0.0;
  __syncthreads();
  const uint64_t ng = n / E, ldg = ldv / E;
  for (uint64_t i = (uint64_t)blockIdx.x * kBlock + tid; i < ng; i += (uint64_t)gridDim.x * kBlock) {
    double acc[M][E];
#pragma unroll
    for (int j = 0; j < M; j++)
#pragma unroll
      for (int e = 0; e < E; e++) acc[j][e] = 0.0;
    uint32_t t = 0;
    for (; t + U <= k; t += U) {
      double vv[U][E];
#pragma unroll
      for (int u = 0; u < U; u++) ld_group<TV>(V, (uint64_t)(t + u) * ldg + i, vv[u]);
#pragma unroll
      for (int u = 0; u < U; u++)
#pragma unroll
        for (int j = 0; j < M; j++) {
          const double w = s_w[(t + u) * M + j];
#pragma unroll
          for (int e = 0; e < E; e++) acc[j][e] += w * vv[u][e];
        }
    }
    for (; t < k; t++) {
      double vv[E];
      ld_group<TV>(V, (uint64_t)t * ldg + i, vv);
#pragma unroll
      for (int j = 0; j < M; j++)
#pragma unroll
        for (int e = 0; e < E; e++) acc[j][e] += s_w[t * M + j] * vv[e];
    }
#pragma unroll
    for (int j = 0; j < M; j++) {
      double2* y2 = reinterpret_cast<double2*>(Y + (uint64_t)j * ldv);
      double q = 0.0, sm = 0.0;
#pragma unroll
      for (int h = 0; h < E / 2; h++) y2[i * (E / 2) + h] = make_double2(acc[j][2 * h], acc[j][2 * h + 1]);
#pragma unroll
      for (int e = 0; e < E; e++) { q += acc[j][e] * acc[j][e]; sm += acc[j][e]; }
      s_acc[(2 * j) * kBlock + tid] += q;
      s_acc[(2 * j + 1) * kBlock + tid] += sm;
    }
  }
  if (blockIdx.x == 0 && tid == 0)
    for (uint64_t r = ng * E; r < n; r++)
      for (int j = 0; j < M; j++) {
        double a = 0.0;
        for (uint32_t t = 0; t < k; t++) a += s_w[t * M + j] * (double)V[(uint64_t)t * ldv + r];
        Y[(uint64_t)j * ldv + r] = a;
        s_acc[(2 * j) * kBlock] += a * a;
        s_acc[(2 * j + 1) * kBlock] += a;
      }
  __syncthreads();
  const int lane = tid & 31, wid = tid >> 5;
  for (int v = wid; v < 2 * M; v += kWarps) {        // CTA partials: one warp per value, fixed order
    double a = 0.0;
    for (int i = lane; i < kBlock; i += 32) a += s_acc[v * kBlock + i];
    a = warp_sum(a);
    if (lane == 0) partials[(uint64_t)v * gridDim.x + blockIdx.x] = a;
  }
  // last CTA: one warp per value, lanes stride the CTA partials in index order (as k_multidot)
  __syncthreads();
  if (tid == 0) {
    __threadfence();
    const unsigned int tk = atomicAdd(ticket, 1u);
    s_last = (tk == gridDim.x - 1);
  }
  __syncthreads();
  if (!s_last) return;
  __threadfence();
  for (int v = wid; v < 2 * M; v += kWarps) {
    double a = 0.0;
    for (unsigned int i = lane; i < gridDim.x; i += 32) a += __ldcg(partials + (uint64_t)v * gridDim.x + i);
    a = warp_sum(a);
    if (lane == 0) ((v & 1) ? vsum : nrm2)[v >> 1] = a;
  }
  if (tid == 0) *ticket = 0u;
}

// sum_i v[i] (m = 1: the sign of the vector k_combine built)
__global__ void __launch_bounds__(kBlock) k_vsum(const double* __restrict__ v, uint64_t n, double* partials, unsigned int* ticket, double* out) {
  __shared__ double sm[kWarps];
  __shared__ bool s_last;
  double acc = 0.0;
  for (uint64_t i = (uint64_t)blockIdx.x * kBlock + threadIdx.x; i < n; i += (uint64_t)gridDim.x * kBlock) acc += v[i];
  acc = block_sum(acc, sm);
  grid_sum_finish(acc, partials, ticket, out, sm, &s_last);
}

// max of non-negative doubles through their bit patterns (ordered like the values): exact, so the order of arrival does not matter
__device__ __forceinline__ void block_max_to(double v, double* sm, unsigned long long* out) {
  for (int o = 16; o > 0; o >>= 1) v = fmax(v, __shfl_xor_sync(0xffffffffu, v, o));
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  __syncthreads();
  if (lane == 0) sm[wid] = v;
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int w = 1; w < kWarps; w++) v = fmax(v, sm[w]);
    atomicMax(out, (unsigned long long)__double_as_longlong(v));
  }
}

// y_j *= sgn(vsum_j) / sqrt(nrm2_j) for j < m (unit 2-norm, sum_i y_j(i) >= 0); max |y_0| -> *absmax0 (bits of a double)
__global__ void __launch_bounds__(kBlock) k_ritz_scale(double* __restrict__ Y, uint64_t ldv, uint32_t m, uint64_t n, const double* __restrict__ nrm2,
                                                       const double* __restrict__ vsum, unsigned long long* absmax0) {
  __shared__ double sm[kWarps];
  double mx = 0.0;
  for (uint32_t j = 0; j < m; j++) {
    const double s = (vsum[j] < 0.0 ? -1.0 : 1.0) / sqrt(nrm2[j]);
    double* y = Y + (uint64_t)j * ldv;
    for (uint64_t i = (uint64_t)blockIdx.x * kBlock + threadIdx.x; i < n; i += (uint64_t)gridDim.x * kBlock) {
      const double v = y[i] * s;
      y[i] = v;
      if (j == 0) mx = fmax(mx, fabs(v));
    }
  }
  block_max_to(mx, sm, absmax0);
}

// Collatz-Wielandt weights z = max(|y_0|, delta * max|y_0|) > 0, entry-wise; z may be y (several GPUs: in place on the gathered vector)
__global__ void __launch_bounds__(kBlock) k_cw_z(const double* y, double* z, uint64_t n, const double* __restrict__ absmax,
                                                 double delta) {
  const double floor_v = delta * *absmax;
  for (uint64_t i = (uint64_t)blockIdx.x * kBlock + threadIdx.x; i < n; i += (uint64_t)gridDim.x * kBlock) z[i] = fmax(fabs(y[i]), floor_v);
}

// max over this rank's vertices (padding slots excluded) of (A z)_i / z_i -> *out (bits of a double). zfull is the gathered z.
__global__ void __launch_bounds__(kBlock) k_cw_bound(const double* __restrict__ az, const double* __restrict__ zfull, uint64_t n, uint64_t cl,
                                                     uint32_t world, uint32_t rank, const uint32_t* __restrict__ new2old,
                                                     unsigned long long* out) {
  __shared__ double sm[kWarps];
  double mx = 0.0;
  for (uint64_t l = (uint64_t)blockIdx.x * kBlock + threadIdx.x; l < n; l += (uint64_t)gridDim.x * kBlock) {
    const uint64_t slot = xfull_index(l, cl, world, rank);
    if (new2old[slot] != 0xFFFFFFFFu) mx = fmax(mx, az[l] / zfull[slot]);
  }
  block_max_to(mx, sm, out);
}

inline unsigned stream_grid(const lz_ctx* c, uint64_t work_items /* per-thread items */) {
  uint64_t want = (work_items + kBlock - 1) / kBlock;
  uint64_t cap = (uint64_t)c->sm_count * 8;
  if (want < 1) want = 1;
  return (unsigned)(want < cap ? want : cap);
}

}  // namespace

#define LZ_LAUNCH_CHECK()                                                                         \
  do {                                                                                            \
    cudaError_t e_ = cudaGetLastError();                                                          \
    if (e_ != cudaSuccess) return lz_fail(LZ_ERR_CUDA, "%s:%d launch -> %s", __FILE__, __LINE__, cudaGetErrorString(e_)); \
    c->launches++;                                                                                \
  } while (0)

static int ensure_partials(lz_ctx* c, uint64_t count) {
  if (count <= c->partials_cap) return LZ_OK;
  // only grows between runs; in-flight kernels are ordered on the same stream, and cudaFree synchronises
  cudaFree(c->partials);
  c->partials = nullptr; c->partials_cap = 0;
  LZ_CUDA(cudaMalloc((void**)&c->partials, count * sizeof(double)));
  c->partials_cap = (uint32_t)count;
  return LZ_OK;
}

static lz_red make_red(const lz_ctx* c, unsigned long long seq) {
  lz_red red;
  memset(&red, 0, sizeof(red));
  red.seq = seq; red.world = (uint32_t)c->world; red.rank = (uint32_t)c->rank;
  if (seq)
    for (int r = 0; r < LZ_MAX_WORLD; r++)
      red.area[r] = c->peer_flags[r] ? reinterpret_cast<lz_red_slot*>(c->peer_flags[r] + (size_t)LZ_MAX_COLBLK * LZ_MAX_WORLD) : nullptr;
  return red;
}

int lz_k_spmv_dot(lz_ctx* c, const double* x_gather, const double* q_local, double* w_out, double* alpha_out, unsigned long long wait_seq,
                  const double* push_src, unsigned long long red_seq, const double* alpha_div) {
  const lz_red red = make_red(c, red_seq);
  for (uint32_t blk = 0; blk < c->ncolblk; blk++) {
    lz_push_job job;
    memset(&job, 0, sizeof(job));
    if (push_src && blk + 1 < c->ncolblk) {      // this pass also sends chunk blk + 1 of the vector being gathered
      for (int r = 0; r < LZ_MAX_WORLD; r++) { job.peers.x[r] = c->peer_xfull[r]; job.peers.f[r] = c->peer_flags[r]; }
      job.src = push_src; job.ticket = c->push_ticket; job.seq = wait_seq; job.cl = c->chunk_rows;
      job.chunk = blk + 1; job.rank = (uint32_t)c->rank; job.nctas = c->push_ctas ? c->push_ctas : (uint32_t)c->sm_count / 4;   // 37 of 148: measured best at 8 GPUs (74: -4 %, 148: -10 %)
    }
    const int acc = blk > 0, fin = blk + 1 == c->ncolblk;
    // pass `blk` gathers from chunk `blk` of the gathered vector only: wait for exactly that piece of the all-gather
    if (c->chunks_in_flight) LZ_CUDA(cudaStreamWaitEvent(c->stream, c->ev_chunk[blk], 0));
    if (c->spmv_variant == LZ_SPMV_AUTO) {          // sliced layout: long rows warp-per-row, short rows 32 per warp
      uint32_t grid = (uint32_t)c->sm_count * c->spmv_ctas_per_sm;
      uint32_t group = (c->n_items >= 64u * grid * kWarps) ? 4u : 1u;   // quads only when every warp still gets >= 16 of them
      if (c->sell_group_force) group = c->sell_group_force;              // test knob (LZ_SELL_GROUP): small inputs through the quad paths
      const bool narrow = c->sell_narrow[blk] && group == 4;
      if (narrow && c->spmv_ctas_per_sm > 4) grid = (uint32_t)c->sm_count * 4;   // 64 registers: 4 resident CTAs per SM, one wave
      // the sender CTAs of the fused exchange take resident slots: gatherers + senders must still fit in ONE wave, or the
      // gatherers left over start when the first ones finish and the pass takes twice as long (measured at 8 GPUs: 205 vs 105 us)
      if (job.nctas && grid > job.nctas + (uint32_t)c->sm_count) grid -= job.nctas;
      const uint32_t need = ((c->n_items + group - 1) / group + kWarps - 1) / kWarps;
      if (grid > need) grid = need;
      if (grid < 1) grid = 1;
      LZ_TRY(ensure_partials(c, grid));
      grid += job.nctas;
      const bool peer = c->world > 1;
      auto kern = narrow ? (peer ? k_spmv_sell<true, true> : k_spmv_sell<true, false>) : (peer ? k_spmv_sell<false, true> : k_spmv_sell<false, false>);
      kern<<<grid, kBlock, 0, c->stream>>>(c->sell_sp + (uint64_t)blk * c->n_items, c->sell_col, c->n_long, c->n_items,
                                           (uint32_t)c->n_loc, x_gather, q_local, w_out, c->partials, c->ticket + 0, alpha_out, acc, fin,
                                           c->flags, blk, (uint32_t)c->world, wait_seq, job, group, red, alpha_div);
    } else {                                         // CSR: vector (sub-warp) per row by degree bin, or warp per row
      const lz_spmv_plan& plan = (c->spmv_variant == LZ_SPMV_WARP) ? c->plan_warp : c->plan_auto[blk];
      if (plan.nitems == 0) return lz_fail(LZ_ERR_ARG, "empty SpMV plan");
      uint32_t grid = (uint32_t)c->sm_count * c->spmv_ctas_per_sm;
      if (grid > plan.nitems) grid = plan.nitems;
      LZ_TRY(ensure_partials(c, grid));
      auto kern = c->world > 1 ? k_spmv_dot<true> : k_spmv_dot<false>;
      kern<<<grid, kBlock, 0, c->stream>>>(plan, c->seg[blk], c->seg[blk] + 1, c->col, x_gather, q_local, w_out, c->partials,
                                           c->ticket + 0, alpha_out, acc, fin, c->flags, blk, (uint32_t)c->world, wait_seq, alpha_div);
    }
    LZ_LAUNCH_CHECK();
  }
  c->chunks_in_flight = false;
  return LZ_OK;
}

int lz_k_update_norm(lz_ctx* c, double* w, const double* qj, const double* qprev, double* alpha, const double* beta_prev,
                     double* norm2_out, unsigned long long red_seq) {
  unsigned g = stream_grid(c, c->n_loc / 2 + 1);
  LZ_TRY(ensure_partials(c, g));
  k_update_norm<<<g, kBlock, 0, c->stream>>>(w, qj, qprev, alpha, beta_prev, c->n_loc, c->partials, c->ticket + 1, norm2_out,
                                             make_red(c, red_seq), alpha);
  LZ_LAUNCH_CHECK();
  return LZ_OK;
}

int lz_k_update_lagged(lz_ctx* c, const double* t, const double* uj, const double* uprev, const double* alpha, const double* norm2_j,
                       const double* norm2_prev, double* u_next, double* norm2_out, double* beta_out, float* u32_next) {
  unsigned g = stream_grid(c, c->n_loc / 2 + 1);
  LZ_TRY(ensure_partials(c, g));
  k_update_lagged<<<g, kBlock, 0, c->stream>>>(t, uj, uprev, alpha, norm2_j, norm2_prev, c->n_loc, u_next, c->partials, c->ticket + 1,
                                               norm2_out, beta_out, u32_next);
  LZ_LAUNCH_CHECK();
  return LZ_OK;
}
int lz_k_update_lagged_push(lz_ctx* c, const double* t, const double* uj, const double* uprev, double* u_next, uint32_t j,
                            unsigned long long push_seq, uint32_t push_chunks, unsigned long long red_seq, float* u32_next) {
  lz_peers peers;
  for (int r = 0; r < LZ_MAX_WORLD; r++) { peers.x[r] = c->peer_xfull[r]; peers.f[r] = c->peer_flags[r]; }
  lz_push_lists lists;
  lists.list = c->push_list;
  for (int r = 0; r <= LZ_MAX_WORLD; r++) lists.off[r] = c->push_off[r];
  // the same grid whatever the exchange mode: the partition of the ||u||^2 partial sums (hence its bits) must not depend on it
  unsigned g = stream_grid(c, c->chunk_rows / 2 + 1);
  const unsigned cap = (unsigned)c->sm_count * 4;
  if (g > cap) g = cap;
  LZ_TRY(ensure_partials(c, g));
  auto kern = c->sparse_push ? k_update_lagged_push<true> : k_update_lagged_push<false>;
  kern<<<g, kBlock, 0, c->stream>>>(t, uj, uprev, c->n_loc, u_next, c->norm2v, j, c->alpha, c->beta, peers, c->chunk_rows, c->ncolblk, push_chunks,
                                    (uint32_t)c->world, (uint32_t)c->rank, push_seq, c->push_ticket, c->partials, c->ticket + 1, make_red(c, red_seq), lists,
                                    u32_next);
  LZ_LAUNCH_CHECK();
  return LZ_OK;
}
int lz_k_lagged_finish(lz_ctx* c, uint32_t j, unsigned long long red_seq) {
  k_lagged_finish<<<1, 32, 0, c->stream>>>(j, c->norm2v, c->alpha, c->beta, make_red(c, red_seq));
  LZ_LAUNCH_CHECK();
  return LZ_OK;
}
int lz_k_set_trace(lz_ctx* c, unsigned long long* buf_device) {
  LZ_CUDA(cudaMemcpyToSymbolAsync(g_trace, &buf_device, sizeof(buf_device), 0, cudaMemcpyHostToDevice, c->stream));
  return LZ_OK;
}
int lz_k_set_peer_timeout(lz_ctx* c, double seconds) {
  const unsigned long long ns = seconds <= 0.0 ? 0ull : (unsigned long long)(seconds * 1e9);
  LZ_CUDA(cudaMemcpyToSymbol(g_peer_timeout_ns, &ns, sizeof(ns)));
  return LZ_OK;
}
int lz_k_coef_scale(lz_ctx* c, const double* coef, const double* norm2, uint32_t k, double* out) {
  k_coef_scale<<<(k + 127) / 128, 128, 0, c->stream>>>(coef, norm2, k, out);
  LZ_LAUNCH_CHECK();
  return LZ_OK;
}
int lz_k_div_sqrt(lz_ctx* c, double* v, uint64_t n, const double* norm2) {
  k_div_sqrt<<<stream_grid(c, n), kBlock, 0, c->stream>>>(v, n, norm2);
  LZ_LAUNCH_CHECK();
  return LZ_OK;
}

int lz_k_convert(lz_ctx* c, const double* src64, float* dst32, const float* src32, double* dst64, uint64_t n) {
  if (dst32) k_to_f32<<<stream_grid(c, n), kBlock, 0, c->stream>>>(src64, dst32, n);
  else k_to_f64<<<stream_grid(c, n), kBlock, 0, c->stream>>>(src32, dst64, n);
  LZ_LAUNCH_CHECK();
  return LZ_OK;
}
int lz_k_scale(lz_ctx* c, const double* w, const double* norm2, double* q_next, double* xfull, double* beta_out, float* q32_next) {
  unsigned g = stream_grid(c, c->n_loc / 2 + 1);
  k_scale<<<g, kBlock, 0, c->stream>>>(w, norm2, c->n_loc, q_next, xfull, c->chunk_rows, (uint32_t)c->world, (uint32_t)c->rank, beta_out, q32_next);
  LZ_LAUNCH_CHECK();
  return LZ_OK;
}

int lz_k_scale_push(lz_ctx* c, const double* w, const double* norm2, double* q_next, double* beta_out, unsigned long long seq,
                    uint32_t push_chunks, unsigned long long red_seq) {
  lz_peers peers;
  for (int r = 0; r < LZ_MAX_WORLD; r++) { peers.x[r] = c->peer_xfull[r]; peers.f[r] = c->peer_flags[r]; }
  if (c->sparse_push) {            // needed-columns exchange: all chunks are sent (and flagged) by this one launch
    lz_push_lists lists;
    lists.list = c->push_list;
    for (int r = 0; r <= LZ_MAX_WORLD; r++) lists.off[r] = c->push_off[r];
    k_scale_push_sparse<<<stream_grid(c, c->n_loc / 2 + 1), kBlock, 0, c->stream>>>(w, norm2, c->n_loc, q_next, peers, c->chunk_rows, c->ncolblk,
                                                                                   (uint32_t)c->world, (uint32_t)c->rank, seq, c->push_ticket,
                                                                                   beta_out, make_red(c, red_seq), lists);
    LZ_LAUNCH_CHECK();
    return LZ_OK;
  }
  // few CTAs suffice to saturate NVLink; cap so the per-chunk ticketing stays cheap
  unsigned g = stream_grid(c, c->chunk_rows / 2 + 1);
  const unsigned cap = (unsigned)c->sm_count * 2;
  if (g > cap) g = cap;
  k_scale_push<<<g, kBlock, 0, c->stream>>>(w, norm2, c->n_loc, q_next, peers, c->chunk_rows, c->ncolblk, push_chunks, (uint32_t)c->world,
                                            (uint32_t)c->rank, seq, c->push_ticket, beta_out, make_red(c, red_seq));
  LZ_LAUNCH_CHECK();
  return LZ_OK;
}

int lz_k_permute_in_local(lz_ctx* c, const double* x_orig, const double* norm2, double* q0_local) {
  k_permute_in_local<<<stream_grid(c, c->n_loc), kBlock, 0, c->stream>>>(x_orig, c->new2old, c->n_loc, c->chunk_rows, (uint32_t)c->world,
                                                                        (uint32_t)c->rank, norm2, c->x_exp, q0_local);
  LZ_LAUNCH_CHECK();
  return LZ_OK;
}

int lz_k_spread(lz_ctx* c, const double* local, double* xfull) {
  unsigned g = stream_grid(c, c->n_loc / 2 + 1);
  k_spread_collect<<<g, kBlock, 0, c->stream>>>(const_cast<double*>(local), xfull, c->n_loc, c->chunk_rows, (uint32_t)c->world,
                                                (uint32_t)c->rank, 0);
  LZ_LAUNCH_CHECK();
  return LZ_OK;
}

int lz_k_collect(lz_ctx* c, const double* xfull, double* local) {
  unsigned g = stream_grid(c, c->n_loc / 2 + 1);
  k_spread_collect<<<g, kBlock, 0, c->stream>>>(local, const_cast<double*>(xfull), c->n_loc, c->chunk_rows, (uint32_t)c->world,
                                                (uint32_t)c->rank, 1);
  LZ_LAUNCH_CHECK();
  return LZ_OK;
}

int lz_k_norm2(lz_ctx* c, const double* v, uint64_t len, int e, double* out) {
  unsigned g = stream_grid(c, len);
  LZ_TRY(ensure_partials(c, g));
  k_norm2<<<g, kBlock, 0, c->stream>>>(v, len, e, c->partials, c->ticket + 2, out);
  LZ_LAUNCH_CHECK();
  return LZ_OK;
}

int lz_k_absmax_bits(lz_ctx* c, const double* v, uint64_t len, unsigned long long* out) {
  k_absmax_bits<<<stream_grid(c, len), kBlock, 0, c->stream>>>(v, len, out);
  LZ_LAUNCH_CHECK();
  return LZ_OK;
}

int lz_k_multidot(lz_ctx* c, const void* V, bool f32, uint32_t nvec, const double* w, double* h_out, const int* skip, const double* h_div) {
  unsigned g = (unsigned)c->sm_count * 4;
  uint64_t want = (c->n_loc / (f32 ? 4 : 2) + kBlock) / kBlock;
  if (want < g) g = (unsigned)(want ? want : 1);
  LZ_TRY(ensure_partials(c, (uint64_t)g * nvec));
  if (f32) k_multidot<float><<<g, kBlock, 0, c->stream>>>((const float*)V, c->ldv, nvec, w, c->n_loc, c->partials, c->ticket + 3, h_out, skip, h_div);
  else k_multidot<double><<<g, kBlock, 0, c->stream>>>((const double*)V, c->ldv, nvec, w, c->n_loc, c->partials, c->ticket + 3, h_out, skip, h_div);
  LZ_LAUNCH_CHECK();
  return LZ_OK;
}

int lz_k_combine(lz_ctx* c, const void* V, bool f32, uint32_t nvec, const double* coef, double coef_sign, const double* base, double* out,
                 double* norm2_out, const int* skip, float* out32) {
  unsigned g = stream_grid(c, c->n_loc / 2 + 1);
  LZ_TRY(ensure_partials(c, g));
  if (f32) k_combine<float><<<g, kBlock, nvec * sizeof(double), c->stream>>>((const float*)V, c->ldv, nvec, coef, coef_sign, base, out, c->n_loc,
                                                                             c->partials, c->ticket + 4, norm2_out, skip, out32);
  else k_combine<double><<<g, kBlock, nvec * sizeof(double), c->stream>>>((const double*)V, c->ldv, nvec, coef, coef_sign, base, out, c->n_loc,
                                                                          c->partials, c->ticket + 4, norm2_out, skip, out32);
  LZ_LAUNCH_CHECK();
  return LZ_OK;
}

int lz_k_reorth_decide(lz_ctx* c, const double* norm2_before, const double* norm2_after, int* skip, unsigned int* second_passes) {
  static const int always = getenv("LZ_REORTH_ALWAYS_TWICE") && atoi(getenv("LZ_REORTH_ALWAYS_TWICE")) != 0;   // test knob
  k_reorth_decide<<<1, 1, 0, c->stream>>>(norm2_before, norm2_after, skip, second_passes, always);
  LZ_LAUNCH_CHECK();
  return LZ_OK;
}
int lz_k_reorth_select(lz_ctx* c, const int* skip, const double* norm2_second, double* norm2, double* norm2_copy, double* beta_out) {
  k_reorth_select<<<1, 1, 0, c->stream>>>(skip, norm2_second, norm2, norm2_copy, beta_out);
  LZ_LAUNCH_CHECK();
  return LZ_OK;
}

// Same solve for the leading k x k block into caller-provided scratch (convergence estimate; nothing of the ctx's result is touched).
int lz_k_tridiag_expv_into(lz_ctx* c, uint32_t k, double* eigvals, double* eigvecs, double* work, double* coef, int* status,
                           const double* ls_in, double* ls_out) {
  if (k > (uint32_t)kEigMax) return lz_fail(LZ_ERR_ARG, "krylov dimension %u exceeds the on-device eigensolver limit %d", k, kEigMax);
  const size_t zt_bytes = (size_t)k * k * sizeof(double);
  const int in_smem = zt_bytes <= 180 * 1024;
  if (in_smem) LZ_CUDA(cudaFuncSetAttribute(k_tridiag_expv, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)zt_bytes));
  k_tridiag_expv<<<1, kBlock, in_smem ? zt_bytes : 0, c->stream>>>(k, c->alpha, c->beta, c->scal + 2, c->x_exp, eigvals, eigvecs, work, coef, status, in_smem,
                                                                  c->matfun_kind, c->matfun_param, ls_in, ls_out);
  LZ_LAUNCH_CHECK();
  return LZ_OK;
}

int lz_k_tridiag_expv(lz_ctx* c, uint32_t k) {
  return lz_k_tridiag_expv_into(c, k, c->eigvals, c->eigvecs, c->eigwork, c->coef, c->status, nullptr, c->scal + 5);
}

int lz_k_permute_in(lz_ctx* c, const double* x_orig, const double* norm2, uint64_t first, uint64_t count, double* dst) {
  unsigned g = stream_grid(c, count);
  if (norm2) k_permute_in<<<g, kBlock, 0, c->stream>>>(x_orig, c->new2old, first, count, norm2, c->x_exp, dst);
  else k_permute_in_raw<<<g, kBlock, 0, c->stream>>>(x_orig, c->new2old, first, count, dst);
  LZ_LAUNCH_CHECK();
  return LZ_OK;
}

int lz_k_permute_out(lz_ctx* c, const double* y_new_full, double* y_orig) {
  uint64_t count = c->n_loc * (uint64_t)c->world;
  unsigned g = stream_grid(c, count);
  k_permute_out<<<g, kBlock, 0, c->stream>>>(y_new_full, c->new2old, count, y_orig);
  LZ_LAUNCH_CHECK();
  return LZ_OK;
}

int lz_k_fill(lz_ctx* c, double* p, uint64_t n, double value) {
  k_fill<<<stream_grid(c, n), kBlock, 0, c->stream>>>(p, n, value);
  LZ_LAUNCH_CHECK();
  return LZ_OK;
}

int lz_k_reserve_partials(lz_ctx* c, uint64_t count) { return ensure_partials(c, count); }

int lz_k_ritz_select(lz_ctx* c, uint32_t k, uint32_t m, uint32_t M, const double* eigvals, const double* eigvecs, const double* norm2, double* W,
                     double* theta) {
  k_ritz_select<<<1, kBlock, 0, c->stream>>>(k, m, M, eigvals, eigvecs, norm2, W, theta);
  LZ_LAUNCH_CHECK();
  return LZ_OK;
}

template <class TV, int M>
static int launch_ritz_combine(lz_ctx* c, const TV* V, uint32_t k, const double* W, double* Y, double* partials, double* nrm2, double* vsum) {
  const unsigned g = stream_grid(c, c->n_loc / 2 + 1);
  const size_t smem = ((size_t)k * M + 2 * M * kBlock) * sizeof(double);
  if (smem > 48 * 1024) LZ_CUDA(cudaFuncSetAttribute(k_ritz_combine<TV, M>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  k_ritz_combine<TV, M><<<g, kBlock, smem, c->stream>>>(V, c->ldv, k, W, Y, c->n_loc, partials, c->ticket + 5, nrm2, vsum);
  LZ_LAUNCH_CHECK();
  return LZ_OK;
}

int lz_k_ritz_combine(lz_ctx* c, const void* V, bool f32, uint32_t k, uint32_t M, const double* W, double* Y, double* partials, double* nrm2,
                      double* vsum) {
  if (k > (uint32_t)kEigMax) return lz_fail(LZ_ERR_ARG, "krylov dimension %u exceeds %d", k, kEigMax);
  static_assert(((size_t)kEigMax * 16 + 2 * 16 * kBlock) * sizeof(double) <= 227 * 1024, "W of the largest k must fit in shared memory");
#define LZ_RITZ_CASE(MM)                                                                                                  \
  case MM:                                                                                                                \
    return f32 ? launch_ritz_combine<float, MM>(c, (const float*)V, k, W, Y, partials, nrm2, vsum)                      \
               : launch_ritz_combine<double, MM>(c, (const double*)V, k, W, Y, partials, nrm2, vsum);
  switch (M) {
    LZ_RITZ_CASE(2)
    LZ_RITZ_CASE(4)
    LZ_RITZ_CASE(8)
    LZ_RITZ_CASE(16)
    default: return lz_fail(LZ_ERR_ARG, "Ritz block width %u is not 2, 4, 8 or 16", M);
  }
#undef LZ_RITZ_CASE
}

int lz_k_vsum(lz_ctx* c, const double* v, uint64_t n, double* partials, double* out) {
  k_vsum<<<stream_grid(c, n), kBlock, 0, c->stream>>>(v, n, partials, c->ticket + 5, out);
  LZ_LAUNCH_CHECK();
  return LZ_OK;
}

int lz_k_ritz_scale(lz_ctx* c, double* Y, uint32_t m, const double* nrm2, const double* vsum, unsigned long long* absmax0) {
  k_ritz_scale<<<stream_grid(c, c->n_loc), kBlock, 0, c->stream>>>(Y, c->ldv, m, c->n_loc, nrm2, vsum, absmax0);
  LZ_LAUNCH_CHECK();
  return LZ_OK;
}

int lz_k_cw_z(lz_ctx* c, const double* y, double* z, uint64_t n, const double* absmax, double delta) {
  k_cw_z<<<stream_grid(c, n), kBlock, 0, c->stream>>>(y, z, n, absmax, delta);
  LZ_LAUNCH_CHECK();
  return LZ_OK;
}

int lz_k_cw_bound(lz_ctx* c, const double* az, const double* zfull, unsigned long long* out) {
  k_cw_bound<<<stream_grid(c, c->n_loc), kBlock, 0, c->stream>>>(az, zfull, c->n_loc, c->chunk_rows, (uint32_t)c->world, (uint32_t)c->rank,
                                                                c->new2old, out);
  LZ_LAUNCH_CHECK();
  return LZ_OK;
}
