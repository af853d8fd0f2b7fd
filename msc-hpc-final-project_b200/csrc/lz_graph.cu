// lz_graph.cu — adjacency matrix on the device: synthetic-graph construction, relabelling, sharding, SpMV launch plan.
//
// Replaces, for the B200 path, the host loader adjMatrix::populate_sparse_matrix (reference
// parallel-final/lib/adjMatrix.cc:21-46; std::set, 8-55 s per graph in the published runs) and the per-GPU offset
// rebasing of parallel-two-cards/lib/cu_lanczos.cu:21-27,62-69. CUB is used for the (setup-time) sorts and scans; the
// hot-path kernels are in lz_kernels.cu.
//
// Internal vertex order. Vertices are sorted by degree (descending, ties by original id) and dealt cyclically to the
// `world` ranks: the vertex at sorted position s lives on rank s % world at local row s / world and gets the new global
// id (s % world) * n_loc + s / world. Consequences: (1) every rank owns the same number of rows with a near-identical
// degree profile, so nnz, vector work and basis memory are balanced without a separate partitioner; (2) local rows are
// sorted by length, so each SpMV degree bin is a contiguous row range served by one lanes-per-row variant with no
// intra-warp imbalance; (3) high-degree (= most frequently gathered) entries of x are contiguous, which keeps the hot
// part of x resident in L2; (4) ownership blocks are equal-sized and contiguous in the new numbering, so the Krylov
// vector is exchanged with a plain ncclAllGather.
#include "lz_ctx.h"
#include "lz_gen.h"

#include <cub/cub.cuh>
#include <stdlib.h>
#include <vector>

namespace {

__global__ void k_gen_keys(lz_gen_params p, uint64_t* __restrict__ keys) {
  uint64_t e = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (e > p.m) return;
  uint32_t u, v;
  lz_gen_edge(p, e, &u, &v);
  uint64_t a = ~0ull, b = ~0ull;   // sentinel sorts last
  if (u != v) { a = ((uint64_t)u << 32) | v; b = ((uint64_t)v << 32) | u; }
  keys[2 * e] = a;
  keys[2 * e + 1] = b;
}

// ro[r] = number of keys with row < r  (keys sorted, unique, no sentinel)
__global__ void k_row_offsets_from_keys(const uint64_t* __restrict__ keys, uint64_t nnz, uint64_t n, uint32_t* __restrict__ ro) {
  uint64_t r = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (r > n) return;
  uint64_t target = r << 32, lo = 0, hi = nnz;
  while (lo < hi) {
    uint64_t mid = (lo + hi) >> 1;
    if (keys[mid] < target) lo = mid + 1; else hi = mid;
  }
  ro[r] = (uint32_t)lo;
}

__global__ void k_low32(const uint64_t* __restrict__ keys, uint64_t nnz, uint32_t* __restrict__ out) {
  uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < nnz) out[i] = (uint32_t)keys[i];
}

__global__ void k_iota_u32(uint32_t* p, uint64_t n) {
  uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) p[i] = (uint32_t)i;
}

// number of stored entries whose column is within `radius` of the row (how band-like the natural numbering is)
__global__ void k_locality(const uint32_t* __restrict__ ro, const uint32_t* __restrict__ ci, uint64_t n, uint64_t radius,
                           unsigned long long* __restrict__ out) {
  unsigned long long acc = 0;
  for (uint64_t r = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; r < n; r += (uint64_t)gridDim.x * blockDim.x)
    for (uint32_t j = ro[r]; j < ro[r + 1]; j++) {
      const uint64_t cc = ci[j];
      acc += (cc > r ? cc - r : r - cc) <= radius;
    }
  for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
  if ((threadIdx.x & 31) == 0 && acc) atomicAdd(out, acc);
}

__global__ void k_fill_u32(uint32_t* p, uint64_t n, uint32_t v) {
  uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) p[i] = v;
}

// sorted position s -> new id; builds old2new and new2old. Rank = s % world, local row l = s / world; the global
// numbering is chunk-major: id = (l / cl) * (world * cl) + rank * cl + (l % cl), so chunk c of every rank's rows forms
// one contiguous window of the gathered vector (= one column block = one piece of the pipelined all-gather).
// block_rows == 0: positions are dealt cyclically (degree order); > 0: contiguous blocks of block_rows positions per rank
// (natural order, keeps the locality of banded / mesh-like graphs).
__global__ void k_relabel(const uint32_t* __restrict__ sorted_old, uint64_t n, uint32_t world, uint64_t cl, uint64_t block_rows,
                          uint32_t* __restrict__ old2new, uint32_t* __restrict__ new2old) {
  uint64_t s = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= n) return;
  uint32_t old = sorted_old[s];
  const uint64_t r = block_rows ? s / block_rows : s % world, l = block_rows ? s % block_rows : s / world;
  uint32_t nw = (uint32_t)((l / cl) * (world * cl) + r * cl + (l % cl));
  old2new[old] = nw;
  new2old[nw] = old;
}

// one warp per local row: keys[row_ptr[l] + j] = (colblock << (32 + rowbits)) | (l << 32) | newcol, newcol = old2new[ci[ro[old] + j]]
// Sorting these keys lays col[] out column-block-major (each SpMV pass streams one contiguous piece), row-major inside
// a block, ascending column inside a row slice.
__global__ void k_local_keys(const uint32_t* __restrict__ sorted_old, const uint32_t* __restrict__ ro, const uint32_t* __restrict__ ci,
                             const uint32_t* __restrict__ old2new, const uint32_t* __restrict__ row_ptr, uint64_t n, uint32_t world,
                             uint32_t rank, uint64_t n_loc, uint64_t block_rows, uint64_t width, int rowbits, uint64_t* __restrict__ keys) {
  uint64_t warp = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  uint32_t lane = threadIdx.x & 31;
  if (warp >= n_loc) return;
  uint64_t s = block_rows ? (uint64_t)rank * block_rows + warp : warp * world + rank;
  if (s >= n) return;
  uint32_t old = sorted_old[s];
  uint32_t b = ro[old], e = ro[old + 1], dst = row_ptr[warp];
  for (uint32_t j = b + lane; j < e; j += 32) {
    const uint32_t nc = old2new[ci[j]];
    keys[dst + (j - b)] = ((uint64_t)(nc / width) << (32 + rowbits)) | (warp << 32) | nc;
  }
}

// blk_rp[b * (n_loc + 1) + row] = first key position of (block b, row); row == n_loc gives the end of block b
__global__ void k_block_row_ptr(const uint64_t* __restrict__ keys, uint64_t nnz, uint64_t n_loc, uint32_t nblk, int rowbits,
                                uint32_t* __restrict__ blk_rp) {
  uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (uint64_t)nblk * (n_loc + 1)) return;
  const uint64_t b = i / (n_loc + 1), row = i % (n_loc + 1);
  const uint64_t target = (b << (32 + rowbits)) + (row << 32);   // row == n_loc may carry into the block field: intended
  uint64_t lo = 0, hi = nnz;
  while (lo < hi) {
    uint64_t mid = (lo + hi) >> 1;
    if (keys[mid] < target) lo = mid + 1; else hi = mid;
  }
  blk_rp[i] = (uint32_t)lo;
}

// first local row whose length is <= thr[t]  (lengths are non-increasing)
__global__ void k_bin_bounds(const uint32_t* __restrict__ row_ptr, uint32_t n_loc, const uint32_t* __restrict__ thr, uint32_t nthr,
                             uint32_t* __restrict__ out) {
  uint32_t t = threadIdx.x;
  if (t >= nthr) return;
  uint32_t lo = 0, hi = n_loc;
  while (lo < hi) {
    uint32_t mid = (lo + hi) >> 1;
    uint32_t len = row_ptr[mid + 1] - row_ptr[mid];
    if (len > thr[t]) lo = mid + 1; else hi = mid;
  }
  out[t] = lo;
}

// out[bin * nblk + b] = number of entries of column block b in the rows of bin `bin`  (grid = (nbins, nblk))
__global__ void k_bin_block_nnz(const uint32_t* const* __restrict__ seg, const uint32_t* __restrict__ bin_rows /* [nbins+1] */,
                                uint32_t nblk, unsigned long long* __restrict__ out) {
  const uint32_t bin = blockIdx.x, b = blockIdx.y;
  const uint32_t* lo = seg[b];
  const uint32_t* hi = seg[b] + 1;
  unsigned long long acc = 0;
  for (uint32_t r = bin_rows[bin] + threadIdx.x; r < bin_rows[bin + 1]; r += blockDim.x) acc += hi[r] - lo[r];
  __shared__ unsigned long long sm[256];
  sm[threadIdx.x] = acc;
  __syncthreads();
  for (int o = 128; o > 0; o >>= 1) {
    if ((int)threadIdx.x < o) sm[threadIdx.x] += sm[threadIdx.x + o];
    __syncthreads();
  }
  if (threadIdx.x == 0) out[bin * nblk + b] = sm[0];
}

// ---- sliced layout (see lz_ctx.h) -------------------------------------------------------------------------------
// width (in chunks of 32 entries) of every (block, item). One warp per (block, item).
__global__ void k_sell_widths(const uint32_t* const* __restrict__ seg, uint32_t nblk, uint32_t n_long, uint32_t n_items, uint32_t n_loc,
                              uint32_t* __restrict__ widths /* [nblk * n_items + 1] */) {
  const uint64_t gw = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const uint32_t lane = threadIdx.x & 31;
  if (gw >= (uint64_t)nblk * n_items) return;
  const uint32_t b = (uint32_t)(gw / n_items), item = (uint32_t)(gw % n_items);
  const uint32_t* rp = seg[b];
  uint32_t wdt;
  if (item < n_long) {
    wdt = (rp[item + 1] - rp[item] + 31) >> 5;
  } else {
    const uint32_t row = n_long + (item - n_long) * 32 + lane;
    uint32_t len = row < n_loc ? rp[row + 1] - rp[row] : 0u;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) len = max(len, __shfl_xor_sync(0xffffffffu, len, o));
    wdt = len;
  }
  if (lane == 0) widths[gw] = wdt;
}

__global__ void k_sell_fill(const uint32_t* const* __restrict__ seg, const uint32_t* __restrict__ col, const uint32_t* __restrict__ sp,
                            uint32_t nblk, uint32_t n_long, uint32_t n_items, uint32_t n_loc, uint32_t* __restrict__ out) {
  const uint64_t gw = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const uint32_t lane = threadIdx.x & 31;
  if (gw >= (uint64_t)nblk * n_items) return;
  const uint32_t b = (uint32_t)(gw / n_items), item = (uint32_t)(gw % n_items);
  const uint32_t* rp = seg[b];
  const uint32_t c0 = sp[gw], nchunk = sp[gw + 1] - c0;
  uint32_t* dst = out + (uint64_t)c0 * 32 + lane;
  if (item < n_long) {
    const uint32_t beg = rp[item], len = rp[item + 1] - beg;
    for (uint32_t j = 0; j < nchunk; j++) {
      const uint32_t idx = j * 32 + lane;
      dst[(uint64_t)j * 32] = idx < len ? col[beg + idx] : 0xFFFFFFFFu;
    }
  } else {
    const uint32_t row = n_long + (item - n_long) * 32 + lane;
    const uint32_t beg = row < n_loc ? rp[row] : 0u, len = row < n_loc ? rp[row + 1] - beg : 0u;
    for (uint32_t j = 0; j < nchunk; j++) dst[(uint64_t)j * 32] = j < len ? col[beg + j] : 0xFFFFFFFFu;
  }
}


// ---- needed-columns exchange (multi-GPU) -------------------------------------------------------------------------------
// bitmap[c >> 5] bit (c & 31) = "some local row references column c" (new numbering, over the padded length)
__global__ void k_mark_cols(const uint32_t* __restrict__ col, uint64_t m, uint32_t* __restrict__ bitmap) {
  for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < m; i += (uint64_t)gridDim.x * blockDim.x) {
    const uint32_t c = col[i], bit = 1u << (c & 31);
    if (!(bitmap[c >> 5] & bit)) atomicOr(bitmap + (c >> 5), bit);
  }
}
// Does peer `r` (bitmap bm_r) reference local row l of rank `rank`?  Chunk-major numbering as in k_relabel.
struct NeedPred {
  const uint32_t* bm;
  uint64_t cl;
  uint32_t world, rank;
  __host__ __device__ bool operator()(uint32_t l) const {
    const uint64_t c = l / cl, g = c * (world * cl) + (uint64_t)rank * cl + (l - c * cl);
    return (bm[g >> 5] >> (g & 31)) & 1u;
  }
};
// counts[r] = number of local rows referenced by peer r   (grid.y = world)
__global__ void k_count_need(const uint32_t* __restrict__ bm_all, uint64_t words, uint64_t n_loc, uint64_t cl, uint32_t world, uint32_t rank,
                             unsigned long long* __restrict__ counts) {
  const uint32_t r = blockIdx.y;
  if (r == rank) return;
  const NeedPred pred{bm_all + (uint64_t)r * words, cl, world, rank};
  unsigned long long acc = 0;
  for (uint64_t l = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; l < n_loc; l += (uint64_t)gridDim.x * blockDim.x) acc += pred((uint32_t)l);
  for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
  if ((threadIdx.x & 31) == 0 && acc) atomicAdd(counts + r, acc);
}


inline unsigned grid_for(uint64_t items, unsigned block) { return (unsigned)((items + block - 1) / block); }

struct DevBuf {   // frees on scope exit unless released
  void* p = nullptr;
  ~DevBuf() { if (p) cudaFree(p); }
  template <class T> T* as() { return (T*)p; }
  void* release() { void* q = p; p = nullptr; return q; }
};

int bits_for(uint64_t v) { int b = 0; while ((1ull << b) < v && b < 63) b++; return b < 1 ? 1 : b; }

}  // namespace

void lz_free_graph(lz_ctx* c) {
  cudaFree(c->orig_ro); cudaFree(c->orig_ci); cudaFree(c->row_ptr); cudaFree(c->col); cudaFree(c->new2old); cudaFree(c->seg_store); cudaFree(c->sell_sp); cudaFree(c->sell_col);
  c->orig_ro = c->orig_ci = c->row_ptr = c->col = c->new2old = c->seg_store = c->sell_sp = c->sell_col = nullptr;
  c->n_long = c->n_items = 0; c->sell_entries = 0;
  c->ncolblk = 1;
  c->n = c->nnz = c->n_loc = c->nnz_loc = 0;
}

// Row bins: local rows are sorted by total length (non-increasing); bounds[t] = first row with len <= kThr[t].
// For each column block the lanes-per-row of a bin follow the bin's mean slice length in that block (any choice is
// correct — the kernel loops over longer slices — it only has to keep lanes busy and slices coalesced).
static const uint32_t kThr[7] = {128, 64, 32, 16, 8, 4, 2};
static void make_plans(const uint32_t* bounds, uint32_t n_loc, uint32_t nblk, const unsigned long long* bin_blk_nnz /* [8][nblk] */,
                       lz_spmv_plan* plans) {
  for (uint32_t blk = 0; blk < nblk; blk++) {
    lz_spmv_plan* plan = &plans[blk];
    uint32_t begin = 0, items = 0;
    plan->nbins = 0;
    for (int b = 0; b < 8; b++) {
      uint32_t end = (b < 7) ? bounds[b] : n_loc;
      if (end > begin) {
        const double mean = (double)bin_blk_nnz[b * nblk + blk] / (double)(end - begin);
        uint16_t lg, per;
        if (mean > 48.0) { lg = 5; per = 8; }
        else {
          per = 2;
          lg = 0;
          while (lg < 5 && (double)(2u << lg) < mean * 1.25) lg++;   // 2 * L >= 1.25 * mean slice length
        }
        lz_spmv_bin& bin = plan->bin[plan->nbins++];
        bin.row_begin = begin; bin.row_end = end; bin.log2_lanes = lg; bin.per_lane = per; bin.item_begin = items;
        const uint32_t rows_per_item = (LZ_SPMV_BLOCK >> lg) * LZ_SPMV_ROWS_PER_GROUP;
        items += (end - begin + rows_per_item - 1) / rows_per_item;
      }
      begin = end;
    }
    plan->nitems = items;
  }
}

// ---- ingest, in stages shared by the two sources of a graph ---------------------------------------------------------------
//   (1) a full original-order CSR on this device (lz_csr_upload, lz_graph_generate on one GPU)
//   (2) the counter-based generator, evaluated shard-wise on several GPUs (generate_sharded below): no rank ever holds more
//       than its own rows
// Both produce a degree array and then the keys (column block, local row, new column) of this rank's entries.
struct Order {
  DevBuf sorted_old, old2new;
  bool natural = false;
  uint64_t cl = 0, n_loc = 0, block_rows = 0, width = 0;
  uint32_t nblk = 1;
  int rowbits = 1;
};

__global__ void k_deg_from_ro(const uint32_t* __restrict__ ro, uint64_t n, uint32_t* __restrict__ deg) {
  uint64_t v = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (v < n) deg[v] = ro[v + 1] - ro[v];
}
__global__ void k_degree_keys_deg(const uint32_t* __restrict__ deg, uint64_t n, uint32_t* __restrict__ key, uint32_t* __restrict__ val) {
  uint64_t v = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (v >= n) return;
  key[v] = ~deg[v];
  val[v] = (uint32_t)v;
}
__global__ void k_local_lengths_deg(const uint32_t* __restrict__ sorted_old, const uint32_t* __restrict__ deg, uint64_t n, uint32_t world,
                                    uint32_t rank, uint64_t n_loc, uint64_t block_rows, uint32_t* __restrict__ len) {
  uint64_t l = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (l >= n_loc) return;
  uint64_t s = block_rows ? (uint64_t)rank * block_rows + l : l * world + rank;
  len[l] = s < n ? deg[sorted_old[s]] : 0u;
}
struct IsZero { __host__ __device__ uint64_t operator()(uint32_t d) const { return d == 0u ? 1ull : 0ull; } };
struct AsU64 { __host__ __device__ uint64_t operator()(uint32_t d) const { return (uint64_t)d; } };

// Stage 1-3: vertex order from the degrees, relabelling, local row pointer. `near` = stored entries within the locality radius
// of the diagonal (global). Sets n, nnz, max_degree, empty_rows, natural_order, chunk_rows, ncolblk, n_loc, nnz_loc, new2old, row_ptr.
static int make_order(lz_ctx* c, uint64_t n, uint64_t nnz, const uint32_t* deg_d, unsigned long long near, uint64_t radius, Order& o) {
  c->n = n; c->nnz = nnz;
  const uint32_t world = (uint32_t)c->world, rank = (uint32_t)c->rank;
  cudaStream_t st = c->stream;
  // 1. vertex order. Degree order (stable radix sort => ties keep ascending original id) by default; the natural order when
  //    the graph is band-like and not skewed (there the original numbering already has the locality that sorting would destroy).
  DevBuf key_in, key_out, val_in, len, tmp, cnt;
  LZ_CUDA(cudaMalloc(&key_in.p, n * 4)); LZ_CUDA(cudaMalloc(&key_out.p, n * 4));
  LZ_CUDA(cudaMalloc(&val_in.p, n * 4)); LZ_CUDA(cudaMalloc(&o.sorted_old.p, n * 4));
  k_degree_keys_deg<<<grid_for(n, 256), 256, 0, st>>>(deg_d, n, key_in.as<uint32_t>(), val_in.as<uint32_t>());
  size_t tb = 0;
  LZ_CUDA(cub::DeviceRadixSort::SortPairs(nullptr, tb, key_in.as<uint32_t>(), key_out.as<uint32_t>(), val_in.as<uint32_t>(),
                                          o.sorted_old.as<uint32_t>(), (int64_t)n, 0, 32, st));
  LZ_CUDA(cudaMalloc(&tmp.p, tb ? tb : 1));
  LZ_CUDA(cub::DeviceRadixSort::SortPairs(tmp.p, tb, key_in.as<uint32_t>(), key_out.as<uint32_t>(), val_in.as<uint32_t>(),
                                          o.sorted_old.as<uint32_t>(), (int64_t)n, 0, 32, st));
  uint32_t kfirst = 0;   // key = ~deg ascending: the first key belongs to the largest degree
  LZ_CUDA(cudaMemcpyAsync(&kfirst, key_out.p, 4, cudaMemcpyDeviceToHost, st));
  {  // isolated vertices
    size_t b5 = 0; DevBuf t5;
    LZ_CUDA(cudaMalloc(&cnt.p, 8));
    cub::TransformInputIterator<uint64_t, IsZero, const uint32_t*> it(deg_d, IsZero());
    LZ_CUDA(cub::DeviceReduce::Sum(nullptr, b5, it, cnt.as<uint64_t>(), (int64_t)n, st));
    LZ_CUDA(cudaMalloc(&t5.p, b5 ? b5 : 1));
    LZ_CUDA(cub::DeviceReduce::Sum(t5.p, b5, it, cnt.as<uint64_t>(), (int64_t)n, st));
    LZ_CUDA(cudaMemcpyAsync(&c->empty_rows, cnt.p, 8, cudaMemcpyDeviceToHost, st));
    LZ_CUDA(cudaStreamSynchronize(st));
  }
  c->max_degree = ~kfirst;
  const double avg_deg = (double)nnz / (double)n;
  bool natural = radius < n / 8 && c->max_degree <= LZ_SELL_LONG && (double)c->max_degree <= 8.0 * (avg_deg > 1.0 ? avg_deg : 1.0) &&
                 (double)near >= 0.5 * (double)nnz;
  if (const char* e = getenv("LZ_ORDER")) natural = (e[0] == 'n');
  c->natural_order = natural;
  o.natural = natural;

  // Rows per rank and column blocks. A column block (= chunk) is `cl` rows of every rank: a window of world * cl
  // entries of the gathered vector that one SpMV pass gathers from; it is sized to stay L2-resident (64 MiB measured
  // best on C3, profiles/), and for world > 1 it is also the unit of the pipelined exchange. With the natural order the
  // gathers are local anyway: a single block on any number of GPUs.
  uint64_t window = 64ull << 20;
  if (const char* e = getenv("LZ_SPMV_WINDOW_MB")) { long v = atol(e); if (v >= 1) window = (uint64_t)v << 20; }
  const uint64_t rows32 = (((n + world - 1) / world) + 31) & ~31ull;
  uint64_t cl = (window / 8 / world) & ~31ull;
  if (cl < 32) cl = 32;
  if (natural) cl = rows32;   // one block: the gathers are local, and the exchange sends only the referenced entries (lz_build_push_lists)
  if (const char* e = getenv("LZ_SPMV_COLBLOCKS")) { int v = atoi(e); if (v >= 1) cl = (((rows32 + v - 1) / v) + 31) & ~31ull; }
  if (cl > rows32) cl = rows32;
  uint32_t nblk = (uint32_t)((rows32 + cl - 1) / cl);
  if (nblk > LZ_MAX_COLBLK) { cl = (((rows32 + LZ_MAX_COLBLK - 1) / LZ_MAX_COLBLK) + 31) & ~31ull; nblk = (uint32_t)((rows32 + cl - 1) / cl); }
  while (nblk > 1 && 32 + bits_for((uint64_t)nblk * cl) + bits_for(nblk) > 64) { cl *= 2; nblk = (uint32_t)((rows32 + cl - 1) / cl); }
  const uint64_t n_loc = (uint64_t)nblk * cl, n_pad = n_loc * world;
  const uint64_t block_rows = natural ? n_loc : 0;   // natural order: rank r owns positions [r * n_loc, (r + 1) * n_loc)
  c->chunk_rows = cl;
  if (n_pad > 0xFFFFFFFEull) return lz_fail(LZ_ERR_ARG, "n = %llu too large for 32-bit vertex ids", (unsigned long long)n);
  c->n_loc = n_loc;
  c->ncolblk = nblk;
  o.cl = cl; o.n_loc = n_loc; o.block_rows = block_rows; o.nblk = nblk; o.rowbits = bits_for(n_loc); o.width = (uint64_t)world * cl;
  LZ_CUDA(cudaMalloc(&o.old2new.p, n * 4)); LZ_CUDA(cudaMalloc(&len.p, (n_loc + 1) * 4));
  LZ_CUDA(cudaMalloc((void**)&c->new2old, n_pad * 4));
  LZ_CUDA(cudaMalloc((void**)&c->row_ptr, (n_loc + 1) * 4));
  if (natural) k_iota_u32<<<grid_for(n, 256), 256, 0, st>>>(o.sorted_old.as<uint32_t>(), n);

  // 2. relabel
  k_fill_u32<<<grid_for(n_pad, 256), 256, 0, st>>>(c->new2old, n_pad, 0xFFFFFFFFu);
  k_relabel<<<grid_for(n, 256), 256, 0, st>>>(o.sorted_old.as<uint32_t>(), n, world, cl, block_rows, o.old2new.as<uint32_t>(), c->new2old);

  // 3. local row pointer (total row lengths)
  k_local_lengths_deg<<<grid_for(n_loc, 256), 256, 0, st>>>(o.sorted_old.as<uint32_t>(), deg_d, n, world, rank, n_loc, block_rows, len.as<uint32_t>());
  LZ_CUDA(cudaMemsetAsync(len.as<uint32_t>() + n_loc, 0, 4, st));
  {
    DevBuf t2; size_t b2 = 0;
    LZ_CUDA(cub::DeviceScan::ExclusiveSum(nullptr, b2, len.as<uint32_t>(), c->row_ptr, (int64_t)(n_loc + 1), st));
    LZ_CUDA(cudaMalloc(&t2.p, b2 ? b2 : 1));
    LZ_CUDA(cub::DeviceScan::ExclusiveSum(t2.p, b2, len.as<uint32_t>(), c->row_ptr, (int64_t)(n_loc + 1), st));
  }
  {
    // the scan is 32-bit: guard against wrap-around by summing lengths in 64 bit
    DevBuf t3, s64; size_t b3 = 0;
    LZ_CUDA(cudaMalloc(&s64.p, 8));
    cub::TransformInputIterator<uint64_t, AsU64, const uint32_t*> it(len.as<uint32_t>(), AsU64());
    LZ_CUDA(cub::DeviceReduce::Sum(nullptr, b3, it, s64.as<uint64_t>(), (int64_t)n_loc, st));
    LZ_CUDA(cudaMalloc(&t3.p, b3 ? b3 : 1));
    LZ_CUDA(cub::DeviceReduce::Sum(t3.p, b3, it, s64.as<uint64_t>(), (int64_t)n_loc, st));
    uint64_t total = 0;
    LZ_CUDA(cudaMemcpyAsync(&total, s64.p, 8, cudaMemcpyDeviceToHost, st));
    LZ_CUDA(cudaStreamSynchronize(st));
    if (total > 0xFFFFFFFFull) return lz_fail(LZ_ERR_ARG, "local nnz %llu does not fit 32-bit row offsets", (unsigned long long)total);
    c->nnz_loc = total;
  }
  return LZ_OK;
}

// Stage 5-7: sort this rank's keys (column-block-major, row-major, ascending column), optionally dropping duplicates (generator
// candidates), then the per-block row pointers, the CSR launch plans and the sliced layout.
static int finish_local(lz_ctx* c, const Order& o, DevBuf& k_in, uint64_t nkeys, bool dedupe) {
  cudaStream_t st = c->stream;
  const uint64_t n_loc = o.n_loc;
  const uint32_t nblk = o.nblk;
  const int rowbits = o.rowbits;
  const bool natural = o.natural;
  {
    DevBuf k_out, t4; size_t b4 = 0;
    const uint64_t m = c->nnz_loc;
    LZ_CUDA(cudaMalloc(&k_out.p, (nkeys ? nkeys : 1) * 8));
    LZ_CUDA(cudaMalloc((void**)&c->col, (m ? m : 1) * 4));
    LZ_CUDA(cudaMalloc((void**)&c->seg_store, (uint64_t)nblk * (n_loc + 1) * 4));
    const uint64_t* sorted = k_out.as<uint64_t>();
    if (nkeys) {
      int end_bit = 32 + rowbits + (nblk > 1 ? bits_for(nblk) : 0);
      if (end_bit > 64) end_bit = 64;
      LZ_CUDA(cub::DeviceRadixSort::SortKeys(nullptr, b4, k_in.as<uint64_t>(), k_out.as<uint64_t>(), (int64_t)nkeys, 0, end_bit, st));
      LZ_CUDA(cudaMalloc(&t4.p, b4 ? b4 : 1));
      LZ_CUDA(cub::DeviceRadixSort::SortKeys(t4.p, b4, k_in.as<uint64_t>(), k_out.as<uint64_t>(), (int64_t)nkeys, 0, end_bit, st));
      if (dedupe) {
        DevBuf nsel, tu; size_t ub = 0;
        LZ_CUDA(cudaMalloc(&nsel.p, 8));
        LZ_CUDA(cub::DeviceSelect::Unique(nullptr, ub, k_out.as<uint64_t>(), k_in.as<uint64_t>(), nsel.as<int64_t>(), (int64_t)nkeys, st));
        LZ_CUDA(cudaMalloc(&tu.p, ub ? ub : 1));
        LZ_CUDA(cub::DeviceSelect::Unique(tu.p, ub, k_out.as<uint64_t>(), k_in.as<uint64_t>(), nsel.as<int64_t>(), (int64_t)nkeys, st));
        int64_t nu = 0;
        LZ_CUDA(cudaMemcpyAsync(&nu, nsel.p, 8, cudaMemcpyDeviceToHost, st));
        LZ_CUDA(cudaStreamSynchronize(st));
        if ((uint64_t)nu != m)
          return lz_fail(LZ_ERR_ARG, "sharded graph construction is inconsistent: %lld distinct local entries, degrees say %llu", (long long)nu,
                         (unsigned long long)m);
        sorted = k_in.as<uint64_t>();
      } else if (nkeys != m) {
        return lz_fail(LZ_ERR_ARG, "local key count %llu != local nnz %llu", (unsigned long long)nkeys, (unsigned long long)m);
      }
      if (m) k_low32<<<grid_for(m, 256), 256, 0, st>>>(sorted, m, c->col);
    }
    k_block_row_ptr<<<grid_for((uint64_t)nblk * (n_loc + 1), 256), 256, 0, st>>>(sorted, m, n_loc, nblk, rowbits, c->seg_store);
    LZ_CUDA(cudaStreamSynchronize(st));
    for (uint32_t b = 0; b < nblk; b++) c->seg[b] = c->seg_store + (uint64_t)b * (n_loc + 1);
    c->seg[nblk] = nullptr;
  }

  // 6. SpMV plans
  {
    DevBuf thr_d, out_d, segp_d, binrows_d, cnt_d;
    uint32_t out_h[7];
    LZ_CUDA(cudaMalloc(&thr_d.p, sizeof(kThr))); LZ_CUDA(cudaMalloc(&out_d.p, sizeof(out_h)));
    LZ_CUDA(cudaMemcpyAsync(thr_d.p, kThr, sizeof(kThr), cudaMemcpyHostToDevice, st));
    k_bin_bounds<<<1, 32, 0, st>>>(c->row_ptr, (uint32_t)n_loc, thr_d.as<uint32_t>(), 7, out_d.as<uint32_t>());
    LZ_CUDA(cudaMemcpyAsync(out_h, out_d.p, sizeof(out_h), cudaMemcpyDeviceToHost, st));
    LZ_CUDA(cudaStreamSynchronize(st));
    if (natural) for (int b = 0; b < 7; b++) out_h[b] = 0;   // rows are not length-sorted: one bin, lanes from the mean length
    uint32_t bin_rows[9];
    bin_rows[0] = 0;
    for (int b = 0; b < 7; b++) bin_rows[b + 1] = out_h[b];
    bin_rows[8] = (uint32_t)n_loc;
    std::vector<unsigned long long> cnt_h(8 * nblk);
    LZ_CUDA(cudaMalloc(&segp_d.p, sizeof(uint32_t*) * (nblk + 1))); LZ_CUDA(cudaMalloc(&binrows_d.p, sizeof(bin_rows)));
    LZ_CUDA(cudaMalloc(&cnt_d.p, 8 * nblk * sizeof(unsigned long long)));
    LZ_CUDA(cudaMemcpyAsync(segp_d.p, c->seg, sizeof(uint32_t*) * (nblk + 1), cudaMemcpyHostToDevice, st));   // synchronous w.r.t. host memory: pageable source
    LZ_CUDA(cudaMemcpyAsync(binrows_d.p, bin_rows, sizeof(bin_rows), cudaMemcpyHostToDevice, st));
    k_bin_block_nnz<<<dim3(8, nblk), 256, 0, st>>>((const uint32_t* const*)segp_d.p, binrows_d.as<uint32_t>(), nblk,
                                                    (unsigned long long*)cnt_d.p);
    LZ_CUDA(cudaMemcpyAsync(cnt_h.data(), cnt_d.p, 8 * nblk * sizeof(unsigned long long), cudaMemcpyDeviceToHost, st));
    LZ_CUDA(cudaStreamSynchronize(st));
    make_plans(out_h, (uint32_t)n_loc, nblk, cnt_h.data(), c->plan_auto);
    // warp-per-row for everything
    c->plan_warp.nbins = 1;
    c->plan_warp.bin[0] = {0u, (uint32_t)n_loc, (uint16_t)5, (uint16_t)2, 0u};
    {
      const uint32_t rows_per_item = (LZ_SPMV_BLOCK >> 5) * LZ_SPMV_ROWS_PER_GROUP;
      c->plan_warp.nitems = (uint32_t)((n_loc + rows_per_item - 1) / rows_per_item);
    }
  }
  // 7. sliced layout for the default SpMV
  {
    uint32_t n_long = 0;   // rows with total length > LZ_SELL_LONG (lengths are non-increasing): binary search on the device row_ptr
    {
      DevBuf thr_d, out_d;
      const uint32_t thr = LZ_SELL_LONG;
      LZ_CUDA(cudaMalloc(&thr_d.p, 4)); LZ_CUDA(cudaMalloc(&out_d.p, 4));
      LZ_CUDA(cudaMemcpyAsync(thr_d.p, &thr, 4, cudaMemcpyHostToDevice, st));
      k_bin_bounds<<<1, 32, 0, st>>>(c->row_ptr, (uint32_t)n_loc, thr_d.as<uint32_t>(), 1, out_d.as<uint32_t>());
      LZ_CUDA(cudaMemcpyAsync(&n_long, out_d.p, 4, cudaMemcpyDeviceToHost, st));
      LZ_CUDA(cudaStreamSynchronize(st));
      if (natural) n_long = 0;   // not length-sorted; all rows go through the 32-row slices
    }
    const uint32_t n_items = n_long + (uint32_t)((n_loc - n_long + 31) / 32);
    const uint64_t tot_items = (uint64_t)nblk * n_items;
    c->n_long = n_long; c->n_items = n_items;
    DevBuf widths, segp_d, t7, last2;
    size_t b7 = 0;
    LZ_CUDA(cudaMalloc(&widths.p, (tot_items + 1) * 4));
    LZ_CUDA(cudaMalloc((void**)&c->sell_sp, (tot_items + 1) * 4));
    LZ_CUDA(cudaMalloc(&segp_d.p, sizeof(uint32_t*) * (nblk + 1)));
    LZ_CUDA(cudaMemcpy(segp_d.p, c->seg, sizeof(uint32_t*) * (nblk + 1), cudaMemcpyHostToDevice));
    LZ_CUDA(cudaMemsetAsync(widths.as<uint32_t>() + tot_items, 0, 4, st));
    k_sell_widths<<<grid_for(tot_items * 32, 256), 256, 0, st>>>((const uint32_t* const*)segp_d.p, nblk, n_long, n_items, (uint32_t)n_loc,
                                                                  widths.as<uint32_t>());
    LZ_CUDA(cub::DeviceScan::ExclusiveSum(nullptr, b7, widths.as<uint32_t>(), c->sell_sp, (int64_t)(tot_items + 1), st));
    LZ_CUDA(cudaMalloc(&t7.p, b7 ? b7 : 1));
    LZ_CUDA(cub::DeviceScan::ExclusiveSum(t7.p, b7, widths.as<uint32_t>(), c->sell_sp, (int64_t)(tot_items + 1), st));
    uint32_t total_chunks = 0;
    LZ_CUDA(cudaMemcpyAsync(&total_chunks, c->sell_sp + tot_items, 4, cudaMemcpyDeviceToHost, st));
    LZ_CUDA(cudaStreamSynchronize(st));
    c->sell_entries = (uint64_t)total_chunks * 32;
    {  // Batched-quad instantiation for natural-order blocks with narrow slices (HBM-bound, gathers hit L1: more loads in flight
       // pay: banded 2^26 SpMV 0.558 -> 0.489 ms). Not for the cold column block of a degree-sorted graph, which is bound by the
       // L1-miss request rate and loses from the lower occupancy (C3: 1.194 -> 1.234 ms per SpMV when it was tried).
      int force = -1;
      if (const char* e = getenv("LZ_SELL_NARROW")) force = atoi(e) != 0;
      for (uint32_t b = 0; b < nblk; b++) {
        uint32_t lo = 0, hi = 0;
        LZ_CUDA(cudaMemcpy(&lo, c->sell_sp + (uint64_t)b * n_items + n_long, 4, cudaMemcpyDeviceToHost));
        LZ_CUDA(cudaMemcpy(&hi, c->sell_sp + (uint64_t)(b + 1) * n_items, 4, cudaMemcpyDeviceToHost));
        const double slices = (double)(n_items - n_long);
        c->sell_narrow[b] = force >= 0 ? force != 0 : (natural && slices > 0 && (double)(hi - lo) / slices <= 6.0);
      }
    }
    // 32-bit chunk counter wrapped, or absurd padding. The first slice of a block may be as wide as a row of LZ_SELL_LONG entries (a star
    // K_{1,100}: 3296 entries for 200 non-zeros), so that much padding per block is always allowed.
    if (c->sell_entries > 6 * c->nnz_loc + 64 * (uint64_t)tot_items + 1024 + 32ull * LZ_SELL_LONG * nblk)
      return lz_fail(LZ_ERR_ARG, "sliced layout too large (%llu entries for %llu non-zeros)", (unsigned long long)c->sell_entries,
                     (unsigned long long)c->nnz_loc);
    LZ_CUDA(cudaMalloc((void**)&c->sell_col, (c->sell_entries ? c->sell_entries : 1) * 4));
    k_sell_fill<<<grid_for(tot_items * 32, 256), 256, 0, st>>>((const uint32_t* const*)segp_d.p, c->col, c->sell_sp, nblk, n_long, n_items,
                                                                (uint32_t)n_loc, c->sell_col);
    LZ_CUDA(cudaStreamSynchronize(st));
  }
  LZ_CUDA(cudaGetLastError());
  return LZ_OK;
}

// Takes ownership of ro_d / ci_d (original-order CSR on the device).
int lz_ingest_device_csr(lz_ctx* c, uint64_t n, uint64_t nnz, uint32_t* ro_d, uint32_t* ci_d) {
  lz_free_graph(c);
  c->epoch++;   // any cached CUDA graph of the step loop refers to the old matrix
  c->graph_id++;
  c->orig_ro = ro_d; c->orig_ci = ci_d;
  const uint32_t world = (uint32_t)c->world, rank = (uint32_t)c->rank;
  cudaStream_t st = c->stream;
  DevBuf deg, loc_d;
  LZ_CUDA(cudaMalloc(&deg.p, n * 4)); LZ_CUDA(cudaMalloc(&loc_d.p, 8));
  k_deg_from_ro<<<grid_for(n, 256), 256, 0, st>>>(ro_d, n, deg.as<uint32_t>());
  unsigned long long near = 0;
  const uint64_t radius = (n / 256 > 65536) ? n / 256 : 65536;
  LZ_CUDA(cudaMemsetAsync(loc_d.p, 0, 8, st));
  k_locality<<<(unsigned)c->sm_count * 8, 256, 0, st>>>(ro_d, ci_d, n, radius, (unsigned long long*)loc_d.p);
  LZ_CUDA(cudaMemcpyAsync(&near, loc_d.p, 8, cudaMemcpyDeviceToHost, st));
  LZ_CUDA(cudaStreamSynchronize(st));
  Order o;
  LZ_TRY(make_order(c, n, nnz, deg.as<uint32_t>(), near, radius, o));
  // 5. local column lists in the new numbering: one key per stored entry of this rank's rows
  DevBuf k_in;
  const uint64_t m = c->nnz_loc;
  LZ_CUDA(cudaMalloc(&k_in.p, (m ? m : 1) * 8));
  if (m)
    k_local_keys<<<grid_for(o.n_loc * 32, 256), 256, 0, st>>>(o.sorted_old.as<uint32_t>(), ro_d, ci_d, o.old2new.as<uint32_t>(), c->row_ptr, n,
                                                               world, rank, o.n_loc, o.block_rows, o.width, o.rowbits, k_in.as<uint64_t>());
  LZ_TRY(finish_local(c, o, k_in, m, false));
  // The original-order CSR only serves lz_csr_download (a test / oracle hook). On several GPUs it is dead weight on every rank
  // (C4: 9.1 GB per GPU): dropped unless LZ_KEEP_CSR=1 asks for it. One GPU keeps it (LZ_KEEP_CSR=0 drops it there too).
  bool keep = c->world == 1;
  if (const char* e = getenv("LZ_KEEP_CSR")) keep = atoi(e) != 0;
  if (!keep) {
    cudaFree(c->orig_ro); cudaFree(c->orig_ci);
    c->orig_ro = c->orig_ci = nullptr;
  }
  return LZ_OK;
}

// ---- sharded construction of a generated graph (several GPUs) ---------------------------------------------------------------
// The generators are pure functions of the candidate index, so no rank needs the whole graph:
//   A. every rank scans all candidates and keeps the oriented entries whose ORIGINAL row lies in its slice of [0, n): sort +
//      unique gives the degrees of that slice; the slices are all-gathered (4 n bytes), as is the locality count.
//   B. every rank derives the same vertex order and relabelling from the degree array (make_order).
//   C. every rank scans the candidates again and keeps the oriented entries whose row it OWNS in the new numbering, directly as
//      (column block, local row, new column) keys; sort + unique must leave exactly the number of entries the degrees promise.
// Work and memory per rank are O(nnz / world + n) (plus two cheap scans of the candidate space); the reference builds the
// whole matrix in a std::set on one host thread (adjMatrix.cc:21-46).
struct SelRange {      // phase A: original row in [lo, hi)
  uint32_t lo, hi;
  __device__ bool operator()(uint32_t r, uint32_t cidx, uint64_t* key) const {
    if (r < lo || r >= hi) return false;
    *key = ((uint64_t)r << 32) | cidx;
    return true;
  }
};
struct SelOwner {      // phase C: row owned by this rank in the new numbering (chunk-major ids, see k_relabel)
  const uint32_t* old2new;
  uint64_t cl, width;
  uint32_t world, rank;
  int rowbits;
  __device__ bool operator()(uint32_t r, uint32_t cidx, uint64_t* key) const {
    const uint64_t nr = old2new[r];
    const uint64_t ch = nr / width, rem = nr - ch * width;
    if (rem / cl != rank) return false;
    const uint64_t l = ch * cl + (rem - (uint64_t)rank * cl);
    const uint64_t nc = old2new[cidx];
    *key = ((nc / width) << (32 + rowbits)) | (l << 32) | nc;
    return true;
  }
};
template <class Sel>
__global__ void __launch_bounds__(256) k_gen_select(lz_gen_params p, Sel sel, uint64_t* __restrict__ out, unsigned long long* __restrict__ cursor) {
  const uint32_t lane = threadIdx.x & 31;
  const uint64_t total = (p.m + 1 + 31) & ~31ull;      // whole warps stay converged for the ballots
  for (uint64_t e = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (uint64_t)gridDim.x * blockDim.x) {
    uint32_t u = 0, v = 0;
    if (e <= p.m) lz_gen_edge(p, e, &u, &v);
    const bool edge = e <= p.m && u != v;
#pragma unroll
    for (int orient = 0; orient < 2; orient++) {
      uint64_t key = 0;
      const bool take = edge && sel(orient ? v : u, orient ? u : v, &key);
      const unsigned mask = __ballot_sync(0xffffffffu, take);
      if (!mask) continue;
      const int leader = __ffs(mask) - 1;
      unsigned long long base = 0;
      if ((int)lane == leader) base = atomicAdd(cursor, (unsigned long long)__popc(mask));
      base = __shfl_sync(0xffffffffu, base, leader);
      if (take && out) out[base + __popc(mask & ((1u << lane) - 1u))] = key;
    }
  }
}
// deg[i] = number of (sorted, unique) keys with row lo + i, i < rows
__global__ void k_range_degrees(const uint64_t* __restrict__ keys, uint64_t nkeys, uint32_t lo, uint32_t rows, uint32_t n, uint32_t* __restrict__ deg) {
  const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= rows) return;
  const uint64_t r = (uint64_t)lo + i;
  if (r >= n) { deg[i] = 0u; return; }
  auto lower = [&](uint64_t target) {
    uint64_t a = 0, b = nkeys;
    while (a < b) { const uint64_t mid = (a + b) >> 1; if (keys[mid] < target) a = mid + 1; else b = mid; }
    return a;
  };
  deg[i] = (uint32_t)(lower((r + 1) << 32) - lower(r << 32));
}
__global__ void k_locality_keys(const uint64_t* __restrict__ keys, uint64_t nkeys, uint64_t radius, unsigned long long* __restrict__ out) {
  unsigned long long acc = 0;
  for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < nkeys; i += (uint64_t)gridDim.x * blockDim.x) {
    const uint64_t r = keys[i] >> 32, cc = keys[i] & 0xFFFFFFFFull;
    acc += (cc > r ? cc - r : r - cc) <= radius;
  }
  for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
  if ((threadIdx.x & 31) == 0 && acc) atomicAdd(out, acc);
}

template <class Sel>
static int gen_select(lz_ctx* c, const lz_gen_params& p, const Sel& sel, DevBuf& keys, uint64_t* nkeys_out) {
  cudaStream_t st = c->stream;
  DevBuf cur;
  LZ_CUDA(cudaMalloc(&cur.p, 8));
  const unsigned grid = (unsigned)c->sm_count * 16;
  unsigned long long cnt = 0;
  LZ_CUDA(cudaMemsetAsync(cur.p, 0, 8, st));
  k_gen_select<Sel><<<grid, 256, 0, st>>>(p, sel, nullptr, (unsigned long long*)cur.p);          // count
  LZ_CUDA(cudaMemcpyAsync(&cnt, cur.p, 8, cudaMemcpyDeviceToHost, st));
  LZ_CUDA(cudaStreamSynchronize(st));
  if (cudaMalloc(&keys.p, (cnt ? cnt : 1) * 8) != cudaSuccess) { cudaGetLastError(); return lz_fail(LZ_ERR_ALLOC, "cannot allocate %llu shard keys", cnt); }
  LZ_CUDA(cudaMemsetAsync(cur.p, 0, 8, st));
  k_gen_select<Sel><<<grid, 256, 0, st>>>(p, sel, keys.as<uint64_t>(), (unsigned long long*)cur.p);   // emit (order irrelevant: sorted next)
  LZ_CUDA(cudaStreamSynchronize(st));
  *nkeys_out = cnt;
  return LZ_OK;
}

static int generate_sharded(lz_ctx* c, const lz_gen_params& p) {
  lz_free_graph(c);
  c->epoch++;
  c->graph_id++;
  cudaStream_t st = c->stream;
  const uint32_t world = (uint32_t)c->world, rank = (uint32_t)c->rank;
  const uint64_t n = p.n;
  const uint64_t rows_per = (n + world - 1) / world;
  const uint64_t lo = (uint64_t)rank * rows_per, hi = lo + rows_per < n ? lo + rows_per : n;
  DevBuf deg_all, near_d;
  LZ_CUDA(cudaMalloc(&deg_all.p, rows_per * world * 4));
  LZ_CUDA(cudaMalloc(&near_d.p, 16));
  LZ_CUDA(cudaMemsetAsync(near_d.p, 0, 16, st));
  const uint64_t radius = (n / 256 > 65536) ? n / 256 : 65536;
  {  // A. degrees of my slice of the original numbering
    DevBuf ka, kb, tmp, nsel;
    uint64_t na = 0;
    LZ_TRY(gen_select(c, p, SelRange{(uint32_t)(lo < n ? lo : n), (uint32_t)hi}, ka, &na));
    LZ_CUDA(cudaMalloc(&kb.p, (na ? na : 1) * 8)); LZ_CUDA(cudaMalloc(&nsel.p, 8));
    int64_t nu = 0;
    if (na) {
      size_t tb = 0, ub = 0;
      LZ_CUDA(cub::DeviceRadixSort::SortKeys(nullptr, tb, ka.as<uint64_t>(), kb.as<uint64_t>(), (int64_t)na, 0, 64, st));
      LZ_CUDA(cub::DeviceSelect::Unique(nullptr, ub, kb.as<uint64_t>(), ka.as<uint64_t>(), nsel.as<int64_t>(), (int64_t)na, st));
      LZ_CUDA(cudaMalloc(&tmp.p, (tb > ub ? tb : ub) + 1));
      LZ_CUDA(cub::DeviceRadixSort::SortKeys(tmp.p, tb, ka.as<uint64_t>(), kb.as<uint64_t>(), (int64_t)na, 0, 64, st));
      LZ_CUDA(cub::DeviceSelect::Unique(tmp.p, ub, kb.as<uint64_t>(), ka.as<uint64_t>(), nsel.as<int64_t>(), (int64_t)na, st));
      LZ_CUDA(cudaMemcpyAsync(&nu, nsel.p, 8, cudaMemcpyDeviceToHost, st));
      LZ_CUDA(cudaStreamSynchronize(st));
    }
    uint32_t* mine = deg_all.as<uint32_t>() + (uint64_t)rank * rows_per;
    k_range_degrees<<<grid_for(rows_per, 256), 256, 0, st>>>(ka.as<uint64_t>(), (uint64_t)nu, (uint32_t)lo, (uint32_t)rows_per, (uint32_t)n, mine);
    if (nu) k_locality_keys<<<(unsigned)c->sm_count * 8, 256, 0, st>>>(ka.as<uint64_t>(), (uint64_t)nu, radius, (unsigned long long*)near_d.p);
    LZ_NCCL(lz_nccl()->AllGather(mine, deg_all.p, rows_per, ncclUint32, c->comm, st));
    LZ_NCCL(lz_nccl()->AllReduce(near_d.p, near_d.p, 1, ncclUint64, ncclSum, c->comm, st));
    LZ_CUDA(cudaStreamSynchronize(st));
  }
  unsigned long long near = 0;
  LZ_CUDA(cudaMemcpy(&near, near_d.p, 8, cudaMemcpyDeviceToHost));
  uint64_t nnz = 0;
  {
    DevBuf s64, t3; size_t b3 = 0;
    LZ_CUDA(cudaMalloc(&s64.p, 8));
    cub::TransformInputIterator<uint64_t, AsU64, const uint32_t*> it(deg_all.as<uint32_t>(), AsU64());
    LZ_CUDA(cub::DeviceReduce::Sum(nullptr, b3, it, s64.as<uint64_t>(), (int64_t)n, st));
    LZ_CUDA(cudaMalloc(&t3.p, b3 ? b3 : 1));
    LZ_CUDA(cub::DeviceReduce::Sum(t3.p, b3, it, s64.as<uint64_t>(), (int64_t)n, st));
    LZ_CUDA(cudaMemcpyAsync(&nnz, s64.p, 8, cudaMemcpyDeviceToHost, st));
    LZ_CUDA(cudaStreamSynchronize(st));
  }
  // B. the same order on every rank
  Order o;
  LZ_TRY(make_order(c, n, nnz, deg_all.as<uint32_t>(), near, radius, o));
  cudaFree(deg_all.release());
  // C. my rows, straight in the final key form
  DevBuf kc;
  uint64_t nc = 0;
  LZ_TRY(gen_select(c, p, SelOwner{o.old2new.as<uint32_t>(), o.cl, o.width, world, rank, o.rowbits}, kc, &nc));
  return finish_local(c, o, kc, nc, true);
}

// Needed-columns exchange (SURVEY 8f-2), set up once per graph/vector allocation; collective over the NCCL communicator.
// Every rank marks the columns its rows reference, the bitmaps are all-gathered, and each rank derives, per peer, the
// ascending list of its own rows that the peer gathers from. When those lists are short (band-like / mesh-like graphs in
// natural order: a halo plus a few chords) the Krylov vector is exchanged entry by entry over NVLink instead of in full
// (k_scale_push_sparse); for graphs whose ranks reference most of each other's rows (R-MAT) the dense push stays.
// The reference's two-card split copies the whole half vector every step (parallel-two-cards/lib/cu_lanczos.cu:116-165).
int lz_build_push_lists(lz_ctx* c) {
  cudaFree(c->push_list); c->push_list = nullptr;
  c->sparse_push = false;
  c->push_graph_id = c->graph_id;
  for (int r = 0; r <= LZ_MAX_WORLD; r++) c->push_off[r] = 0;
  if (c->world == 1 || !c->peer_push) return LZ_OK;
  int force = -1;
  if (const char* e = getenv("LZ_SPARSE_PUSH")) force = atoi(e) != 0;
  cudaStream_t st = c->stream;
  const uint32_t world = (uint32_t)c->world, rank = (uint32_t)c->rank;
  const uint64_t n_pad = c->n_loc * (uint64_t)world, words = (n_pad + 31) / 32;
  DevBuf bm, cnt_d;
  LZ_CUDA(cudaMalloc(&bm.p, words * 4 * world));
  LZ_CUDA(cudaMalloc(&cnt_d.p, sizeof(unsigned long long) * (LZ_MAX_WORLD + 1)));
  uint32_t* mine = bm.as<uint32_t>() + (uint64_t)rank * words;
  LZ_CUDA(cudaMemsetAsync(mine, 0, words * 4, st));
  LZ_CUDA(cudaMemsetAsync(cnt_d.p, 0, sizeof(unsigned long long) * (LZ_MAX_WORLD + 1), st));
  if (c->nnz_loc) k_mark_cols<<<(unsigned)c->sm_count * 8, 256, 0, st>>>(c->col, c->nnz_loc, mine);
  LZ_NCCL(lz_nccl()->AllGather(mine, bm.p, words, ncclUint32, c->comm, st));
  k_count_need<<<dim3((unsigned)c->sm_count * 2, world), 256, 0, st>>>(bm.as<uint32_t>(), words, c->n_loc, c->chunk_rows, world, rank,
                                                                        (unsigned long long*)cnt_d.p);
  unsigned long long cnt_h[LZ_MAX_WORLD + 1] = {};
  LZ_CUDA(cudaMemcpyAsync(cnt_h, cnt_d.p, sizeof(unsigned long long) * world, cudaMemcpyDeviceToHost, st));
  LZ_CUDA(cudaStreamSynchronize(st));
  unsigned long long total = 0;
  for (uint32_t r = 0; r < world; r++) total += cnt_h[r];
  // the decision must be the same on every rank: compare the global volume with the dense one
  double tot_d = (double)total;
  double* buf = c->scal + 10;
  LZ_CUDA(cudaMemcpyAsync(buf, &tot_d, 8, cudaMemcpyHostToDevice, st));
  LZ_NCCL(lz_nccl()->AllReduce(buf, buf, 1, ncclDouble, ncclSum, c->comm, st));
  LZ_CUDA(cudaMemcpyAsync(&tot_d, buf, 8, cudaMemcpyDeviceToHost, st));
  LZ_CUDA(cudaStreamSynchronize(st));
  const double dense = (double)world * (double)(world - 1) * (double)c->n_loc;
  const bool sparse = force >= 0 ? force != 0 : tot_d < 0.5 * dense;
  c->push_need_frac = dense > 0 ? tot_d / dense : 1.0;
  if (!sparse) return LZ_OK;
  if (total > 0xFFFFFFF0ull) return LZ_OK;   // offsets are 32-bit; such a graph is dense anyway
  LZ_CUDA(cudaMalloc((void**)&c->push_list, (total ? total : 1) * 4));
  DevBuf nsel, tmp;
  LZ_CUDA(cudaMalloc(&nsel.p, 8));
  size_t tb = 0;
  cub::CountingInputIterator<uint32_t> it(0u);
  LZ_CUDA(cub::DeviceSelect::If(nullptr, tb, it, c->push_list, nsel.as<int64_t>(), (int64_t)c->n_loc, NeedPred{bm.as<uint32_t>(), c->chunk_rows, world, rank}, st));
  LZ_CUDA(cudaMalloc(&tmp.p, tb ? tb : 1));
  uint64_t off = 0;
  for (uint32_t r = 0; r < world; r++) {
    c->push_off[r] = (uint32_t)off;
    if (r == rank || cnt_h[r] == 0) continue;
    LZ_CUDA(cub::DeviceSelect::If(tmp.p, tb, it, c->push_list + off, nsel.as<int64_t>(), (int64_t)c->n_loc,
                                  NeedPred{bm.as<uint32_t>() + (uint64_t)r * words, c->chunk_rows, world, rank}, st));
    off += cnt_h[r];
  }
  for (uint32_t r = world; r <= LZ_MAX_WORLD; r++) c->push_off[r] = (uint32_t)off;
  LZ_CUDA(cudaStreamSynchronize(st));
  c->sparse_push = true;
  return LZ_OK;
}

extern "C" int lz_csr_upload(lz_ctx* c, uint64_t n, const uint32_t* row_offset, const uint32_t* col_idx) {
  if (!c || !row_offset || !col_idx || n == 0) return lz_fail(LZ_ERR_ARG, "lz_csr_upload: null argument or n == 0");
  LZ_CUDA(cudaSetDevice(c->device));
  uint64_t nnz = row_offset[n];
  uint32_t *ro_d = nullptr, *ci_d = nullptr;
  LZ_CUDA(cudaMalloc((void**)&ro_d, (n + 1) * 4));
  if (cudaMalloc((void**)&ci_d, (nnz ? nnz : 1) * 4) != cudaSuccess) { cudaFree(ro_d); return lz_fail(LZ_ERR_ALLOC, "device allocation of col_idx failed"); }
  // the three H2D copies of cu_lanczos.cu:88-90, minus the vector
  cudaError_t e1 = cudaMemcpyAsync(ro_d, row_offset, (n + 1) * 4, cudaMemcpyHostToDevice, c->stream);
  cudaError_t e2 = cudaMemcpyAsync(ci_d, col_idx, nnz * 4, cudaMemcpyHostToDevice, c->stream);
  if (e1 != cudaSuccess || e2 != cudaSuccess) { cudaFree(ro_d); cudaFree(ci_d); return lz_fail(LZ_ERR_CUDA, "H2D copy of CSR failed"); }
  c->have_x = c->have_tridiag = c->have_coef = c->have_ans = false;
  return lz_ingest_device_csr(c, n, nnz, ro_d, ci_d);
}

extern "C" int lz_graph_generate(lz_ctx* c, const lz_graph_spec* spec) {
  if (!c || !spec) return lz_fail(LZ_ERR_ARG, "lz_graph_generate: null argument");
  LZ_CUDA(cudaSetDevice(c->device));
  lz_gen_params p;
  if (lz_gen_prepare(spec, &p)) return lz_fail(LZ_ERR_ARG, "bad graph spec (kind %u)", spec->kind);
  cudaStream_t st = c->stream;
  bool sharded = c->world > 1;
  if (const char* e = getenv("LZ_KEEP_CSR")) if (atoi(e) != 0) sharded = false;      // the full CSR is wanted back (lz_csr_download)
  if (const char* e = getenv("LZ_SHARDED_INGEST")) sharded = c->world > 1 && atoi(e) != 0;
  if (sharded) {
    c->have_x = c->have_tridiag = c->have_coef = c->have_ans = false;
    return generate_sharded(c, p);
  }
  const uint64_t nkeys = 2 * (p.m + 1);
  DevBuf k_in, k_out, tmp, nsel;
  LZ_CUDA(cudaMalloc(&k_in.p, nkeys * 8)); LZ_CUDA(cudaMalloc(&k_out.p, nkeys * 8)); LZ_CUDA(cudaMalloc(&nsel.p, 8));
  k_gen_keys<<<grid_for(p.m + 1, 256), 256, 0, st>>>(p, k_in.as<uint64_t>());
  size_t tb = 0;
  int end_bit = 64;   // sentinel uses all bits
  LZ_CUDA(cub::DeviceRadixSort::SortKeys(nullptr, tb, k_in.as<uint64_t>(), k_out.as<uint64_t>(), (int64_t)nkeys, 0, end_bit, st));
  LZ_CUDA(cudaMalloc(&tmp.p, tb ? tb : 1));
  LZ_CUDA(cub::DeviceRadixSort::SortKeys(tmp.p, tb, k_in.as<uint64_t>(), k_out.as<uint64_t>(), (int64_t)nkeys, 0, end_bit, st));
  size_t ub = 0;
  LZ_CUDA(cub::DeviceSelect::Unique(nullptr, ub, k_out.as<uint64_t>(), k_in.as<uint64_t>(), nsel.as<int64_t>(), (int64_t)nkeys, st));
  if (ub > tb) { cudaFree(tmp.release()); LZ_CUDA(cudaMalloc(&tmp.p, ub)); }
  LZ_CUDA(cub::DeviceSelect::Unique(tmp.p, ub, k_out.as<uint64_t>(), k_in.as<uint64_t>(), nsel.as<int64_t>(), (int64_t)nkeys, st));
  int64_t nuniq = 0;
  uint64_t last = 0;
  LZ_CUDA(cudaMemcpyAsync(&nuniq, nsel.p, 8, cudaMemcpyDeviceToHost, st));
  LZ_CUDA(cudaStreamSynchronize(st));
  if (nuniq > 0) {
    LZ_CUDA(cudaMemcpy(&last, k_in.as<uint64_t>() + (nuniq - 1), 8, cudaMemcpyDeviceToHost));
    if (last == ~0ull) nuniq--;   // drop the sentinel
  }
  uint64_t nnz = (uint64_t)nuniq;
  if (nnz > 0xFFFFFFFFull) return lz_fail(LZ_ERR_ARG, "nnz %llu does not fit 32-bit row offsets", (unsigned long long)nnz);
  cudaFree(k_out.release());
  uint32_t *ro_d = nullptr, *ci_d = nullptr;
  LZ_CUDA(cudaMalloc((void**)&ro_d, (p.n + 1) * 4));
  if (cudaMalloc((void**)&ci_d, (nnz ? nnz : 1) * 4) != cudaSuccess) { cudaFree(ro_d); return lz_fail(LZ_ERR_ALLOC, "device allocation of col_idx failed"); }
  k_row_offsets_from_keys<<<grid_for(p.n + 1, 256), 256, 0, st>>>(k_in.as<uint64_t>(), nnz, p.n, ro_d);
  if (nnz) k_low32<<<grid_for(nnz, 256), 256, 0, st>>>(k_in.as<uint64_t>(), nnz, ci_d);
  LZ_CUDA(cudaStreamSynchronize(st));
  cudaFree(k_in.release()); cudaFree(tmp.release());
  c->have_x = c->have_tridiag = c->have_coef = c->have_ans = false;
  return lz_ingest_device_csr(c, p.n, nnz, ro_d, ci_d);
}

extern "C" int lz_graph_info_get(lz_ctx* c, lz_graph_info* out) {
  if (!c || !out) return lz_fail(LZ_ERR_ARG, "null argument");
  if (!c->row_ptr) return lz_fail(LZ_ERR_ARG, "no graph loaded");
  out->n = c->n; out->nnz = c->nnz; out->n_local = c->n_loc; out->nnz_local = c->nnz_loc;
  out->max_degree = c->max_degree; out->pad_ = 0; out->empty_rows = c->empty_rows;
  return LZ_OK;
}

extern "C" int lz_csr_download(lz_ctx* c, uint32_t* row_offset_out, uint32_t* col_idx_out) {
  if (!c || !row_offset_out || !col_idx_out) return lz_fail(LZ_ERR_ARG, "null argument");
  if (!c->row_ptr) return lz_fail(LZ_ERR_ARG, "no graph loaded");
  if (!c->orig_ro) return lz_fail(LZ_ERR_ARG, "the original-order CSR was not kept (multi-GPU contexts drop it; set LZ_KEEP_CSR=1 before loading the graph)");
  LZ_CUDA(cudaSetDevice(c->device));
  LZ_CUDA(cudaMemcpyAsync(row_offset_out, c->orig_ro, (c->n + 1) * 4, cudaMemcpyDeviceToHost, c->stream));
  LZ_CUDA(cudaMemcpyAsync(col_idx_out, c->orig_ci, c->nnz * 4, cudaMemcpyDeviceToHost, c->stream));
  LZ_CUDA(cudaStreamSynchronize(c->stream));
  return LZ_OK;
}
