// lz_api.cu — C ABI entry points (include/lz.h): context, start vector, the Lanczos driver loop, tridiagonal solve,
// multOut, read-back, test hooks and timing. Host orchestration only; kernels are in lz_kernels.cu.
//
// The driver loop replaces lanczosDecomp<T>::cu_decompose (reference parallel-final/lib/cu_lanczos.cu:97-128), which
// issues 8 launches + one D2H copy of q_j per step on three streams. Here one step is the SpMV passes (one per column block)
// plus ONE vector kernel, on one GPU and on several; the basis never leaves HBM, and the multi-GPU exchange and scalar
// reductions are peer stores / peer-memory slots fused into those kernels (NCCL only as fallback, for the reorthogonalisation
// coefficients and for the rendezvous that opens a run).
#include "lz_ctx.h"

#include <dlfcn.h>
#include <math.h>
#include <new>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <unistd.h>

namespace {
struct NcclBinding {
  lz_nccl_api api{};
  bool ok = false;
  char err[256] = "";
  NcclBinding() {
    void* h = dlopen("libnccl.so.2", RTLD_NOW | RTLD_NOLOAD);   // share a copy that is already in the process
    if (!h) h = dlopen("libnccl.so.2", RTLD_NOW | RTLD_LOCAL);
    if (!h) h = dlopen("libnccl.so", RTLD_NOW | RTLD_LOCAL);
    if (!h) { snprintf(err, sizeof(err), "libnccl.so.2 could not be loaded: %s", dlerror()); return; }
    bool all = true;
    auto sym = [&](const char* name) { void* p = dlsym(h, name); if (!p) all = false; return p; };
    api.GetUniqueId = (decltype(api.GetUniqueId))sym("ncclGetUniqueId");
    api.CommInitRank = (decltype(api.CommInitRank))sym("ncclCommInitRank");
    api.CommDestroy = (decltype(api.CommDestroy))sym("ncclCommDestroy");
    api.CommAbort = (decltype(api.CommAbort))sym("ncclCommAbort");
    api.CommSplit = (decltype(api.CommSplit))dlsym(h, "ncclCommSplit");   // optional
    api.AllReduce = (decltype(api.AllReduce))sym("ncclAllReduce");
    api.AllGather = (decltype(api.AllGather))sym("ncclAllGather");
    api.Broadcast = (decltype(api.Broadcast))sym("ncclBroadcast");
    api.GetErrorString = (decltype(api.GetErrorString))sym("ncclGetErrorString");
    api.GetVersion = (decltype(api.GetVersion))sym("ncclGetVersion");
    if (!all) { snprintf(err, sizeof(err), "libnccl.so.2 lacks a required symbol"); return; }
    ok = true;
  }
};
}  // namespace
// One host thread per GPU in one process is a supported mode (lib/final.cc run_multi): the binding is a function-local
// static, whose initialisation C++11 makes thread-safe.
const lz_nccl_api* lz_nccl() {
  static const NcclBinding binding;
  if (!binding.ok) { lz_fail(LZ_ERR_NCCL, "%s", binding.err); return nullptr; }
  return &binding.api;
}

static void drop_graph(lz_ctx* c) {
  if (c->graph_exec) { cudaGraphExecDestroy(c->graph_exec); c->graph_exec = nullptr; }
}

namespace {

int set_dev(lz_ctx* c) {
  LZ_CUDA(cudaSetDevice(c->device));
  return LZ_OK;
}

void close_peers(lz_ctx* c) {
  for (int r = 0; r < LZ_MAX_WORLD; r++) {
    if (c->peer_ipc[r]) {
      if (c->peer_xfull[r]) cudaIpcCloseMemHandle(c->peer_xfull[r]);
      if (c->peer_flags[r]) cudaIpcCloseMemHandle(c->peer_flags[r]);
    }
    c->peer_xfull[r] = nullptr; c->peer_flags[r] = nullptr; c->peer_ipc[r] = false;
  }
  c->peer_push = false;
  cudaFree(c->push_list); c->push_list = nullptr;
  c->sparse_push = false;
}

void free_vectors(lz_ctx* c) {
  close_peers(c);
  cudaFree(c->flags); cudaFree(c->push_ticket); cudaFree(c->gfull);
  c->flags = nullptr; c->push_ticket = nullptr; c->gfull = nullptr;
  cudaFree(c->V); cudaFree(c->w); cudaFree(c->xfull); cudaFree(c->xstage); cudaFree(c->ans);
  cudaFree(c->V32); cudaFree(c->q0_64);
  for (double*& r : c->ring) { cudaFree(r); r = nullptr; }
  c->V32 = nullptr; c->q0_64 = nullptr;
  cudaFree(c->alpha); cudaFree(c->beta); cudaFree(c->hcoef); cudaFree(c->eigvals); cudaFree(c->eigvecs); cudaFree(c->eigwork);
  cudaFree(c->coef); cudaFree(c->norm2v);
  c->norm2v = nullptr;
  c->lagged_done = false;
  c->V = c->w = c->xfull = c->xstage = c->ans = c->alpha = c->beta = c->hcoef = c->eigvals = c->eigvecs = c->eigwork = c->coef = nullptr;
  c->k_cap = 0;
  c->have_x = c->have_tridiag = c->have_coef = c->have_ans = false;
  cudaFree(c->ritz_R); c->ritz_R = nullptr; c->ritz_rows = 0; c->ritz_m = 0;
}

// Peer exchange set-up (collective: every rank calls it at the same point). Each rank publishes CUDA IPC handles of its
// gathered vector and arrival counters; ranks living in the same process (one host thread per GPU) use the raw pointers
// with peer access enabled instead. The decision to use the peer path is agreed by an all-reduce so no rank diverges.
struct lz_xchg {
  cudaIpcMemHandle_t hx, hf;
  unsigned long long pid, px, pf;
  int device, ok;
};

int setup_peers(lz_ctx* c) {
  c->peer_push = false;
  if (c->world == 1) return LZ_OK;
  bool want = c->world <= LZ_MAX_WORLD;
  if (const char* e = getenv("LZ_PEER_PUSH")) want = want && atoi(e) != 0;
  // arrival counters [LZ_MAX_COLBLK][LZ_MAX_WORLD] followed by the scalar exchange area [2 kinds][2][LZ_MAX_WORLD] x 16 B
  const size_t flag_bytes = sizeof(unsigned long long) * LZ_MAX_COLBLK * LZ_MAX_WORLD + 16 * 2 * 2 * LZ_MAX_WORLD;
  LZ_CUDA(cudaMalloc((void**)&c->flags, flag_bytes));
  LZ_CUDA(cudaMemsetAsync(c->flags, 0, flag_bytes, c->stream));
  c->red_seq = 0;
  LZ_CUDA(cudaMalloc((void**)&c->push_ticket, sizeof(unsigned int) * LZ_MAX_COLBLK));
  LZ_CUDA(cudaMemsetAsync(c->push_ticket, 0, sizeof(unsigned int) * LZ_MAX_COLBLK, c->stream));
  c->push_seq = 0;
  const int W = c->world;
  std::vector<lz_xchg> all(W);
  lz_xchg mine;
  memset(&mine, 0, sizeof(mine));
  mine.pid = (unsigned long long)getpid(); mine.px = (unsigned long long)c->xfull; mine.pf = (unsigned long long)c->flags;
  mine.device = c->device;
  mine.ok = want && cudaIpcGetMemHandle(&mine.hx, c->xfull) == cudaSuccess && cudaIpcGetMemHandle(&mine.hf, c->flags) == cudaSuccess;
  cudaGetLastError();
  struct DBuf { lz_xchg* p = nullptr; ~DBuf() { cudaFree(p); } } dguard;
  LZ_CUDA(cudaMalloc((void**)&dguard.p, sizeof(lz_xchg) * W));
  lz_xchg* dbuf = dguard.p;
  LZ_CUDA(cudaMemcpyAsync(dbuf + c->rank, &mine, sizeof(mine), cudaMemcpyHostToDevice, c->stream));
  LZ_NCCL(lz_nccl()->AllGather(dbuf + c->rank, dbuf, sizeof(lz_xchg), ncclChar, c->comm, c->stream));
  LZ_CUDA(cudaMemcpyAsync(all.data(), dbuf, sizeof(lz_xchg) * W, cudaMemcpyDeviceToHost, c->stream));
  LZ_CUDA(cudaStreamSynchronize(c->stream));
  int ok = 1;
  for (int r = 0; r < W; r++) ok &= all[r].ok;
  for (int r = 0; r < W && ok; r++) {
    if (r == c->rank) { c->peer_xfull[r] = c->xfull; c->peer_flags[r] = c->flags; continue; }
    if (all[r].pid == mine.pid) {                       // same process, another host thread: raw pointers + peer access
      int can = 0;
      if (cudaDeviceCanAccessPeer(&can, c->device, all[r].device) != cudaSuccess || !can) { ok = 0; break; }
      cudaError_t e = cudaDeviceEnablePeerAccess(all[r].device, 0);
      if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled) { ok = 0; break; }
      cudaGetLastError();
      c->peer_xfull[r] = (double*)all[r].px; c->peer_flags[r] = (unsigned long long*)all[r].pf;
    } else {
      void *px = nullptr, *pf = nullptr;
      if (cudaIpcOpenMemHandle(&px, all[r].hx, cudaIpcMemLazyEnablePeerAccess) != cudaSuccess ||
          cudaIpcOpenMemHandle(&pf, all[r].hf, cudaIpcMemLazyEnablePeerAccess) != cudaSuccess) {
        cudaGetLastError();
        if (px) cudaIpcCloseMemHandle(px);
        ok = 0;
        break;
      }
      c->peer_xfull[r] = (double*)px; c->peer_flags[r] = (unsigned long long*)pf; c->peer_ipc[r] = true;
    }
  }
  // agree: the peer path is used only if every rank mapped every peer
  double* flag_d = c->scal + 8;
  double okd = ok ? 1.0 : 0.0;
  LZ_CUDA(cudaMemcpyAsync(flag_d, &okd, 8, cudaMemcpyHostToDevice, c->stream));
  LZ_NCCL(lz_nccl()->AllReduce(flag_d, flag_d, 1, ncclDouble, ncclMin, c->comm, c->stream));
  LZ_CUDA(cudaMemcpyAsync(&okd, flag_d, 8, cudaMemcpyDeviceToHost, c->stream));
  LZ_CUDA(cudaStreamSynchronize(c->stream));
  if (okd < 0.5) { close_peers(c); return LZ_OK; }
  c->peer_push = true;
  return lz_build_push_lists(c);
}

// Vectors that depend only on the graph size.
int ensure_graph_vectors(lz_ctx* c) {
  if (!c->row_ptr) return lz_fail(LZ_ERR_ARG, "no graph loaded (call lz_csr_upload or lz_graph_generate first)");
  const uint64_t ldv = (c->n_loc + 31) & ~31ull;
  if (c->w && c->ldv == ldv && c->vec_n == c->n && c->vec_nloc == c->n_loc) {
    // same shape, possibly another graph: the exchange lists follow the graph, not the shape
    if (c->world > 1 && c->peer_push && c->push_graph_id != c->graph_id) LZ_TRY(lz_build_push_lists(c));
    return LZ_OK;
  }
  if (c->world > 1 && c->xfull) {
    // peers may still map this rank's buffers: everybody unmaps first, then (after a barrier) everybody frees
    close_peers(c);
    double* b = c->scal + 9;
    LZ_NCCL(lz_nccl()->AllReduce(b, b, 1, ncclDouble, ncclSum, c->comm, c->stream));
    LZ_CUDA(cudaStreamSynchronize(c->stream));
  }
  free_vectors(c);
  c->ldv = ldv; c->vec_n = c->n; c->vec_nloc = c->n_loc;
  c->epoch++;
  LZ_CUDA(cudaMalloc((void**)&c->w, ldv * 8));
  LZ_CUDA(cudaMalloc((void**)&c->ans, ldv * 8));
  LZ_CUDA(cudaMalloc((void**)&c->xstage, c->n * 8));
  LZ_CUDA(cudaMalloc((void**)&c->xfull, c->n_loc * (uint64_t)c->world * 8));
  LZ_CUDA(cudaMemsetAsync(c->w, 0, ldv * 8, c->stream));
  LZ_CUDA(cudaMemsetAsync(c->ans, 0, ldv * 8, c->stream));
  LZ_CUDA(cudaMemsetAsync(c->xfull, 0, c->n_loc * (uint64_t)c->world * 8, c->stream));
  if (c->world > 1) LZ_CUDA(cudaMalloc((void**)&c->gfull, c->n_loc * (uint64_t)c->world * 8));
  LZ_TRY(setup_peers(c));
  return LZ_OK;
}

// Row j of the Krylov basis as the fp64 vector the recurrence and the SpMV work on (fp32-basis mode: the ring), and as stored.
inline double* vec64(lz_ctx* c, uint32_t j) { return c->basis_f32 ? c->ring[j % 3] : c->V + (uint64_t)j * c->ldv; }
inline float* vec32(lz_ctx* c, uint32_t j) { return c->basis_f32 ? c->V32 + (uint64_t)j * c->ldv : nullptr; }
inline const void* basis_ptr(const lz_ctx* c) { return c->basis_f32 ? (const void*)c->V32 : (const void*)c->V; }

// Basis and k-sized arrays. Growing keeps row 0 (the start vector).
int ensure_k(lz_ctx* c, uint32_t k) {
  LZ_TRY(ensure_graph_vectors(c));
  if (k <= c->k_cap) return LZ_OK;
  LZ_CUDA(cudaStreamSynchronize(c->stream));
  if (c->basis_f32) {
    float* nv32 = nullptr;
    if (cudaMalloc((void**)&nv32, (uint64_t)k * c->ldv * 4) != cudaSuccess) {
      cudaGetLastError();
      return lz_fail(LZ_ERR_ALLOC, "cannot allocate the fp32 Lanczos basis: %u x %llu floats", k, (unsigned long long)c->ldv);
    }
    LZ_CUDA(cudaMemsetAsync(nv32, 0, (uint64_t)k * c->ldv * 4, c->stream));
    if (!c->q0_64) {
      LZ_CUDA(cudaMalloc((void**)&c->q0_64, c->ldv * 8));
      LZ_CUDA(cudaMemsetAsync(c->q0_64, 0, c->ldv * 8, c->stream));
      for (double*& r : c->ring) { LZ_CUDA(cudaMalloc((void**)&r, c->ldv * 8)); LZ_CUDA(cudaMemsetAsync(r, 0, c->ldv * 8, c->stream)); }
    }
    if (c->V32 && c->have_x) LZ_CUDA(cudaMemcpyAsync(nv32, c->V32, c->ldv * 4, cudaMemcpyDeviceToDevice, c->stream));
    LZ_CUDA(cudaStreamSynchronize(c->stream));
    cudaFree(c->V32);
    c->V32 = nv32;
  } else {
    double* nv = nullptr;
    if (cudaMalloc((void**)&nv, (uint64_t)k * c->ldv * 8) != cudaSuccess) {
      cudaGetLastError();
      return lz_fail(LZ_ERR_ALLOC, "cannot allocate the Lanczos basis: %u x %llu doubles", k, (unsigned long long)c->ldv);
    }
    LZ_CUDA(cudaMemsetAsync(nv, 0, (uint64_t)k * c->ldv * 8, c->stream));
    if (c->V && c->have_x) LZ_CUDA(cudaMemcpyAsync(nv, c->V, c->ldv * 8, cudaMemcpyDeviceToDevice, c->stream));
    LZ_CUDA(cudaStreamSynchronize(c->stream));
    cudaFree(c->V);
    c->V = nv;
  }
  // k-sized arrays: allocate the new set first, swap on success, so a failed cudaMalloc leaves a consistent (old) state
  double* fresh[8] = {};
  const size_t bytes[8] = {(size_t)(k + 1) * 8, (size_t)k * 8, (size_t)k * 8, (size_t)k * 8, (size_t)k * 8, (size_t)k * k * 8, (size_t)k * k * 8, (size_t)k * 8};
  for (int i = 0; i < 8; i++)
    if (cudaMalloc((void**)&fresh[i], bytes[i]) != cudaSuccess) {
      cudaGetLastError();
      for (int t = 0; t < i; t++) cudaFree(fresh[t]);
      // the basis already has k rows but the small arrays do not: fall back to "nothing allocated" rather than a half state
      cudaFree(c->V); c->V = nullptr; cudaFree(c->V32); c->V32 = nullptr; c->k_cap = 0; c->have_x = false;
      c->have_tridiag = c->have_coef = c->have_ans = false;
      return lz_fail(LZ_ERR_ALLOC, "cannot allocate the k-sized work arrays for k = %u", k);
    }
  double** slot[8] = {&c->norm2v, &c->alpha, &c->beta, &c->hcoef, &c->eigvals, &c->eigvecs, &c->eigwork, &c->coef};
  for (int i = 0; i < 8; i++) { cudaFree(*slot[i]); *slot[i] = fresh[i]; }
  c->lagged_done = false;
  c->k_cap = k;
  c->have_tridiag = c->have_coef = c->have_ans = false;
  return LZ_OK;
}

cudaEvent_t next_event(lz_ctx* c) {
  if (c->ev_used == c->ev_pool.size()) {
    cudaEvent_t e;
    cudaEventCreate(&e);
    c->ev_pool.push_back(e);
  }
  return c->ev_pool[c->ev_used++];
}
// profiling marks: kind 0 spmv, 1 update/scale, 2 comm, 3 reorth
struct Mark { int kind; cudaEvent_t a, b; };
thread_local std::vector<Mark> g_marks;

struct Scope {
  lz_ctx* c; int kind; cudaEvent_t a = nullptr;
  Scope(lz_ctx* c_, int kind_) : c(c_), kind(kind_) {
    if (c->profiling) { a = next_event(c); cudaEventRecord(a, c->stream); }
  }
  ~Scope() {
    if (c->profiling) { cudaEvent_t b = next_event(c); cudaEventRecord(b, c->stream); g_marks.push_back({kind, a, b}); }
  }
};

int allreduce_sum(lz_ctx* c, double* buf, size_t count) {
  if (c->world == 1) return LZ_OK;
  Scope s(c, 2);
  LZ_NCCL(lz_nccl()->AllReduce(buf, buf, count, ncclDouble, ncclSum, c->comm, c->stream));
  return LZ_OK;
}
// All-gather of the chunk-major vector `full` (every rank has already stored its own slots). One in-place ncclAllGather
// per chunk. async: issued on the communication stream behind `stream`, one event per chunk, so SpMV pass b can start as
// soon as chunk b has arrived while later chunks are still in flight. Otherwise: on `stream`, fully ordered.
int allgather_chunks(lz_ctx* c, double* full, bool async) {
  if (c->world == 1) return LZ_OK;
  const uint64_t cl = c->chunk_rows, span = cl * (uint64_t)c->world;
  if (async && c->comm_overlap) {
    LZ_CUDA(cudaEventRecord(c->ev_scaled, c->stream));
    LZ_CUDA(cudaStreamWaitEvent(c->comm_stream, c->ev_scaled, 0));
    cudaEvent_t a = nullptr;
    if (c->profiling) { a = next_event(c); cudaEventRecord(a, c->comm_stream); }
    for (uint32_t b = 0; b < c->ncolblk; b++) {
      double* base = full + (uint64_t)b * span;
      LZ_NCCL(lz_nccl()->AllGather(base + (uint64_t)c->rank * cl, base, cl, ncclDouble, c->comm_ag, c->comm_stream));
      LZ_CUDA(cudaEventRecord(c->ev_chunk[b], c->comm_stream));
    }
    if (c->profiling) { cudaEvent_t e = next_event(c); cudaEventRecord(e, c->comm_stream); g_marks.push_back({2, a, e}); }
    c->chunks_in_flight = true;
  } else {
    Scope s(c, 2);
    for (uint32_t b = 0; b < c->ncolblk; b++) {
      double* base = full + (uint64_t)b * span;
      LZ_NCCL(lz_nccl()->AllGather(base + (uint64_t)c->rank * cl, base, cl, ncclDouble, c->comm, c->stream));
    }
    c->chunks_in_flight = false;
  }
  return LZ_OK;
}

}  // namespace

extern "C" int lz_device_count(int* count_out) {
  if (!count_out) return lz_fail(LZ_ERR_ARG, "null argument");
  LZ_CUDA(cudaGetDeviceCount(count_out));
  return LZ_OK;
}

static int create_body(lz_ctx* c, int device, int rank, int world, const void* uid);

static int create_common(int device, int rank, int world, const void* uid, lz_ctx** out) {
  if (!out) return lz_fail(LZ_ERR_ARG, "null ctx_out");
  *out = nullptr;
  if (world < 1 || rank < 0 || rank >= world) return lz_fail(LZ_ERR_ARG, "bad rank %d / world %d", rank, world);
  int ndev = 0;
  cudaError_t e = cudaGetDeviceCount(&ndev);
  if (e != cudaSuccess || ndev == 0)
    return lz_fail(LZ_ERR_CUDA, "no CUDA device available (%s); this library has no CPU fallback", e != cudaSuccess ? cudaGetErrorString(e) : "0 devices");
  if (device < 0 || device >= ndev) return lz_fail(LZ_ERR_ARG, "device %d out of range (have %d)", device, ndev);
  LZ_CUDA(cudaSetDevice(device));
  lz_ctx* c = new (std::nothrow) lz_ctx();
  if (!c) return lz_fail(LZ_ERR_ALLOC, "out of host memory");
  const int rc = create_body(c, device, rank, world, uid);
  if (rc != LZ_OK) {          // keep the message of the failure, release whatever was created
    char msg[512];
    snprintf(msg, sizeof(msg), "%s", lz_last_error());
    lz_destroy(c);
    return lz_fail(rc, "%s", msg);
  }
  *out = c;
  return LZ_OK;
}

static int create_body(lz_ctx* c, int device, int rank, int world, const void* uid) {
  c->device = device; c->rank = rank; c->world = world;
  cudaDeviceProp prop;
  LZ_CUDA(cudaGetDeviceProperties(&prop, device));
  c->sm_count = prop.multiProcessorCount;
  if (const char* e = getenv("LZ_SPMV_VARIANT")) { int v = atoi(e); if (v >= 0 && v <= LZ_SPMV_WARP) c->spmv_variant = v; }     // tuning knob
  if (const char* e = getenv("LZ_SPMV_CTAS")) { int v = atoi(e); if (v >= 1 && v <= 32) c->spmv_ctas_per_sm = (uint32_t)v; }   // tuning knob
  if (const char* e = getenv("LZ_LAGGED_NORM")) c->lagged = atoi(e) != 0;
  if (const char* e = getenv("LZ_BASIS")) c->basis_f32 = (e[0] == 'f' || e[0] == 'F') && strstr(e, "32") != nullptr;   // "f32": experiments
  if (const char* e = getenv("LZ_PUSH_CTAS")) { int v = atoi(e); if (v >= 1 && v <= 1024) c->push_ctas = (uint32_t)v; }        // tuning knob
  if (const char* e = getenv("LZ_SELL_GROUP")) { int v = atoi(e); if (v == 1 || v == 4) c->sell_group_force = (uint32_t)v; }      // test knob
  // watchdog of the in-kernel waits on peers (seconds; 0 = none). A trap poisons the CUDA context: the ctx must be destroyed.
  if (world > 1) LZ_TRY(lz_k_set_peer_timeout(c, getenv("LZ_PEER_TIMEOUT_S") ? atof(getenv("LZ_PEER_TIMEOUT_S")) : 20.0));
  LZ_CUDA(cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking));
  LZ_CUDA(cudaEventCreate(&c->ev_a)); LZ_CUDA(cudaEventCreate(&c->ev_b));
  LZ_CUDA(cudaEventCreate(&c->ev_e0)); LZ_CUDA(cudaEventCreate(&c->ev_e1));
  LZ_CUDA(cudaEventCreate(&c->ev_m0)); LZ_CUDA(cudaEventCreate(&c->ev_m1));
  LZ_CUDA(cudaEventCreate(&c->ev_t0)); LZ_CUDA(cudaEventCreate(&c->ev_t1));
  LZ_CUDA(cudaMalloc((void**)&c->scal, 16 * 8));
  LZ_CUDA(cudaMemset(c->scal, 0, 16 * 8));
  LZ_CUDA(cudaMalloc((void**)&c->ticket, 16 * sizeof(unsigned int)));
  LZ_CUDA(cudaMemset(c->ticket, 0, 16 * sizeof(unsigned int)));
  LZ_CUDA(cudaMalloc((void**)&c->status, 4 * sizeof(int)));
  LZ_CUDA(cudaMemset(c->status, 0, 4 * sizeof(int)));
  if (world > 1) {
    if (!uid) return lz_fail(LZ_ERR_ARG, "world > 1 needs an NCCL unique id");
    ncclUniqueId id;
    static_assert(sizeof(ncclUniqueId) == LZ_NCCL_UID_BYTES, "NCCL unique id size");
    memcpy(&id, uid, sizeof(id));
    if (!lz_nccl()) return LZ_ERR_NCCL;
    LZ_NCCL(lz_nccl()->CommInitRank(&c->comm, world, id, rank));
    if (const char* e = getenv("LZ_COMM_OVERLAP")) c->comm_overlap = atoi(e) != 0;
    // a second communicator so the chunked all-gather (communication stream) never serialises with the all-reduces
    if (c->comm_overlap && lz_nccl()->CommSplit && lz_nccl()->CommSplit(c->comm, 0, rank, &c->comm_ag, nullptr) != ncclSuccess) c->comm_ag = nullptr;
    if (!c->comm_ag) c->comm_overlap = false;
    LZ_CUDA(cudaStreamCreateWithFlags(&c->comm_stream, cudaStreamNonBlocking));
    LZ_CUDA(cudaEventCreateWithFlags(&c->ev_scaled, cudaEventDisableTiming));
    for (int b = 0; b < LZ_MAX_COLBLK; b++) LZ_CUDA(cudaEventCreateWithFlags(&c->ev_chunk[b], cudaEventDisableTiming));
  }
  return LZ_OK;
}

extern "C" int lz_create(int device, lz_ctx** ctx_out) { return create_common(device, 0, 1, nullptr, ctx_out); }

extern "C" int lz_nccl_unique_id(void* uid_out) {
  if (!uid_out) return lz_fail(LZ_ERR_ARG, "null argument");
  ncclUniqueId id;
  if (!lz_nccl()) return LZ_ERR_NCCL;
  LZ_NCCL(lz_nccl()->GetUniqueId(&id));
  memcpy(uid_out, &id, sizeof(id));
  return LZ_OK;
}

extern "C" int lz_create_dist(int device, int rank, int world, const void* uid, lz_ctx** ctx_out) {
  return create_common(device, rank, world, uid, ctx_out);
}

extern "C" int lz_destroy(lz_ctx* c) {
  if (!c) return LZ_OK;
  cudaSetDevice(c->device);
  const bool healthy = !c->stream || cudaStreamSynchronize(c->stream) == cudaSuccess;
  // after a device fault a collective may never complete on the peers: abort instead of the (blocking) destroy
  if (c->comm_stream) cudaStreamSynchronize(c->comm_stream);
  if (c->comm_ag && lz_nccl()) { if (healthy) lz_nccl()->CommDestroy(c->comm_ag); else lz_nccl()->CommAbort(c->comm_ag); }
  if (c->comm && lz_nccl()) { if (healthy) lz_nccl()->CommDestroy(c->comm); else lz_nccl()->CommAbort(c->comm); }
  if (c->comm_stream) cudaStreamDestroy(c->comm_stream);
  if (c->ev_scaled) cudaEventDestroy(c->ev_scaled);
  for (int b = 0; b < LZ_MAX_COLBLK; b++) if (c->ev_chunk[b]) cudaEventDestroy(c->ev_chunk[b]);
  drop_graph(c);
  free_vectors(c);
  lz_free_graph(c);
  lz_free_rank(c);
  cudaFree(c->trace_buf);
  cudaFree(c->scal); cudaFree(c->partials); cudaFree(c->ticket); cudaFree(c->status); cudaFree(c->flush_buf);
  for (cudaEvent_t e : c->ev_pool) cudaEventDestroy(e);
  for (cudaEvent_t e : {c->ev_a, c->ev_b, c->ev_e0, c->ev_e1, c->ev_m0, c->ev_m1, c->ev_t0, c->ev_t1})
    if (e) cudaEventDestroy(e);
  if (c->stream) cudaStreamDestroy(c->stream);
  cudaGetLastError();
  delete c;
  return LZ_OK;
}

extern "C" int lz_sync(lz_ctx* c) {
  if (!c) return lz_fail(LZ_ERR_ARG, "null ctx");
  LZ_TRY(set_dev(c));
  LZ_CUDA(cudaStreamSynchronize(c->stream));
  return LZ_OK;
}

extern "C" int lz_set_basis_precision(lz_ctx* c, int precision) {
  if (!c || (precision != LZ_BASIS_F64 && precision != LZ_BASIS_F32)) return lz_fail(LZ_ERR_ARG, "bad basis precision");
  if ((precision == LZ_BASIS_F32) == c->basis_f32) return LZ_OK;
  LZ_TRY(set_dev(c));
  LZ_CUDA(cudaStreamSynchronize(c->stream));
  drop_graph(c);
  // the basis and the start vector are re-created in the new precision by the next lz_set_start_vector
  cudaFree(c->V); c->V = nullptr; cudaFree(c->V32); c->V32 = nullptr;
  cudaFree(c->q0_64); c->q0_64 = nullptr;
  for (double*& r : c->ring) { cudaFree(r); r = nullptr; }
  c->k_cap = 0;
  c->epoch++;
  c->basis_f32 = precision == LZ_BASIS_F32;
  c->have_x = c->have_tridiag = c->have_coef = c->have_ans = false;
  c->lagged_done = false;
  return LZ_OK;
}

static const char* const kIndefiniteMsg =
    "resolvent: 1 - alpha * theta <= 0 for a Ritz value theta, (I - alpha A) is not positive definite (alpha >= 1 / lambda_max)";

// Only the coefficient solve depends on the function: the tridiagonal and the basis stay valid, the coefficients and the answer go.
extern "C" int lz_set_matfun(lz_ctx* c, int kind, double param) {
  if (!c) return lz_fail(LZ_ERR_ARG, "null ctx");
  if (kind != LZ_MATFUN_EXP && kind != LZ_MATFUN_EXP_SCALED && kind != LZ_MATFUN_RESOLVENT)
    return lz_fail(LZ_ERR_ARG, "unknown matrix function %d", kind);
  if (!isfinite(param)) return lz_fail(LZ_ERR_ARG, "matrix function parameter must be finite");
  c->matfun_kind = kind;
  c->matfun_param = param;
  c->have_coef = c->have_ans = false;
  return LZ_OK;
}

extern "C" int lz_get_matfun_scale(lz_ctx* c, double* log_scale_out) {
  if (!c || !log_scale_out) return lz_fail(LZ_ERR_ARG, "null argument");
  if (!c->have_coef) return lz_fail(LZ_ERR_ARG, "lz_tridiag_expv must be called before lz_get_matfun_scale");
  LZ_TRY(set_dev(c));
  LZ_CUDA(cudaMemcpyAsync(log_scale_out, c->scal + 5, 8, cudaMemcpyDeviceToHost, c->stream));
  LZ_CUDA(cudaStreamSynchronize(c->stream));
  return LZ_OK;
}

extern "C" int lz_set_spmv_variant(lz_ctx* c, int variant) {
  if (!c || variant < 0 || variant > LZ_SPMV_WARP) return lz_fail(LZ_ERR_ARG, "bad SpMV variant");
  c->spmv_variant = variant;
  return LZ_OK;
}

// x -> device, ||2^-e x||^2 -> scal[2] with e = x_exp the exponent of max|x|, q_0 = x/||x|| -> V[0] (and the gathered buffer when
// world > 1). Squaring x as it is underflows below |x_i| ~ 1e-154 (||x|| loses digits, q_0 is not a unit vector) and overflows above
// ~1e154; 2^-e x has max in [1, 2) and the same q_0. For every x whose squares stay normal the bits are those of the unscaled sum.
// Replaces cu_lanczos.cu:30-34 (host normalisation) + :88 (H2D of q_0).
// root < 0: every rank passes the vector itself (or NULL = ones). root >= 0: only `root` reads x_host; the other ranks
// receive it over NVLink (one PCIe upload instead of `world` concurrent ones).
static int set_start_vector_impl(lz_ctx* c, const double* x_host, int root) {
  if (!c) return lz_fail(LZ_ERR_ARG, "null ctx");
  if (root >= c->world) return lz_fail(LZ_ERR_ARG, "root %d out of range", root);
  LZ_TRY(set_dev(c));
  LZ_TRY(ensure_k(c, c->k_cap ? c->k_cap : 2));
  if (root >= 0 && c->world > 1) {
    if (c->rank == root) {
      if (!x_host) return lz_fail(LZ_ERR_ARG, "the root rank must pass the start vector");
      LZ_CUDA(cudaMemcpyAsync(c->xstage, x_host, c->n * 8, cudaMemcpyHostToDevice, c->stream));
    }
    LZ_NCCL(lz_nccl()->Broadcast(c->xstage, c->xstage, c->n, ncclDouble, root, c->comm, c->stream));
  } else if (x_host) {
    LZ_CUDA(cudaMemcpyAsync(c->xstage, x_host, c->n * 8, cudaMemcpyHostToDevice, c->stream));
  } else {
    LZ_TRY(lz_k_fill(c, c->xstage, c->n, 1.0));   // all ones, as every reference driver uses (main.cu:79)
  }
  c->x_exp = 0;
  c->have_x = c->have_tridiag = c->have_coef = c->have_ans = false;
  if (x_host || (root >= 0 && c->world > 1)) {    // a caller's vector: one read-back of max|x| (ones: e = 0)
    auto* mx_d = reinterpret_cast<unsigned long long*>(c->scal + 6);
    LZ_CUDA(cudaMemsetAsync(mx_d, 0, 8, c->stream));
    LZ_TRY(lz_k_absmax_bits(c, c->xstage, c->n, mx_d));
    double mx = 0.0;
    LZ_CUDA(cudaMemcpyAsync(&mx, mx_d, 8, cudaMemcpyDeviceToHost, c->stream));
    LZ_CUDA(cudaStreamSynchronize(c->stream));
    if (!(mx > 0.0) || !isfinite(mx)) return lz_fail(LZ_ERR_ARG, "start vector is zero or not finite (max |x_i| = %g)", mx);
    c->x_exp = ilogb(mx);
  }
  LZ_TRY(lz_k_norm2(c, c->xstage, c->n, c->x_exp, c->scal + 2));
  double* q0 = c->basis_f32 ? c->q0_64 : c->V;
  if (c->world > 1) {
    LZ_TRY(lz_k_permute_in_local(c, c->xstage, c->scal + 2, q0));   // own rows only; the gathered vector is filled by the run
  } else {
    LZ_TRY(lz_k_permute_in(c, c->xstage, c->scal + 2, 0, c->n_loc, q0));
  }
  if (c->basis_f32) LZ_TRY(lz_k_convert(c, q0, c->V32, nullptr, nullptr, c->n_loc));
  c->have_x = true;
  c->have_tridiag = c->have_coef = c->have_ans = false;
  return LZ_OK;
}

// Enqueues the k Lanczos steps on c->stream (also used under stream capture for the CUDA-graph path).
static int enqueue_steps(lz_ctx* c, uint32_t k, int reorth, bool fused_push, bool peer_scalars) {
  const uint64_t ldv = c->ldv;
  const bool dist = c->world > 1;
  LZ_CUDA(cudaMemsetAsync(c->status + 2, 0, sizeof(int), c->stream));
  c->lagged_run = false;
  if (!dist && !reorth && c->lagged) {
    c->lagged_run = true;
    // Lagged normalisation: 2 SpMV passes + ONE vector kernel per step; row j >= 1 of V keeps u_j unnormalised with
    // norm2v[j] = ||u_j||^2 (row 0 is the normalised start vector). See k_update_lagged.
    LZ_TRY(lz_k_fill(c, c->norm2v, 1, 1.0));
    if (c->basis_f32) LZ_CUDA(cudaMemcpyAsync(c->ring[0], c->q0_64, ldv * 8, cudaMemcpyDeviceToDevice, c->stream));
    for (uint32_t j = 0; j < k; j++) {
      double* uj = vec64(c, j);
      {  // t = A u_j ; alpha_j = (t . u_j) / ||u_j||^2
        Scope s(c, 0);
        LZ_TRY(lz_k_spmv_dot(c, uj, uj, c->w, c->alpha + j, 0ull, nullptr, 0ull, c->norm2v + j));
      }
      if (j + 1 == k) break;
      {  // u_{j+1} = t/||u_j|| - alpha_j q_j - beta_{j-1} q_{j-1} ; ||u_{j+1}||^2 ; beta_j
        Scope s(c, 1);
        LZ_TRY(lz_k_update_lagged(c, c->w, uj, j ? vec64(c, j - 1) : nullptr, c->alpha + j, c->norm2v + j, j ? c->norm2v + (j - 1) : nullptr,
                                  vec64(c, j + 1), c->norm2v + (j + 1), c->beta + j, vec32(c, j + 1)));
      }
    }
    return LZ_OK;
  }
  if (!dist && reorth && c->lagged) {
    // Full reorthogonalisation with the lagged normalisation (one GPU): the basis rows stay unnormalised (row j holds u_j, norm2v[j] =
    // ||u_j||^2), the Gram-Schmidt coefficients are (u_t . w) / ||u_t||^2 (divided in k_multidot's last CTA) and the last k_combine
    // of the step writes u_{j+1} straight into its basis row — the normalisation pass (k_scale: one launch, 16 n bytes) is gone.
    c->lagged_run = true;
    LZ_TRY(lz_k_fill(c, c->norm2v, 1, 1.0));
    if (c->basis_f32) LZ_CUDA(cudaMemcpyAsync(c->ring[0], c->q0_64, ldv * 8, cudaMemcpyDeviceToDevice, c->stream));
    int* skip = c->status + 1;
    for (uint32_t j = 0; j < k; j++) {
      double* uj = vec64(c, j);
      {
        Scope s(c, 0);
        LZ_TRY(lz_k_spmv_dot(c, uj, uj, c->w, c->alpha + j, 0ull, nullptr, 0ull, c->norm2v + j));
      }
      if (j + 1 == k) break;
      double* un = vec64(c, j + 1);
      {  // three-term recurrence into the next basis row; ||.||^2 before the projections -> scal[3]
        Scope s(c, 1);
        LZ_TRY(lz_k_update_lagged(c, c->w, uj, j ? vec64(c, j - 1) : nullptr, c->alpha + j, c->norm2v + j, j ? c->norm2v + (j - 1) : nullptr,
                                  un, c->scal + 3, c->beta + j, nullptr));
      }
      {
        Scope s(c, 3);
        LZ_TRY(lz_k_multidot(c, basis_ptr(c), c->basis_f32, j + 1, un, c->hcoef, nullptr, c->norm2v));
        LZ_TRY(lz_k_combine(c, basis_ptr(c), c->basis_f32, j + 1, c->hcoef, -1.0, un, un, c->scal + 1, nullptr, vec32(c, j + 1)));
        LZ_TRY(lz_k_reorth_decide(c, c->scal + 3, c->scal + 1, skip, reinterpret_cast<unsigned int*>(c->status + 2)));
        LZ_TRY(lz_k_multidot(c, basis_ptr(c), c->basis_f32, j + 1, un, c->hcoef, skip, c->norm2v));
        LZ_TRY(lz_k_combine(c, basis_ptr(c), c->basis_f32, j + 1, c->hcoef, -1.0, un, un, c->scal + 4, skip, vec32(c, j + 1)));
        LZ_TRY(lz_k_reorth_select(c, skip, c->scal + 4, c->scal + 1, c->norm2v + (j + 1), c->beta + j));
      }
    }
    return LZ_OK;
  }
  if (dist && !reorth && c->lagged && c->peer_push && peer_scalars) {
    // Lagged normalisation over the peer exchange: SpMV passes + ONE kernel per step (k_update_lagged_push): it waits for
    // alpha, forms u_{j+1} and stores it straight into every rank's gathered vector; ||u_{j+1}||^2 is reduced off the
    // critical path. The gathered vector holds u_j unnormalised.
    LZ_TRY(lz_k_fill(c, c->norm2v, 1, 1.0));
    if (c->basis_f32) LZ_CUDA(cudaMemcpyAsync(c->ring[0], c->q0_64, ldv * 8, cudaMemcpyDeviceToDevice, c->stream));
    const uint32_t push_chunks = fused_push ? 1u : c->ncolblk;
    LZ_TRY(lz_k_scale_push(c, vec64(c, 0), nullptr, vec64(c, 0), nullptr, ++c->push_seq, push_chunks));   // q_0 (a previous run left its last vector there)
    for (uint32_t j = 0; j < k; j++) {
      double* uj = vec64(c, j);
      const double* q_dot = c->ncolblk == 1 ? c->xfull + (uint64_t)c->rank * c->chunk_rows : uj;
      ++c->red_seq;
      {
        Scope s(c, 0);
        LZ_TRY(lz_k_spmv_dot(c, c->xfull, q_dot, c->w, c->alpha + j, c->push_seq, fused_push ? uj : nullptr, c->red_seq));
      }
      if (j + 1 == k) { LZ_TRY(lz_k_lagged_finish(c, j, c->red_seq)); break; }
      {
        Scope s(c, 1);
        LZ_TRY(lz_k_update_lagged_push(c, c->w, uj, j ? vec64(c, j - 1) : nullptr, vec64(c, j + 1), j, ++c->push_seq, push_chunks, c->red_seq,
                                       vec32(c, j + 1)));
      }
    }
    c->lagged_run = true;
    return LZ_OK;
  }
  if (c->basis_f32) LZ_CUDA(cudaMemcpyAsync(c->ring[0], c->q0_64, ldv * 8, cudaMemcpyDeviceToDevice, c->stream));
  if (dist) {   // q_0 into the gathered buffer (a previous run left q_{k-1} there)
    if (c->peer_push) {
      LZ_TRY(lz_k_scale_push(c, vec64(c, 0), nullptr, vec64(c, 0), nullptr, ++c->push_seq, fused_push ? 1u : c->ncolblk));
    } else {
      LZ_TRY(lz_k_spread(c, vec64(c, 0), c->xfull));
      LZ_TRY(allgather_chunks(c, c->xfull, true));
    }
  }
  for (uint32_t j = 0; j < k; j++) {
    double* qj = vec64(c, j);
    double* qprev = j ? vec64(c, j - 1) : nullptr;
    double* qnext = vec64(c, j + 1 < k ? j + 1 : j);
    {  // w = A q_j ; alpha_j = w . q_j                                   (cu_lanczos.cu:101-105)
      Scope s(c, 0);
      const bool last = j + 1 == k;    // the last alpha is read by nobody on the device: reduce it with NCCL into alpha[k-1]
      // with a single chunk this rank's slots of the gathered vector are contiguous and hold the same bits as q_j: read the
      // alpha operand from there, so it shares cache lines with the gathers instead of streaming a second copy from HBM
      const double* q_dot = (dist && c->ncolblk == 1) ? c->xfull + (uint64_t)c->rank * c->chunk_rows : qj;
      LZ_TRY(lz_k_spmv_dot(c, dist ? c->xfull : qj, q_dot, c->w, c->alpha + j, c->peer_push ? c->push_seq : 0ull, fused_push ? qj : nullptr,
                           (peer_scalars && !last) ? ++c->red_seq : 0ull));
    }
    if (!peer_scalars || j + 1 == k) LZ_TRY(allreduce_sum(c, c->alpha + j, 1));
    if (j + 1 == k) break;                                               // last step needs alpha only (cu_lanczos.cu:116)
    {  // w -= alpha_j q_j ; w -= beta_{j-1} q_{j-1} ; ||w||^2             (cu_lanczos.cu:108-120)
      Scope s(c, 1);
      const unsigned long long a_seq = peer_scalars ? c->red_seq : 0ull;   // consumes alpha (kind 0, a_seq), publishes ||w||^2 (kind 1, a_seq)
      LZ_TRY(lz_k_update_norm(c, c->w, qj, qprev, c->alpha + j, j ? c->beta + (j - 1) : nullptr,
                              reorth ? c->scal + 3 : c->scal + 1, a_seq));
    }
    if (reorth) {
      // Full reorthogonalisation against q_0..q_j: classical Gram-Schmidt, repeated only when the first pass removed more
      // than half of ||w||^2 ("twice is enough"); the decision is taken on the device.
      Scope s(c, 3);
      int* skip = c->status + 1;
      LZ_TRY(allreduce_sum(c, c->scal + 3, 1));                                   // ||w||^2 before
      LZ_TRY(lz_k_multidot(c, basis_ptr(c), c->basis_f32, j + 1, c->w, c->hcoef));
      LZ_TRY(allreduce_sum(c, c->hcoef, j + 1));
      LZ_TRY(lz_k_combine(c, basis_ptr(c), c->basis_f32, j + 1, c->hcoef, -1.0, c->w, c->w, c->scal + 1));
      LZ_TRY(allreduce_sum(c, c->scal + 1, 1));                                   // ||w||^2 after pass 1
      LZ_TRY(lz_k_reorth_decide(c, c->scal + 3, c->scal + 1, skip, reinterpret_cast<unsigned int*>(c->status + 2)));
      LZ_TRY(lz_k_multidot(c, basis_ptr(c), c->basis_f32, j + 1, c->w, c->hcoef, skip));
      LZ_TRY(allreduce_sum(c, c->hcoef, j + 1));
      LZ_TRY(lz_k_combine(c, basis_ptr(c), c->basis_f32, j + 1, c->hcoef, -1.0, c->w, c->w, c->scal + 4, skip));
      LZ_TRY(allreduce_sum(c, c->scal + 4, 1));
      LZ_TRY(lz_k_reorth_select(c, skip, c->scal + 4, c->scal + 1));
    }
    if (!peer_scalars && !reorth) LZ_TRY(allreduce_sum(c, c->scal + 1, 1));
    {  // beta_j = ||w|| ; q_{j+1} = w / beta_j                            (cu_lanczos.cu:120-123)
      Scope s(c, 1);
      if (c->peer_push) {
        LZ_TRY(lz_k_scale_push(c, c->w, c->scal + 1, qnext, c->beta + j, ++c->push_seq, fused_push ? 1u : c->ncolblk,
                               peer_scalars ? c->red_seq : 0ull));
        if (c->basis_f32) LZ_TRY(lz_k_convert(c, qnext, vec32(c, j + 1), nullptr, nullptr, c->n_loc));   // fp32 basis row
      } else {
        LZ_TRY(lz_k_scale(c, c->w, c->scal + 1, qnext, dist ? c->xfull : nullptr, c->beta + j, vec32(c, j + 1)));
      }
    }
    if (!c->peer_push) LZ_TRY(allgather_chunks(c, c->xfull, true));
  }
  return LZ_OK;
}

extern "C" int lz_set_start_vector(lz_ctx* c, const double* x_host) { return set_start_vector_impl(c, x_host, -1); }
extern "C" int lz_set_start_vector_root(lz_ctx* c, const double* x_host, int root) {
  if (root < 0) return lz_fail(LZ_ERR_ARG, "root must be >= 0");
  return set_start_vector_impl(c, x_host, root);
}

extern "C" int lz_lanczos_run(lz_ctx* c, uint32_t k, int reorth) {
  if (!c) return lz_fail(LZ_ERR_ARG, "null ctx");
  if (k < 1) return lz_fail(LZ_ERR_ARG, "krylov dimension must be >= 1");
  if (reorth != LZ_REORTH_NONE && reorth != LZ_REORTH_FULL) return lz_fail(LZ_ERR_ARG, "bad reorth mode %d", reorth);
  if (!c->have_x) return lz_fail(LZ_ERR_ARG, "lz_set_start_vector must be called before lz_lanczos_run");
  LZ_TRY(set_dev(c));
  LZ_TRY(ensure_k(c, k));
  // chunk 0 of each new vector is sent by the normalisation kernel, chunk b + 1 by SpMV pass b (sliced variant only)
  bool fused_push = c->peer_push && !c->sparse_push && c->spmv_variant == LZ_SPMV_AUTO && c->ncolblk > 1;
  // plain Lanczos on the sliced variant: alpha and ||w||^2 are reduced through peer memory too (no collective launches)
  bool peer_scalars = c->peer_push && c->spmv_variant == LZ_SPMV_AUTO && reorth == LZ_REORTH_NONE;
  if (const char* e = getenv("LZ_PEER_SCALARS")) peer_scalars = peer_scalars && atoi(e) != 0;
  if (const char* e = getenv("LZ_FUSED_PUSH")) fused_push = fused_push && atoi(e) != 0;
  c->ev_used = 0;
  g_marks.clear();
  // Reduction scratch for every kernel of the loop is reserved here, once: nothing inside enqueue_steps allocates or frees
  // (a cudaFree there would synchronise the device per step, and with one thread per GPU it can deadlock against a peer
  // that is inside a spin kernel or an NCCL call).
  {
    uint64_t need = (uint64_t)c->sm_count * (c->spmv_ctas_per_sm > 8 ? c->spmv_ctas_per_sm : 8);
    if (reorth) need = (uint64_t)c->sm_count * 4 * (k > 2 ? k : 2);
    if (need < (uint64_t)c->sm_count * 8) need = (uint64_t)c->sm_count * 8;
    LZ_TRY(lz_k_reserve_partials(c, need));
  }
  // Several GPUs: open the run with a one-element NCCL all-reduce. NCCL absorbs any start-up skew between the ranks' hosts
  // (it simply waits), so the watchdog of the in-kernel peer waits only ever covers a peer lost in mid-run.
  if (c->world > 1) LZ_NCCL(lz_nccl()->AllReduce(c->scal + 11, c->scal + 11, 1, ncclDouble, ncclSum, c->comm, c->stream));
  // Small problems are launch-bound (3 launches of ~10-80 us per step): replay the whole k-step loop as one CUDA graph.
  // Single GPU only (the peer exchange bakes per-run sequence numbers into kernel arguments), and not while profiling.
  bool use_graph = c->world == 1 && !c->profiling && c->n_loc <= (4u << 20);
  if (const char* e = getenv("LZ_CUDA_GRAPH")) use_graph = c->world == 1 && !c->profiling && atoi(e) != 0;
  LZ_CUDA(cudaEventRecord(c->ev_a, c->stream));
  bool done = false;
  if (use_graph) {
    const bool hit = c->graph_exec && c->graph_k == k && c->graph_reorth == reorth && c->graph_variant == c->spmv_variant &&
                     c->graph_V == (const double*)basis_ptr(c) && c->graph_epoch == c->epoch;
    if (!hit) {
      drop_graph(c);
      const uint32_t launches0 = c->launches;
      cudaGraph_t g = nullptr;
      if (cudaStreamBeginCapture(c->stream, cudaStreamCaptureModeThreadLocal) == cudaSuccess) {
        const int rc = enqueue_steps(c, k, reorth, fused_push, peer_scalars);
        const cudaError_t ce = cudaStreamEndCapture(c->stream, &g);
        if (rc == LZ_OK && ce == cudaSuccess && g && cudaGraphInstantiate(&c->graph_exec, g, 0) == cudaSuccess) {
          c->graph_k = k; c->graph_reorth = reorth; c->graph_variant = c->spmv_variant; c->graph_V = (double*)basis_ptr(c); c->graph_epoch = c->epoch;
          c->graph_launches = c->launches - launches0;
        } else {
          c->graph_exec = nullptr;
        }
        if (g) cudaGraphDestroy(g);
        cudaGetLastError();
        c->launches = launches0;
      }
    }
    if (c->graph_exec && cudaGraphLaunch(c->graph_exec, c->stream) == cudaSuccess) {
      c->launches += c->graph_launches;
      done = true;
    } else {
      cudaGetLastError();
      drop_graph(c);
    }
  }
  if (!done) LZ_TRY(enqueue_steps(c, k, reorth, fused_push, peer_scalars));
  LZ_CUDA(cudaEventRecord(c->ev_b, c->stream));
  c->k_done = k;
  c->run_serial++;
  c->lagged_done = c->lagged_run;
  c->reorth_done = reorth;
  c->have_tridiag = true;
  c->have_coef = c->have_ans = false;
  c->tm.spmv_launches = k;
  return LZ_OK;
}

extern "C" int lz_get_tridiag(lz_ctx* c, double* alpha_out, double* beta_out) {
  if (!c) return lz_fail(LZ_ERR_ARG, "null ctx");
  if (!c->have_tridiag) return lz_fail(LZ_ERR_ARG, "no decomposition available");
  LZ_TRY(set_dev(c));
  if (alpha_out) LZ_CUDA(cudaMemcpyAsync(alpha_out, c->alpha, c->k_done * 8, cudaMemcpyDeviceToHost, c->stream));
  if (beta_out && c->k_done > 1) LZ_CUDA(cudaMemcpyAsync(beta_out, c->beta, (c->k_done - 1) * 8, cudaMemcpyDeviceToHost, c->stream));
  LZ_CUDA(cudaStreamSynchronize(c->stream));
  if (alpha_out)
    for (uint32_t i = 0; i < c->k_done; i++)
      if (!isfinite(alpha_out[i])) return lz_fail(LZ_ERR_NUMERIC, "alpha[%u] is not finite (Lanczos breakdown: a beta was 0)", i);
  return LZ_OK;
}

extern "C" int lz_tridiag_expv(lz_ctx* c) {
  if (!c) return lz_fail(LZ_ERR_ARG, "null ctx");
  if (!c->have_tridiag) return lz_fail(LZ_ERR_ARG, "lz_lanczos_run must be called before lz_tridiag_expv");
  LZ_TRY(set_dev(c));
  LZ_CUDA(cudaEventRecord(c->ev_e0, c->stream));
  LZ_TRY(lz_k_tridiag_expv(c, c->k_done));
  LZ_CUDA(cudaEventRecord(c->ev_e1, c->stream));
  c->have_coef = true;
  c->have_ans = false;
  return LZ_OK;
}

extern "C" int lz_get_eigen(lz_ctx* c, double* eigvals_out, double* eigvecs_out, double* coeff_out) {
  if (!c) return lz_fail(LZ_ERR_ARG, "null ctx");
  if (!c->have_coef) return lz_fail(LZ_ERR_ARG, "lz_tridiag_expv must be called first");
  LZ_TRY(set_dev(c));
  const uint32_t k = c->k_done;
  int st = 0;
  if (eigvals_out) LZ_CUDA(cudaMemcpyAsync(eigvals_out, c->eigvals, k * 8, cudaMemcpyDeviceToHost, c->stream));
  if (eigvecs_out) LZ_CUDA(cudaMemcpyAsync(eigvecs_out, c->eigvecs, (uint64_t)k * k * 8, cudaMemcpyDeviceToHost, c->stream));
  if (coeff_out) LZ_CUDA(cudaMemcpyAsync(coeff_out, c->coef, k * 8, cudaMemcpyDeviceToHost, c->stream));
  LZ_CUDA(cudaMemcpyAsync(&st, c->status, sizeof(int), cudaMemcpyDeviceToHost, c->stream));
  LZ_CUDA(cudaStreamSynchronize(c->stream));
  if (st & 0x3FFFFFFF) return lz_fail(LZ_ERR_NUMERIC, "tridiagonal eigensolver: eigenvalue %d did not converge", (st & 0x3FFFFFFF) - 1);
  if (st & kStatusIndefinite) return lz_fail(LZ_ERR_NUMERIC, kIndefiniteMsg);
  if (st & 0x40000000) return lz_fail(LZ_ERR_NUMERIC, "coefficient vector is not finite (exp of a Ritz value overflowed, or breakdown)");
  return LZ_OK;
}

// A-posteriori convergence estimate (the author's own recommendation, writeup section 11): with an orthonormal basis,
// || y_k - y_k' ||_2 = || c_k - [c_k'; 0] ||_2, so the change of the answer between Krylov dimensions k' < k costs two
// k x k eigen-solves and no pass over the basis.
namespace {
// Under LZ_MATFUN_EXP_SCALED every block uses the shift of the full k x k solve (which runs first), so all c_k' carry the same
// factor e^{-ls} and the relative change is the unscaled one; by interlacing no leading block has a larger t*theta.
struct CoefSolver {   // scratch for solves of leading blocks of the current tridiagonal; nothing of the ctx's result is touched
  lz_ctx* c;
  uint32_t k;
  double *ev = nullptr, *evec = nullptr, *work = nullptr, *coef = nullptr, *ls = nullptr;
  int* st = nullptr;
  CoefSolver(lz_ctx* c_, uint32_t k_) : c(c_), k(k_) {}
  ~CoefSolver() { cudaFree(ev); cudaFree(evec); cudaFree(work); cudaFree(coef); cudaFree(ls); cudaFree(st); }
  int init() {
    LZ_CUDA(cudaMalloc((void**)&ev, k * 8)); LZ_CUDA(cudaMalloc((void**)&evec, (size_t)k * k * 8));
    LZ_CUDA(cudaMalloc((void**)&work, (size_t)k * k * 8)); LZ_CUDA(cudaMalloc((void**)&coef, k * 8));
    LZ_CUDA(cudaMalloc((void**)&ls, 8)); LZ_CUDA(cudaMalloc((void**)&st, sizeof(int)));
    return LZ_OK;
  }
  int solve(uint32_t kk, std::vector<double>& out) {   // out = c_kk (kk entries); solve(k) first
    out.assign(kk, 0.0);
    int sth = 0;
    LZ_TRY(lz_k_tridiag_expv_into(c, kk, ev, evec, work, coef, st, kk == k ? nullptr : ls, kk == k ? ls : nullptr));
    LZ_CUDA(cudaMemcpyAsync(out.data(), coef, kk * 8, cudaMemcpyDeviceToHost, c->stream));
    LZ_CUDA(cudaMemcpyAsync(&sth, st, sizeof(int), cudaMemcpyDeviceToHost, c->stream));
    LZ_CUDA(cudaStreamSynchronize(c->stream));
    if (sth & kStatusIndefinite) return lz_fail(LZ_ERR_NUMERIC, kIndefiniteMsg);
    if (sth) return lz_fail(LZ_ERR_NUMERIC, "tridiagonal solve of the leading %u x %u block failed or overflowed (status %d)", kk, kk, sth);
    return LZ_OK;
  }
};
double rel_change(const std::vector<double>& a, const std::vector<double>& b) {   // || a - [b; 0] || / || a ||
  double num = 0.0, den = 0.0;
  for (size_t i = 0; i < a.size(); i++) {
    const double d = a[i] - (i < b.size() ? b[i] : 0.0);
    num += d * d;
    den += a[i] * a[i];
  }
  return den > 0.0 ? sqrt(num / den) : 0.0;
}
}  // namespace

extern "C" int lz_estimate_change(lz_ctx* c, uint32_t k_prev, double* rel_out) {
  if (!c || !rel_out) return lz_fail(LZ_ERR_ARG, "null argument");
  if (!c->have_tridiag) return lz_fail(LZ_ERR_ARG, "lz_lanczos_run must be called before lz_estimate_change");
  const uint32_t k = c->k_done;
  if (k_prev < 1 || k_prev >= k) return lz_fail(LZ_ERR_ARG, "k_prev must be in [1, %u)", k);
  LZ_TRY(set_dev(c));
  CoefSolver sv(c, k);
  LZ_TRY(sv.init());
  std::vector<double> a, b;
  LZ_TRY(sv.solve(k, a));
  LZ_TRY(sv.solve(k_prev, b));
  *rel_out = rel_change(a, b);
  return LZ_OK;
}

// Smallest Krylov dimension that would have sufficed: scans k' = k-1, k-2, ... while the estimated change of the answer
// between k' and k stays <= tol, so every dimension from *k_out up to k meets the tolerance. *k_out == k means that not even
// k-1 steps reproduce the k-step answer to tol, i.e. convergence at k is not demonstrated; *est_out is the estimate at
// max(*k_out, 1) .. or at k-1 in that case. Costs (k - *k_out + 2) small solves on the device and no pass over the basis.
extern "C" int lz_choose_k(lz_ctx* c, double tol, uint32_t* k_out, double* est_out) {
  if (!c || !k_out) return lz_fail(LZ_ERR_ARG, "null argument");
  if (!(tol > 0.0)) return lz_fail(LZ_ERR_ARG, "tol must be positive");
  if (!c->have_tridiag) return lz_fail(LZ_ERR_ARG, "lz_lanczos_run must be called before lz_choose_k");
  const uint32_t k = c->k_done;
  LZ_TRY(set_dev(c));
  *k_out = k;
  if (est_out) *est_out = 0.0;
  if (k < 2) return LZ_OK;
  CoefSolver sv(c, k);
  LZ_TRY(sv.init());
  std::vector<double> a, b;
  LZ_TRY(sv.solve(k, a));
  for (uint32_t kp = k - 1; kp >= 1; kp--) {
    LZ_TRY(sv.solve(kp, b));
    const double est = rel_change(a, b);
    if (est > tol) {
      if (kp == k - 1 && est_out) *est_out = est;
      break;
    }
    *k_out = kp;
    if (est_out) *est_out = est;
  }
  return LZ_OK;
}

extern "C" int lz_multout(lz_ctx* c) {
  if (!c) return lz_fail(LZ_ERR_ARG, "null ctx");
  if (!c->have_coef) return lz_fail(LZ_ERR_ARG, "lz_tridiag_expv must be called before lz_multout");
  LZ_TRY(set_dev(c));
  LZ_CUDA(cudaEventRecord(c->ev_m0, c->stream));
  const double* coef = c->coef;
  if (c->lagged_done) {   // rows 1.. of V are unnormalised: fold 1/||u_j|| into the coefficients
    LZ_TRY(lz_k_coef_scale(c, c->coef, c->norm2v, c->k_done, c->hcoef));
    coef = c->hcoef;
  }
  LZ_TRY(lz_k_combine(c, basis_ptr(c), c->basis_f32, c->k_done, coef, 1.0, nullptr, c->ans, nullptr));
  LZ_CUDA(cudaEventRecord(c->ev_m1, c->stream));
  c->have_ans = true;
  return LZ_OK;
}

static int gather_to_host(lz_ctx* c, const double* local, double* host_out, const double* norm2_div = nullptr) {
  // local [n_loc] (new order, this rank's slice) -> host [n] original order, on every rank
  const double* full = local;
  if (c->world > 1) {
    LZ_TRY(lz_k_spread(c, local, c->gfull));   // not xfull: a faster peer may already be pushing the next run's q_0 there
    LZ_TRY(allgather_chunks(c, c->gfull, false));
    full = c->gfull;
  }
  if (host_out) {   // ranks that do not need the vector on the host still take part in the gather above
    LZ_TRY(lz_k_permute_out(c, full, c->xstage));
    if (norm2_div) LZ_TRY(lz_k_div_sqrt(c, c->xstage, c->n, norm2_div));
    LZ_CUDA(cudaMemcpyAsync(host_out, c->xstage, c->n * 8, cudaMemcpyDeviceToHost, c->stream));
  }
  LZ_CUDA(cudaStreamSynchronize(c->stream));
  return LZ_OK;
}

extern "C" int lz_get_ans(lz_ctx* c, double* ans_host) {
  if (!c || (!ans_host && c->world == 1)) return lz_fail(LZ_ERR_ARG, "null argument");
  if (!c->have_ans) return lz_fail(LZ_ERR_ARG, "lz_multout must be called before lz_get_ans");
  LZ_TRY(set_dev(c));
  return gather_to_host(c, c->ans, ans_host);
}

// ---- top Ritz pairs -----------------------------------------------------------------------------------------------------
static bool ritz_valid(const lz_ctx* c) { return c->have_tridiag && c->ritz_m && c->ritz_run == c->run_serial; }

// Ritz pairs of the last run, checked against A itself: a k x k solve into scratch (the ctx's coefficients stay as they are), one
// pass over the basis for all m vectors, then per vector an SpMV for the Rayleigh quotient and a combine for the true residual.
// The Collatz-Wielandt SpMV on weights built from y_0 bounds lambda_max from above. Outside the Lanczos loop, so the scalars of
// several GPUs are joined with NCCL.
extern "C" int lz_ritz(lz_ctx* c, uint32_t m) {
  if (!c) return lz_fail(LZ_ERR_ARG, "null ctx");
  if (!c->have_tridiag) return lz_fail(LZ_ERR_ARG, "lz_lanczos_run must be called before lz_ritz");
  const uint32_t k = c->k_done;
  if (m < 1 || m > LZ_RITZ_MAX || m > k) return lz_fail(LZ_ERR_ARG, "lz_ritz: m = %u must be in [1, min(%d, k = %u)]", m, LZ_RITZ_MAX, k);
  LZ_TRY(set_dev(c));
  c->ritz_m = 0;
  c->have_ans = false;   // ans receives y_0
  const uint32_t M = m == 1 ? 1 : m <= 2 ? 2 : m <= 4 ? 4 : m <= 8 ? 8 : 16;
  if (c->ritz_rows < M) {
    LZ_CUDA(cudaStreamSynchronize(c->stream));
    cudaFree(c->ritz_R); c->ritz_R = nullptr; c->ritz_rows = 0;
    if (cudaMalloc((void**)&c->ritz_R, (size_t)M * c->ldv * 8) != cudaSuccess) {
      cudaGetLastError();
      return lz_fail(LZ_ERR_ALLOC, "cannot allocate %u Ritz vectors of %llu doubles", M, (unsigned long long)c->ldv);
    }
    c->ritz_rows = M;
  }
  CoefSolver sv(c, k);
  LZ_TRY(sv.init());
  // scalars [0,16) ||y_j||^2, [16,32) sum y_j, [32,48) theta, [48,64) rho, [64,80) r^2, [80] max|y_0|, [81] Collatz-Wielandt max,
  // [82] unused dot; then W [k][16] and the combine's per-CTA partials
  struct Scratch { double* p = nullptr; ~Scratch() { cudaFree(p); } } aux;
  const size_t n_part = (size_t)2 * LZ_RITZ_MAX * 8 * c->sm_count;
  LZ_CUDA(cudaMalloc((void**)&aux.p, (96 + (size_t)k * LZ_RITZ_MAX + n_part) * 8));
  double* s = aux.p;
  double *nrm2 = s, *vsum = s + 16, *theta = s + 32, *rho = s + 48, *r2 = s + 64, *W = s + 96, *part = W + (size_t)k * LZ_RITZ_MAX;
  auto* absmax = reinterpret_cast<unsigned long long*>(s + 80);
  auto* cwmax = reinterpret_cast<unsigned long long*>(s + 81);
  LZ_CUDA(cudaMemsetAsync(s, 0, 96 * 8, c->stream));
  LZ_TRY(lz_k_tridiag_expv_into(c, k, sv.ev, sv.evec, sv.work, sv.coef, sv.st, nullptr, nullptr));
  LZ_TRY(lz_k_ritz_select(c, k, m, M, sv.ev, sv.evec, c->lagged_done ? c->norm2v : nullptr, W, theta));
  double* R = c->ritz_R;
  if (M == 1) {
    LZ_TRY(lz_k_combine(c, basis_ptr(c), c->basis_f32, k, W, 1.0, nullptr, R, nrm2));
    LZ_TRY(lz_k_vsum(c, R, c->n_loc, part, vsum));
  } else {
    LZ_TRY(lz_k_ritz_combine(c, basis_ptr(c), c->basis_f32, k, M, W, R, part, nrm2, vsum));
  }
  LZ_TRY(allreduce_sum(c, s, 32));
  LZ_TRY(lz_k_ritz_scale(c, R, m, nrm2, vsum, absmax));
  if (c->world > 1) LZ_NCCL(lz_nccl()->AllReduce(s + 80, s + 80, 1, ncclDouble, ncclMax, c->comm, c->stream));
  // with several GPUs the SpMV reads the gathered vector: gfull, not xfull (a faster peer may already push its next q_0 there);
  // one GPU has no gathered vector and xfull is free for the Collatz-Wielandt weights
  double* zfull = c->world > 1 ? c->gfull : c->xfull;
  for (uint32_t j = 0; j < m; j++) {
    const double* y = R + (uint64_t)j * c->ldv;
    const double* yg = y;
    if (c->world > 1) {
      LZ_TRY(lz_k_spread(c, y, c->gfull));
      LZ_TRY(allgather_chunks(c, c->gfull, false));
      yg = c->gfull;
    }
    LZ_TRY(lz_k_spmv_dot(c, yg, y, c->w, rho + j));                                   // w = A y_j, rho_j = y_j . w
    LZ_TRY(allreduce_sum(c, rho + j, 1));
    LZ_TRY(lz_k_combine(c, y, false, 1, rho + j, -1.0, c->w, c->w, r2 + j));          // ||A y_j - rho_j y_j||^2
    LZ_TRY(allreduce_sum(c, r2 + j, 1));
    if (j == 0) {                                                                     // lambda_max <= max_i (A z)_i / z_i
      LZ_TRY(lz_k_cw_z(c, yg, zfull, c->n_loc * (uint64_t)c->world, s + 80, LZ_CW_FLOOR));
      LZ_TRY(lz_k_spmv_dot(c, zfull, y, c->w, s + 82));
      LZ_TRY(lz_k_cw_bound(c, c->w, zfull, cwmax));
      if (c->world > 1) LZ_NCCL(lz_nccl()->AllReduce(s + 81, s + 81, 1, ncclDouble, ncclMax, c->comm, c->stream));
    }
  }
  LZ_CUDA(cudaMemcpyAsync(c->ans, R, c->n_loc * 8, cudaMemcpyDeviceToDevice, c->stream));
  double h[82];
  int st = 0;
  LZ_CUDA(cudaMemcpyAsync(h, s, sizeof(h), cudaMemcpyDeviceToHost, c->stream));
  LZ_CUDA(cudaMemcpyAsync(&st, sv.st, sizeof(int), cudaMemcpyDeviceToHost, c->stream));
  LZ_CUDA(cudaStreamSynchronize(c->stream));
  // bits 30 and 31 belong to the matrix function (overflow, indefinite resolvent): the eigenpairs do not depend on them
  if (st & 0x3FFFFFFF) return lz_fail(LZ_ERR_NUMERIC, "tridiagonal eigensolver: eigenvalue %d did not converge", (st & 0x3FFFFFFF) - 1);
  for (uint32_t j = 0; j < m; j++) {
    if (!(h[j] > 0.0) || !isfinite(h[j])) return lz_fail(LZ_ERR_NUMERIC, "Ritz vector %u is zero or not finite (||V z||^2 = %g)", j, h[j]);
    if (!isfinite(h[32 + j]) || !isfinite(h[48 + j]) || !isfinite(h[64 + j]))
      return lz_fail(LZ_ERR_NUMERIC, "Ritz pair %u is not finite (theta %g, rho %g, r^2 %g)", j, h[32 + j], h[48 + j], h[64 + j]);
  }
  // (A z)_i is a sum of deg_i exact products: computed ratio >= true ratio * (1 - (deg_i + 1) 2^-53); the allowance covers it and the
  // rounding of the product below
  const double cw = h[81];
  if (!isfinite(cw)) return lz_fail(LZ_ERR_NUMERIC, "Collatz-Wielandt bound is not finite");
  const double ulp = 0x1p-52, D = (double)c->max_degree, N = (double)c->n;
  const double hi = cw * (1.0 + (D + 2.0) * ulp);
  // Rounding allowance of the intervals and of lo (u = 2^-53, y the stored Ritz vector, w^ the computed A y, lambda_max <= hi = ||A||_2):
  //  - the SpMV: |w^ - A y| <= gamma_D A|y| entry-wise, so ||w^ - A y|| <= gamma_D hi ||y||;
  //  - the residual combine and its sum of squares: ||w^ - rho y|| <= r^ (1 + gamma_n + 3u) + 2u |rho| ||y||;
  //  - the dot product: |rho - y^T A y| <= c lambda_max ||y||^2 with c = gamma_n (1 + gamma_D) + gamma_D (|y|^T A |y| <= lambda_max ||y||^2);
  //  - the norm: | ||y||^2 - 1 | <= gamma_n + 8u after k_ritz_scale.
  // Krylov-Bogoliubov holds for any centre: some eigenvalue lies within ||A y - rho y|| / ||y|| of rho, which the radius below bounds
  // (with 2u |rho| more, so that rho -/+ r rounded to fp64 still encloses it). For lo, the error of rho is relative to lambda_max, not
  // to rho: y^T A y <= lambda_max ||y||^2 gives rho <= lambda_max ||y||^2 (1 + c) <= lambda_max (1 + gamma_n + 8u)(1 + c), so
  // lambda_max >= rho / ((1 + gamma_n + 8u)(1 + c)) >= rho (1 - (2n + D + 24) 2^-52) when rho > 0; a non-negative A has
  // lambda_max >= 0 >= rho otherwise. The extra units absorb the rounding of these formulas.
  for (uint32_t j = 0; j < m; j++) {
    c->ritz_theta[j] = h[32 + j];
    c->ritz_rho[j] = h[48 + j];
    c->ritz_res[j] = sqrt(h[64 + j]) * (1.0 + (2.0 * N + 24.0) * ulp) + (D + 8.0) * ulp * hi;
  }
  const double rho0 = c->ritz_rho[0];
  c->ritz_lo = rho0 > 0.0 ? rho0 * (1.0 - (2.0 * N + D + 24.0) * ulp) : rho0;
  c->ritz_hi = hi;
  c->ritz_m = m;
  c->ritz_run = c->run_serial;
  c->have_ans = true;
  return LZ_OK;
}

extern "C" int lz_get_ritz(lz_ctx* c, double* theta_out, double* rayleigh_out, double* resid_out) {
  if (!c) return lz_fail(LZ_ERR_ARG, "null ctx");
  if (!ritz_valid(c)) return lz_fail(LZ_ERR_ARG, "lz_ritz must be called after the last lz_lanczos_run");
  for (uint32_t j = 0; j < c->ritz_m; j++) {
    if (theta_out) theta_out[j] = c->ritz_theta[j];
    if (rayleigh_out) rayleigh_out[j] = c->ritz_rho[j];
    if (resid_out) resid_out[j] = c->ritz_res[j];
  }
  return LZ_OK;
}

extern "C" int lz_get_ritz_vector(lz_ctx* c, uint32_t j, double* y_host) {
  if (!c || (!y_host && c->world == 1)) return lz_fail(LZ_ERR_ARG, "null argument");
  if (!ritz_valid(c)) return lz_fail(LZ_ERR_ARG, "lz_ritz must be called after the last lz_lanczos_run");
  if (j >= c->ritz_m) return lz_fail(LZ_ERR_ARG, "Ritz vector %u not available (%u computed)", j, c->ritz_m);
  LZ_TRY(set_dev(c));
  return gather_to_host(c, c->ritz_R + (uint64_t)j * c->ldv, y_host);
}

extern "C" int lz_spectral_radius_bounds(lz_ctx* c, double* lo_out, double* hi_out) {
  if (!c || !lo_out || !hi_out) return lz_fail(LZ_ERR_ARG, "null argument");
  if (!ritz_valid(c)) return lz_fail(LZ_ERR_ARG, "lz_ritz must be called after the last lz_lanczos_run");
  *lo_out = c->ritz_lo;
  *hi_out = c->ritz_hi;
  return LZ_OK;
}

static int expv_impl(lz_ctx* c, const double* x_host, uint32_t k, int reorth, double* ans_host, int root);
extern "C" int lz_expv_host(lz_ctx* c, const double* x_host, uint32_t k, int reorth, double* ans_host) {
  return expv_impl(c, x_host, k, reorth, ans_host, -1);
}
// One caller holds x and wants e^A x: only rank `root` touches host memory (x_host / ans_host are ignored elsewhere).
extern "C" int lz_expv_host_root(lz_ctx* c, const double* x_host, uint32_t k, int reorth, double* ans_host, int root) {
  if (!c || root < 0 || root >= c->world) return lz_fail(LZ_ERR_ARG, "bad root");
  return expv_impl(c, c->rank == root ? x_host : nullptr, k, reorth, c->rank == root ? ans_host : nullptr, root);
}
static int expv_impl(lz_ctx* c, const double* x_host, uint32_t k, int reorth, double* ans_host, int root) {
  LZ_TRY(set_start_vector_impl(c, x_host, root));
  LZ_TRY(lz_lanczos_run(c, k, reorth));
  LZ_TRY(lz_tridiag_expv(c));
  LZ_TRY(lz_multout(c));
  LZ_TRY(lz_get_ans(c, ans_host));
  int st = 0;
  LZ_CUDA(cudaMemcpy(&st, c->status, sizeof(int), cudaMemcpyDeviceToHost));
  if (st & 0x3FFFFFFF) return lz_fail(LZ_ERR_NUMERIC, "tridiagonal eigensolver: eigenvalue %d did not converge", (st & 0x3FFFFFFF) - 1);
  if (st & kStatusIndefinite) return lz_fail(LZ_ERR_NUMERIC, kIndefiniteMsg);
  if (st & 0x40000000) return lz_fail(LZ_ERR_NUMERIC, "result is not finite (exp of a Ritz value overflowed, or Lanczos breakdown)");
  return LZ_OK;
}

extern "C" int lz_spmv_host(lz_ctx* c, const double* x_host, double* y_host) {
  if (!c || !x_host || !y_host) return lz_fail(LZ_ERR_ARG, "null argument");
  LZ_TRY(set_dev(c));
  LZ_TRY(ensure_graph_vectors(c));
  const uint64_t n_pad = c->n_loc * (uint64_t)c->world;
  double *xg = nullptr, *y = nullptr, *dummy = nullptr;
  LZ_CUDA(cudaMalloc((void**)&xg, n_pad * 8));
  LZ_CUDA(cudaMalloc((void**)&y, c->ldv * 8));
  LZ_CUDA(cudaMalloc((void**)&dummy, 8));
  int rc = LZ_OK;
  do {
    if (cudaMemcpyAsync(c->xstage, x_host, c->n * 8, cudaMemcpyHostToDevice, c->stream) != cudaSuccess) { rc = lz_fail(LZ_ERR_CUDA, "H2D failed"); break; }
    if ((rc = lz_k_permute_in(c, c->xstage, nullptr, 0, n_pad, xg)) != LZ_OK) break;
    if ((rc = lz_k_spmv_dot(c, xg, xg + (uint64_t)c->rank * c->n_loc, y, dummy)) != LZ_OK) break;
    rc = gather_to_host(c, y, y_host);
  } while (0);
  cudaStreamSynchronize(c->stream);
  cudaFree(xg); cudaFree(y); cudaFree(dummy);
  return rc;
}

extern "C" int lz_get_basis(lz_ctx* c, uint32_t j, double* q_host) {
  if (!c || !q_host) return lz_fail(LZ_ERR_ARG, "null argument");
  if (!c->have_x || j >= (c->have_tridiag ? c->k_done : 1u)) return lz_fail(LZ_ERR_ARG, "basis vector %u not available", j);
  LZ_TRY(set_dev(c));
  // after a lagged-normalisation run rows 1.. hold u_j = ||u_j|| q_j
  const double* row = c->basis_f32 ? c->w : c->V + (uint64_t)j * c->ldv;
  if (c->basis_f32) LZ_TRY(lz_k_convert(c, nullptr, nullptr, c->V32 + (uint64_t)j * c->ldv, c->w, c->n_loc));   // w is scratch between runs
  return gather_to_host(c, row, q_host, (c->lagged_done && c->have_tridiag && j > 0) ? c->norm2v + j : nullptr);
}

extern "C" int lz_set_profiling(lz_ctx* c, int on) {
  if (!c) return lz_fail(LZ_ERR_ARG, "null ctx");
  c->profiling = on != 0;
  return LZ_OK;
}

// Measurement hook: device-side timeline of the kernels' internal phases (start, peer wait over, push done, end).
// cap_events > 0 switches the timeline on (and clears it); cap_events == 0 reads it back: out receives (tag, ns) pairs.
extern "C" int lz_debug_trace(lz_ctx* c, uint32_t cap_events, uint64_t* out, uint32_t out_cap_events, uint32_t* count_out) {
  if (!c) return lz_fail(LZ_ERR_ARG, "null ctx");
  LZ_TRY(set_dev(c));
  if (cap_events) {
    if (c->trace_cap < cap_events) {
      LZ_CUDA(cudaStreamSynchronize(c->stream));
      cudaFree(c->trace_buf); c->trace_buf = nullptr; c->trace_cap = 0;
      LZ_CUDA(cudaMalloc((void**)&c->trace_buf, (2 + 2 * (size_t)cap_events) * 8));
      c->trace_cap = cap_events;
    }
    const unsigned long long head[2] = {0ull, cap_events};
    LZ_CUDA(cudaMemcpyAsync(c->trace_buf, head, sizeof(head), cudaMemcpyHostToDevice, c->stream));
    LZ_TRY(lz_k_set_trace(c, c->trace_buf));
    LZ_CUDA(cudaStreamSynchronize(c->stream));
    return LZ_OK;
  }
  if (!c->trace_buf) return lz_fail(LZ_ERR_ARG, "trace is not on");
  LZ_TRY(lz_k_set_trace(c, nullptr));
  unsigned long long head[2] = {0, 0};
  LZ_CUDA(cudaMemcpyAsync(head, c->trace_buf, sizeof(head), cudaMemcpyDeviceToHost, c->stream));
  LZ_CUDA(cudaStreamSynchronize(c->stream));
  uint32_t cnt = (uint32_t)(head[0] < head[1] ? head[0] : head[1]);
  if (cnt > out_cap_events) cnt = out_cap_events;
  if (out && cnt) LZ_CUDA(cudaMemcpy(out, c->trace_buf + 2, (size_t)cnt * 16, cudaMemcpyDeviceToHost));
  if (count_out) *count_out = cnt;
  return LZ_OK;
}

extern "C" int lz_exchange_info(lz_ctx* c, int* mode_out, double* need_frac_out) {
  if (!c || !mode_out) return lz_fail(LZ_ERR_ARG, "null argument");
  if (c->world > 1 && !c->w) return lz_fail(LZ_ERR_ARG, "the exchange is set up by the first lz_set_start_vector / lz_expv_host");
  *mode_out = c->world == 1 ? LZ_EXCHANGE_NONE : !c->peer_push ? LZ_EXCHANGE_NCCL : c->sparse_push ? LZ_EXCHANGE_PEER_SPARSE : LZ_EXCHANGE_PEER_DENSE;
  if (need_frac_out) *need_frac_out = (c->world > 1 && c->peer_push) ? c->push_need_frac : 1.0;
  return LZ_OK;
}

extern "C" int lz_timings_get(lz_ctx* c, lz_timings* out) {
  if (!c || !out) return lz_fail(LZ_ERR_ARG, "null argument");
  LZ_TRY(set_dev(c));
  LZ_CUDA(cudaStreamSynchronize(c->stream));
  float ms = 0.f;
  if (c->have_tridiag && cudaEventElapsedTime(&ms, c->ev_a, c->ev_b) == cudaSuccess) c->tm.lanczos_ms = ms;
  if (c->have_coef && cudaEventElapsedTime(&ms, c->ev_e0, c->ev_e1) == cudaSuccess) c->tm.tridiag_ms = ms;
  if (c->have_ans && cudaEventElapsedTime(&ms, c->ev_m0, c->ev_m1) == cudaSuccess) c->tm.multout_ms = ms;
  double sum[4] = {0, 0, 0, 0};
  int cnt[4] = {0, 0, 0, 0};
  for (const Mark& m : g_marks) {
    if (cudaEventElapsedTime(&ms, m.a, m.b) == cudaSuccess) { sum[m.kind] += ms; cnt[m.kind]++; }
  }
  cudaGetLastError();
  const uint32_t steps = c->k_done ? c->k_done : 1;
  c->tm.spmv_ms_avg = cnt[0] ? (float)(sum[0] / cnt[0]) : 0.f;
  c->tm.update_ms_avg = (float)(sum[1] / steps);
  c->tm.comm_ms_avg = (float)(sum[2] / steps);
  c->tm.reorth_ms_total = (float)sum[3];
  c->tm.kernel_launches = c->launches;
  {
    unsigned int sp = 0;
    if (cudaMemcpy(&sp, c->status + 2, sizeof(sp), cudaMemcpyDeviceToHost) == cudaSuccess) c->tm.reorth_second_passes = sp;
  }
  *out = c->tm;
  return LZ_OK;
}

extern "C" int lz_timer_start(lz_ctx* c) {
  if (!c) return lz_fail(LZ_ERR_ARG, "null ctx");
  LZ_TRY(set_dev(c));
  LZ_CUDA(cudaEventRecord(c->ev_t0, c->stream));
  return LZ_OK;
}
extern "C" int lz_timer_stop(lz_ctx* c, float* ms_out) {
  if (!c || !ms_out) return lz_fail(LZ_ERR_ARG, "null argument");
  LZ_TRY(set_dev(c));
  LZ_CUDA(cudaEventRecord(c->ev_t1, c->stream));
  LZ_CUDA(cudaEventSynchronize(c->ev_t1));
  LZ_CUDA(cudaEventElapsedTime(ms_out, c->ev_t0, c->ev_t1));
  return LZ_OK;
}

extern "C" int lz_flush_l2(lz_ctx* c) {
  if (!c) return lz_fail(LZ_ERR_ARG, "null ctx");
  LZ_TRY(set_dev(c));
  if (!c->flush_buf) {
    c->flush_bytes = 512ull << 20;   // 4x the 126 MB L2
    LZ_CUDA(cudaMalloc(&c->flush_buf, c->flush_bytes));
  }
  LZ_CUDA(cudaMemsetAsync(c->flush_buf, 0, c->flush_bytes, c->stream));
  return LZ_OK;
}
