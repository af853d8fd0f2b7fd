"""ctypes binding of include/lz.h. One method per C entry point; numpy arrays in, numpy arrays out."""
import ctypes as C
import os
import re

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
lib_path = os.path.join(_HERE, "csrc", "liblzb200.so")
_HEADER = os.path.join(_HERE, "..", "include", "lz.h")

if not os.path.exists(lib_path):
    raise ImportError(
        f"{lib_path} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
        "(there is no Python/CPU fallback for the CUDA library)")
lib = C.CDLL(lib_path)

GRAPH_ER, GRAPH_RMAT, GRAPH_BAND = 1, 2, 3
REORTH_NONE, REORTH_FULL = 0, 1
EXCHANGE_NONE, EXCHANGE_NCCL, EXCHANGE_PEER_DENSE, EXCHANGE_PEER_SPARSE = 0, 1, 2, 3
SPMV_AUTO, SPMV_VECTOR, SPMV_WARP = 0, 1, 2
BASIS_F64, BASIS_F32 = 0, 1
MATFUN_EXP, MATFUN_EXP_SCALED, MATFUN_RESOLVENT = 0, 1, 2
RITZ_MAX = 16
CW_FLOOR = 1e-6
NCCL_UID_BYTES = 128


class LzError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"lz error {code}: {msg}")
        self.code = code


class GraphSpec(C.Structure):
    _fields_ = [("kind", C.c_uint32), ("scale", C.c_uint32), ("n", C.c_uint64), ("param_a", C.c_uint64),
                ("seed", C.c_uint64), ("rmat_a", C.c_double), ("rmat_b", C.c_double), ("rmat_c", C.c_double)]

    @staticmethod
    def er(n, m, seed):
        return GraphSpec(GRAPH_ER, 0, n, m, seed, 0, 0, 0)

    @staticmethod
    def rmat(scale, edge_factor, seed, a=0.0, b=0.0, c=0.0):
        return GraphSpec(GRAPH_RMAT, scale, 0, edge_factor, seed, a, b, c)

    @staticmethod
    def band(n, seed):
        return GraphSpec(GRAPH_BAND, 0, n, 0, seed, 0, 0, 0)


class GraphInfo(C.Structure):
    _fields_ = [("n", C.c_uint64), ("nnz", C.c_uint64), ("n_local", C.c_uint64), ("nnz_local", C.c_uint64),
                ("max_degree", C.c_uint32), ("pad_", C.c_uint32), ("empty_rows", C.c_uint64)]


class Timings(C.Structure):
    _fields_ = [("lanczos_ms", C.c_float), ("tridiag_ms", C.c_float), ("multout_ms", C.c_float),
                ("spmv_ms_avg", C.c_float), ("update_ms_avg", C.c_float), ("comm_ms_avg", C.c_float),
                ("reorth_ms_total", C.c_float), ("spmv_launches", C.c_uint32), ("kernel_launches", C.c_uint32),
                ("reorth_second_passes", C.c_uint32)]


_P = C.POINTER
_u32p, _u64p, _f64p = _P(C.c_uint32), _P(C.c_uint64), _P(C.c_double)
_ctx = C.c_void_p


def _sig(name, *argtypes, restype=C.c_int):
    f = getattr(lib, name)
    f.argtypes = list(argtypes)
    f.restype = restype
    return f


_sig("lz_last_error", restype=C.c_char_p)
_sig("lz_version")
_sig("lz_free_host", C.c_void_p, restype=None)
_sig("lz_graph_generate_host", _P(GraphSpec), _u64p, _u64p, _P(_u32p), _P(_u32p))
_sig("lz_csr_from_edges", C.c_uint64, C.c_uint64, _u32p, _u32p, _u64p, _P(_u32p), _P(_u32p))
_sig("lz_csr_read_text", C.c_char_p, _u64p, _u64p, _P(_u32p), _P(_u32p))
_sig("lz_csr_write_text", C.c_char_p, C.c_uint64, _u32p, _u32p)
_sig("lz_csr_read_bin", C.c_char_p, _u64p, _u64p, _P(_u32p), _P(_u32p))
_sig("lz_csr_write_bin", C.c_char_p, C.c_uint64, _u32p, _u32p)
_sig("lz_device_count", _P(C.c_int))
_sig("lz_create", C.c_int, _P(_ctx))
_sig("lz_nccl_unique_id", C.c_void_p)
_sig("lz_create_dist", C.c_int, C.c_int, C.c_int, C.c_void_p, _P(_ctx))
_sig("lz_destroy", _ctx)
_sig("lz_sync", _ctx)
_sig("lz_csr_upload", _ctx, C.c_uint64, _u32p, _u32p)
_sig("lz_graph_generate", _ctx, _P(GraphSpec))
_sig("lz_graph_info_get", _ctx, _P(GraphInfo))
_sig("lz_csr_download", _ctx, _u32p, _u32p)
_sig("lz_set_start_vector", _ctx, _f64p)
_sig("lz_lanczos_run", _ctx, C.c_uint32, C.c_int)
_sig("lz_get_tridiag", _ctx, _f64p, _f64p)
_sig("lz_tridiag_expv", _ctx)
_sig("lz_get_eigen", _ctx, _f64p, _f64p, _f64p)
_sig("lz_estimate_change", _ctx, C.c_uint32, _P(C.c_double))
_sig("lz_choose_k", _ctx, C.c_double, _P(C.c_uint32), _P(C.c_double))
_sig("lz_multout", _ctx)
_sig("lz_get_ans", _ctx, _f64p)
_sig("lz_top_k", _ctx, C.c_uint32, _u32p, _f64p, _u32p)
_sig("lz_expv_host", _ctx, _f64p, C.c_uint32, C.c_int, _f64p)
_sig("lz_expv_host_root", _ctx, _f64p, C.c_uint32, C.c_int, _f64p, C.c_int)
_sig("lz_set_start_vector_root", _ctx, _f64p, C.c_int)
_sig("lz_spmv_host", _ctx, _f64p, _f64p)
_sig("lz_get_basis", _ctx, C.c_uint32, _f64p)
_sig("lz_set_spmv_variant", _ctx, C.c_int)
_sig("lz_set_basis_precision", _ctx, C.c_int)
_sig("lz_set_matfun", _ctx, C.c_int, C.c_double)
_sig("lz_get_matfun_scale", _ctx, _P(C.c_double))
_sig("lz_ritz", _ctx, C.c_uint32)
_sig("lz_get_ritz", _ctx, _f64p, _f64p, _f64p)
_sig("lz_get_ritz_vector", _ctx, C.c_uint32, _f64p)
_sig("lz_spectral_radius_bounds", _ctx, _P(C.c_double), _P(C.c_double))
_sig("lz_set_profiling", _ctx, C.c_int)
_sig("lz_exchange_info", _ctx, _P(C.c_int), _P(C.c_double))
_sig("lz_timings_get", _ctx, _P(Timings))
_sig("lz_timer_start", _ctx)
_sig("lz_timer_stop", _ctx, _P(C.c_float))
_sig("lz_flush_l2", _ctx)
_sig("lz_debug_trace", _ctx, C.c_uint32, _u64p, C.c_uint32, _u32p)


def _check(rc):
    if rc != 0:
        raise LzError(rc, lib.lz_last_error().decode(errors="replace"))


def header_symbols():
    """Every function name declared in include/lz.h."""
    txt = open(_HEADER).read()
    txt = re.sub(r"/\*.*?\*/", "", txt, flags=re.S)
    return sorted(set(re.findall(r"\b(lz_[a-z0-9_]+)\s*\(", txt)))


def exported_symbols():
    return [s for s in header_symbols() if hasattr(lib, s)]


def _f64(a):
    return a.ctypes.data_as(_f64p)


def _u32(a):
    return a.ctypes.data_as(_u32p)


def _take_csr(n, nnz, ro, ci):
    n, nnz = int(n.value), int(nnz.value)
    row_offset = np.ctypeslib.as_array(ro, shape=(n + 1,)).copy()
    col_idx = np.ctypeslib.as_array(ci, shape=(max(nnz, 1),))[:nnz].copy()
    lib.lz_free_host(ro)
    lib.lz_free_host(ci)
    return n, row_offset, col_idx


def generate_host(spec):
    """Deterministic host generator -> (n, row_offset[n+1] u32, col_idx[nnz] u32). Needs no GPU."""
    n, nnz, ro, ci = C.c_uint64(), C.c_uint64(), _u32p(), _u32p()
    _check(lib.lz_graph_generate_host(C.byref(spec), C.byref(n), C.byref(nnz), C.byref(ro), C.byref(ci)))
    return _take_csr(n, nnz, ro, ci)


def csr_from_edges(n, u, v):
    u, v = np.ascontiguousarray(u, np.uint32), np.ascontiguousarray(v, np.uint32)
    nnz, ro, ci = C.c_uint64(), _u32p(), _u32p()
    _check(lib.lz_csr_from_edges(n, len(u), _u32(u), _u32(v), C.byref(nnz), C.byref(ro), C.byref(ci)))
    return _take_csr(C.c_uint64(n), nnz, ro, ci)


def read_text(path):
    n, nnz, ro, ci = C.c_uint64(), C.c_uint64(), _u32p(), _u32p()
    _check(lib.lz_csr_read_text(os.fsencode(path), C.byref(n), C.byref(nnz), C.byref(ro), C.byref(ci)))
    return _take_csr(n, nnz, ro, ci)


def read_bin(path):
    n, nnz, ro, ci = C.c_uint64(), C.c_uint64(), _u32p(), _u32p()
    _check(lib.lz_csr_read_bin(os.fsencode(path), C.byref(n), C.byref(nnz), C.byref(ro), C.byref(ci)))
    return _take_csr(n, nnz, ro, ci)


def write_text(path, row_offset, col_idx):
    ro, ci = np.ascontiguousarray(row_offset, np.uint32), np.ascontiguousarray(col_idx, np.uint32)
    _check(lib.lz_csr_write_text(os.fsencode(path), len(ro) - 1, _u32(ro), _u32(ci)))


def write_bin(path, row_offset, col_idx):
    ro, ci = np.ascontiguousarray(row_offset, np.uint32), np.ascontiguousarray(col_idx, np.uint32)
    _check(lib.lz_csr_write_bin(os.fsencode(path), len(ro) - 1, _u32(ro), _u32(ci)))


def device_count():
    k = C.c_int(0)
    _check(lib.lz_device_count(C.byref(k)))
    return k.value


def nccl_unique_id():
    buf = C.create_string_buffer(NCCL_UID_BYTES)
    _check(lib.lz_nccl_unique_id(buf))
    return buf.raw


class Context:
    """One GPU (one rank). Mirrors the call order of parallel-final/main.cu:115-127 on the C ABI."""

    def __init__(self, device=0, rank=0, world=1, uid=None):
        self._h = _ctx()
        if world > 1:
            _check(lib.lz_create_dist(device, rank, world, C.c_char_p(uid), C.byref(self._h)))
        else:
            _check(lib.lz_create(device, C.byref(self._h)))
        self.rank, self.world = rank, world

    def close(self):
        if self._h:
            lib.lz_destroy(self._h)
            self._h = _ctx()

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # graph
    def csr_upload(self, row_offset, col_idx):
        ro, ci = np.ascontiguousarray(row_offset, np.uint32), np.ascontiguousarray(col_idx, np.uint32)
        _check(lib.lz_csr_upload(self._h, len(ro) - 1, _u32(ro), _u32(ci)))

    def graph_generate(self, spec):
        _check(lib.lz_graph_generate(self._h, C.byref(spec)))

    def graph_info(self):
        gi = GraphInfo()
        _check(lib.lz_graph_info_get(self._h, C.byref(gi)))
        return gi

    def csr_download(self):
        gi = self.graph_info()
        ro, ci = np.empty(gi.n + 1, np.uint32), np.empty(max(gi.nnz, 1), np.uint32)
        _check(lib.lz_csr_download(self._h, _u32(ro), _u32(ci)))
        return ro, ci[:gi.nnz]

    # hot path
    def set_start_vector(self, x=None):
        if x is None:
            _check(lib.lz_set_start_vector(self._h, None))
        else:
            x = np.ascontiguousarray(x, np.float64)
            assert x.shape == (self.graph_info().n,)
            _check(lib.lz_set_start_vector(self._h, _f64(x)))

    def set_start_vector_root(self, x, root=0):
        """Collective: only `root` passes x (one PCIe upload); the other ranks pass None and receive it over NVLink."""
        xp = None if x is None else _f64(np.ascontiguousarray(x, np.float64))
        _check(lib.lz_set_start_vector_root(self._h, xp, root))

    def lanczos_run(self, k, reorth=REORTH_NONE):
        _check(lib.lz_lanczos_run(self._h, k, reorth))
        self._k = k

    def get_tridiag(self):
        a, b = np.empty(self._k), np.empty(max(self._k - 1, 1))
        _check(lib.lz_get_tridiag(self._h, _f64(a), _f64(b)))
        return a, b[:self._k - 1]

    def tridiag_expv(self):
        _check(lib.lz_tridiag_expv(self._h))

    def get_eigen(self):
        k = self._k
        w, z, c = np.empty(k), np.empty((k, k)), np.empty(k)
        _check(lib.lz_get_eigen(self._h, _f64(w), _f64(z), _f64(c)))
        return w, z, c

    def estimate_change(self, k_prev):
        r = C.c_double(0)
        _check(lib.lz_estimate_change(self._h, k_prev, C.byref(r)))
        return r.value

    def choose_k(self, tol):
        """(k', estimate): smallest Krylov dimension whose answer stays within tol of the last run's, by the estimate."""
        k, est = C.c_uint32(0), C.c_double(0)
        _check(lib.lz_choose_k(self._h, tol, C.byref(k), C.byref(est)))
        return k.value, est.value

    def multout(self):
        _check(lib.lz_multout(self._h))

    def get_ans(self, out=None):
        n = self.graph_info().n
        y = np.empty(n) if out is None else out
        _check(lib.lz_get_ans(self._h, _f64(y)))
        return y

    def top_k(self, m=100):
        """(idx, val): the m largest entries of the last multout result, descending, ties -> lower vertex id."""
        idx, val, cnt = np.empty(m, np.uint32), np.empty(m), C.c_uint32(0)
        _check(lib.lz_top_k(self._h, m, _u32(idx), _f64(val), C.byref(cnt)))
        return idx[:cnt.value], val[:cnt.value]

    def expv_host(self, x, k, reorth=REORTH_NONE, out=None, want_result=True):
        """want_result=False (world > 1 only): this rank takes part but does not copy e^A x to its host."""
        n = self.graph_info().n
        y = None
        if want_result:
            y = np.empty(n) if out is None else out
        xp = None if x is None else _f64(np.ascontiguousarray(x, np.float64))
        _check(lib.lz_expv_host(self._h, xp, k, reorth, _f64(y) if want_result else None))
        self._k = k
        return y

    def expv_host_root(self, x, k, reorth=REORTH_NONE, out=None, root=0):
        """One caller: only `root` passes x and receives e^A x (returns None elsewhere)."""
        if self.rank != root:
            _check(lib.lz_expv_host_root(self._h, None, k, reorth, None, root))
            self._k = k
            return None
        n = self.graph_info().n
        y = np.empty(n) if out is None else out
        x = np.ascontiguousarray(x, np.float64)
        _check(lib.lz_expv_host_root(self._h, _f64(x), k, reorth, _f64(y), root))
        self._k = k
        return y

    # hooks
    def spmv_host(self, x):
        x = np.ascontiguousarray(x, np.float64)
        y = np.empty_like(x)
        _check(lib.lz_spmv_host(self._h, _f64(x), _f64(y)))
        return y

    def get_basis(self, j):
        q = np.empty(self.graph_info().n)
        _check(lib.lz_get_basis(self._h, j, _f64(q)))
        return q

    def set_basis_precision(self, p):
        _check(lib.lz_set_basis_precision(self._h, p))

    def set_matfun(self, kind, param):
        """kind: MATFUN_EXP (e^{pA} x), MATFUN_EXP_SCALED (e^{p(A - sI)} x, see matfun_scale) or MATFUN_RESOLVENT
        ((I - pA)^{-1} x, Katz centrality). Keeps the last Lanczos run: tridiag_expv + multout apply the new function."""
        _check(lib.lz_set_matfun(self._h, kind, param))

    def matfun_scale(self):
        """log of the factor the last tridiag_expv left out: f(A) x = answer * exp(matfun_scale())."""
        r = C.c_double(0)
        _check(lib.lz_get_matfun_scale(self._h, C.byref(r)))
        return r.value

    def ritz(self, m):
        """Top m Ritz pairs of the last Lanczos run -> (theta, rayleigh, resid), largest first. [rayleigh - resid, rayleigh + resid]
        contains an eigenvalue of A. Leaves y_0 (eigenvector centrality) as the answer: get_ans / top_k read it."""
        _check(lib.lz_ritz(self._h, m))
        th, rho, res = np.empty(m), np.empty(m), np.empty(m)
        _check(lib.lz_get_ritz(self._h, _f64(th), _f64(rho), _f64(res)))
        return th, rho, res

    def ritz_vector(self, j, want_result=True):
        """y_j in original vertex order (unit 2-norm, non-negative sum). want_result=False (world > 1 only): take part only."""
        if not want_result:
            _check(lib.lz_get_ritz_vector(self._h, j, None))
            return None
        y = np.empty(self.graph_info().n)
        _check(lib.lz_get_ritz_vector(self._h, j, _f64(y)))
        return y

    def spectral_radius_bounds(self):
        """(lo, hi) with lo <= lambda_max <= hi, after ritz()."""
        lo, hi = C.c_double(0), C.c_double(0)
        _check(lib.lz_spectral_radius_bounds(self._h, C.byref(lo), C.byref(hi)))
        return lo.value, hi.value

    def set_spmv_variant(self, v):
        _check(lib.lz_set_spmv_variant(self._h, v))

    def set_profiling(self, on):
        _check(lib.lz_set_profiling(self._h, int(on)))

    def exchange_info(self):
        """(mode, need_frac): mode is one of EXCHANGE_NONE / _NCCL / _PEER_DENSE / _PEER_SPARSE."""
        mode, frac = C.c_int(0), C.c_double(0)
        _check(lib.lz_exchange_info(self._h, C.byref(mode), C.byref(frac)))
        return mode.value, frac.value

    def timings(self):
        t = Timings()
        _check(lib.lz_timings_get(self._h, C.byref(t)))
        return t

    def sync(self):
        _check(lib.lz_sync(self._h))

    def timer_start(self):
        _check(lib.lz_timer_start(self._h))

    def timer_stop(self):
        ms = C.c_float(0)
        _check(lib.lz_timer_stop(self._h, C.byref(ms)))
        return ms.value

    def trace_on(self, cap=4096):
        _check(lib.lz_debug_trace(self._h, cap, None, 0, None))

    def trace_read(self, cap=4096):
        """-> array [(tag, ns)] in order of arrival; switches the timeline off."""
        buf, cnt = np.empty((cap, 2), np.uint64), C.c_uint32(0)
        _check(lib.lz_debug_trace(self._h, 0, buf.ctypes.data_as(_u64p), cap, C.byref(cnt)))
        return buf[:cnt.value]

    def flush_l2(self):
        _check(lib.lz_flush_l2(self._h))
