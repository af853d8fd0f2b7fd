"""B200-native Lanczos e^A·x (graph total-communicability) — Python face of the C ABI in include/lz.h.

The product is `csrc/liblzb200.so` (hand-written sm_100a CUDA + NCCL behind an `extern "C"` boundary) plus the C++
mirror of the reference's `parallel-final/lib` object API in `lib/`. This package is only the ctypes binding that the
tests and `bench.py` use to reach that ABI from Python; it contains no numerical code and there is NO CPU fallback:
if the shared library is missing the import fails, and if no GPU is present `Context()` raises.

The directory name is not a valid Python identifier; load it with `__graft_entry__.load_package()` (which registers it
in `sys.modules` as `msc_hpc_final_project_b200`).
"""
from ._capi import (  # noqa: F401
    LzError, Context, GraphSpec, GraphInfo, Timings, lib, lib_path, generate_host, read_text, write_text, read_bin,
    write_bin, csr_from_edges, device_count, nccl_unique_id, exported_symbols, header_symbols,
    GRAPH_ER, GRAPH_RMAT, GRAPH_BAND, REORTH_NONE, REORTH_FULL, SPMV_AUTO, SPMV_VECTOR, SPMV_WARP,
    EXCHANGE_NONE, EXCHANGE_NCCL, EXCHANGE_PEER_DENSE, EXCHANGE_PEER_SPARSE, BASIS_F64, BASIS_F32,
    MATFUN_EXP, MATFUN_EXP_SCALED, MATFUN_RESOLVENT, RITZ_MAX, CW_FLOOR,
)
