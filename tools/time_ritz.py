"""Cost of lz_ritz on C3 (R-MAT 2^24, ef 8, k = 50, full reorthogonalisation, one GPU), fp64 and fp32 basis, m = 1, 4, 8, 16.
Prints JSON lines, each with the card's name and power limit.

  whole   lz_ritz from call to return (CUDA events on the context's stream around a call that ends in its own synchronise, so host
          gaps inside the call count), median of 10 after 2 warm-ups;
  parts   device time per kernel from a separate torch.profiler run (CUDA activity, 3 calls, the last one kept), grouped in launch
          order: the combine pass (k_ritz_combine, or k_combine + k_vsum for m = 1) with its rate on 8nk + 8nm bytes (fp32 basis:
          4nk + 8nm) against the measured HBM peak DESIGN.md section 3 uses; the residual SpMVs and combines; the Collatz-Wielandt
          weights, SpMV and reduction; the rest (tridiagonal solve, selection, normalisation).
The basis (6.7 GB in fp64) is far larger than L2: no flush.

    python tools/time_ritz.py
"""
import json
import os
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np  # noqa: E402

import __graft_entry__ as g  # noqa: E402
import bench  # noqa: E402

lz = g.load_package()
HBM_PEAK_GBS = 6535.7   # measured HBM peak of DESIGN.md section 3


def card():
    out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                         capture_output=True, text=True, check=True).stdout.strip().split(", ")
    return {"gpu": out[0], "power_limit": out[1]}


def emit(rec):
    print(json.dumps(dict(rec, **card())), flush=True)


def whole_ms(ctx, m, reps=10):
    for _ in range(2):
        ctx.ritz(m)
    ms = []
    for _ in range(reps):
        ctx.timer_start()
        ctx.ritz(m)
        ms.append(ctx.timer_stop())
    return float(np.median(ms)), float(min(ms))


def parts_ms(ctx, m):
    """Kernel device times of the last of 3 lz_ritz calls, grouped by phase (launch order)."""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(3):
            ctx.ritz(m)
    with tempfile.TemporaryDirectory() as td:
        path = os.path.join(td, "trace.json")
        prof.export_chrome_trace(path)
        ev = json.load(open(path))["traceEvents"]
    kern = sorted((e for e in ev if e.get("cat") == "kernel"), key=lambda e: e["ts"])
    starts = [i for i, e in enumerate(kern) if "k_tridiag_expv" in e["name"]]
    if not starts:
        raise RuntimeError("the profiler recorded no lz_ritz kernels")
    call = kern[starts[-1]:]
    out = {"combine": 0.0, "residual": 0.0, "cw": 0.0, "other": 0.0}
    scaled = in_cw = False       # launch order: solve, select, combine, scale, then per vector SpMV + combine; CW after vector 0
    for e in call:
        name = e["name"]
        if "k_ritz_scale" in name or "k_tridiag_expv" in name or "k_ritz_select" in name:
            scaled = scaled or "k_ritz_scale" in name
            key = "other"
        elif not scaled:
            key = "combine"
        elif "k_cw_z" in name or "k_cw_bound" in name:
            in_cw = "k_cw_z" in name
            key = "cw"
        else:
            key = "cw" if in_cw else "residual"
        out[key] += float(e["dur"]) / 1e3
    return out


def main():
    w = bench.WORKLOADS["c3"]
    k = w["k"]
    for basis, bname in ((lz.BASIS_F64, "f64"), (lz.BASIS_F32, "f32")):
        with lz.Context(0) as ctx:
            if basis == lz.BASIS_F32:
                ctx.set_basis_precision(lz.BASIS_F32)
            ctx.graph_generate(bench.make_spec(lz, w))
            n = ctx.graph_info().n
            ctx.set_start_vector(None)
            ctx.lanczos_run(k, lz.REORTH_FULL)
            for m in (1, 4, 8, 16):
                med, best = whole_ms(ctx, m)
                p = parts_ms(ctx, m)
                gb = ((4 if basis == lz.BASIS_F32 else 8) * n * k + 8 * n * m) / 1e9
                rate = gb / (p["combine"] * 1e-3)
                th, rho, res = ctx.ritz(m)
                lo, hi = ctx.spectral_radius_bounds()
                emit({"what": "lz_ritz", "workload": "c3", "n": n, "k": k, "basis": bname, "m": m, "whole_ms_median": med,
                      "whole_ms_min": best, "combine_ms": p["combine"], "combine_gb": gb, "combine_gbs": rate,
                      "combine_of_hbm_peak": rate / HBM_PEAK_GBS, "residual_ms": p["residual"], "cw_ms": p["cw"],
                      "other_ms": p["other"], "theta0": float(th[0]), "resid0": float(res[0]), "lo": lo, "hi": hi})


if __name__ == "__main__":
    main()
