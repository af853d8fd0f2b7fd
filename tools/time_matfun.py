"""Cost of choosing the matrix function (lz_set_matfun). Prints JSON lines, each with the card's name and power limit.

  (a) device time of the coefficient solve (lz_timings.tridiag_ms, median of 20) for EXP t=1 (the default), EXP t=2,
      EXP_SCALED t=2 and RESOLVENT alpha=0.01 at Krylov dimensions 50 / 100 / 200 (on C1's graph; the solve sees only the k x k
      tridiagonal);
  (b) on C3 (R-MAT 2^24, ef 8, k = 50, full reorthogonalisation), a sweep over 8 inverse temperatures with EXP_SCALED: one
      lz_lanczos_run followed by 8 x (lz_tridiag_expv + lz_multout + lz_top_k(100)), against 8 separate pipelines
      (start vector + lz_lanczos_run + lz_tridiag_expv + lz_multout + lz_top_k(100)). Neither side copies the n-vector to the host.
      Wall time around work that ends in a synchronise (lz_top_k synchronises), best of 3 after one warm-up of each side.

    python tools/time_matfun.py
"""
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np  # noqa: E402

import __graft_entry__ as g  # noqa: E402
import bench  # noqa: E402

lz = g.load_package()


def card():
    out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                         capture_output=True, text=True, check=True).stdout.strip().split(", ")
    return {"gpu": out[0], "power_limit": out[1]}


def emit(rec):
    print(json.dumps(dict(rec, **card())), flush=True)


def tridiag_times(ctx):
    funs = [("EXP", lz.MATFUN_EXP, 1.0), ("EXP", lz.MATFUN_EXP, 2.0), ("EXP_SCALED", lz.MATFUN_EXP_SCALED, 2.0),
            ("RESOLVENT", lz.MATFUN_RESOLVENT, 0.01)]
    ctx.graph_generate(bench.make_spec(lz, bench.WORKLOADS["c1"]))
    for k in (50, 100, 200):
        ctx.set_start_vector(None)
        ctx.lanczos_run(k, lz.REORTH_FULL)     # k up to 200 on a 10k-vertex graph: keep the tridiagonal free of ghosts
        for name, kind, p in funs:
            ctx.set_matfun(kind, p)
            ms = []
            for _ in range(21):
                ctx.tridiag_expv()
                ms.append(ctx.timings().tridiag_ms)
            emit({"what": "tridiag_ms", "k": k, "kind": name, "param": p, "median_ms": float(np.median(ms[1:])),
                  "min_ms": float(min(ms[1:]))})
    ctx.set_matfun(lz.MATFUN_EXP, 1.0)


def sweep(ctx):
    w = bench.WORKLOADS["c3"]
    k, reorth = w["k"], lz.REORTH_FULL if w["reorth"] else lz.REORTH_NONE
    ts = [0.125 * 2 ** i for i in range(8)]
    ctx.graph_generate(bench.make_spec(lz, w))

    def shared():
        ctx.set_start_vector(None)
        ctx.lanczos_run(k, reorth)
        for t in ts:
            ctx.set_matfun(lz.MATFUN_EXP_SCALED, t)
            ctx.tridiag_expv()
            ctx.multout()
            ctx.top_k(100)

    def separate():
        for t in ts:
            ctx.set_matfun(lz.MATFUN_EXP_SCALED, t)
            ctx.set_start_vector(None)
            ctx.lanczos_run(k, reorth)
            ctx.tridiag_expv()
            ctx.multout()
            ctx.top_k(100)

    res = {}
    for name, fn in (("one_run_8_functions", shared), ("8_pipelines", separate)):
        fn()
        best = float("inf")
        for _ in range(3):
            ctx.sync()
            t0 = time.perf_counter()
            fn()
            best = min(best, time.perf_counter() - t0)
        res[name] = best * 1e3
    emit({"what": "t_sweep_c3", "workload": w["name"], "ts": ts, "one_run_8_functions_ms": res["one_run_8_functions"],
          "8_pipelines_ms": res["8_pipelines"], "speedup": res["8_pipelines"] / res["one_run_8_functions"]})


if __name__ == "__main__":
    with lz.Context(0) as c:
        tridiag_times(c)
        sweep(c)
