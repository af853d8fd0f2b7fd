#!/usr/bin/env python
"""bench.py — Lanczos e^A·x throughput on B200 (BASELINE.json metric: Lanczos iterations/s + SpMV GB/s vs HBM roofline).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload c3] [--impl reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P bench.py --gpus N ...

One "step" = one full e^A·x evaluation on the workload graph: k Lanczos steps (fused SpMV+alpha, fused update+norm,
scale), the on-device tridiagonal eigen-solve + coefficient vector, and multOut — i.e. what parallel-final/main.cu:115-127
times, with the start vector already resident in HBM. `value` = k*K / (device time of K steps), max over ranks.
`e2e` = the same through the reference-facing call lz_expv_host with pinned HOST buffers (H2D of x and D2H of e^A x inside
the timed region). PyTorch is used only for torch.distributed plumbing and pinned host memory.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
import __graft_entry__ as graft  # noqa: E402

METRIC, UNIT = "lanczos_iterations_per_sec", "iterations/s"
GATHER_CEILING = 275.0   # 1e9 random 8-byte gathers per second, measured on this pool's B200 (one line lookup per clock per SM)

# BASELINE.json configs (SURVEY.md section 8d). `k`/`reorth` are the config's; the default bench line uses plain Lanczos
# (what the reference computes and what the roofline formula 4*nnz + 68*n describes) and reports the config's
# full-reorthogonalisation variant next to it under "detail".
WORKLOADS = {
    "c1": dict(kind="er", n=10000, m=50000, seed=20261018, k=20, reorth=False, name="C1 ER n=10k deg10 k=20"),
    "c2": dict(kind="rmat", scale=20, ef=8, seed=1, k=30, reorth=False, name="C2 R-MAT 2^20 ef8 k=30"),
    "c3": dict(kind="rmat", scale=24, ef=8, seed=1, k=50, reorth=True, name="C3 R-MAT 2^24 ef8 k=50"),
    "c4": dict(kind="rmat", scale=27, ef=8, seed=1, k=50, reorth=False, name="C4 R-MAT 2^27 ef8 k=50"),
    "c5": dict(kind="band", n=1 << 28, seed=5, k=100, reorth=False, name="C5 banded 2^28 k=100"),
}


def make_spec(lz, w, scale_override=None, n_override=None):
    if n_override:
        w = dict(w, n=n_override)
    if w["kind"] == "rmat":
        return lz.GraphSpec.rmat(scale_override or w["scale"], w["ef"], w["seed"])
    if w["kind"] == "er":
        return lz.GraphSpec.er(w["n"], w["m"], w["seed"])
    return lz.GraphSpec.band(w["n"], w["seed"])


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, device):
        self.device, self.rows, self.proc = device, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100",
                                          "-i", str(self.device)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm, mx, reasons, power = [], [], set(), []
        for r in self.rows:
            if len(r) < 9:
                continue
            try:
                sm.append(float(r[1])); mx.append(float(r[2])); power.append(float(r[3]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(power) if power else None, "samples": len(sm), "reasons": sorted(reasons)}


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def ncu_traffic(workload, world):
    """dram bytes per SpMV launch from a committed ncu --set full capture of exactly this (workload, GPU count); else None."""
    p = os.path.join(ROOT, "profiles", "spmv_traffic.json")
    if os.path.exists(p):
        try:
            return json.load(open(p)).get(f"{workload}@{world}")
        except Exception:
            return None
    return None


def step_breakdown(ctx, k, max_over_ranks):
    """Mean microseconds per step of the phases inside the multi-GPU kernels (this rank; waits also as max over ranks)."""
    ctx.trace_on(8192)
    ctx.lanczos_run(k)
    ev = ctx.trace_read(8192)
    tag, t = ev[:, 0].astype(np.int64), ev[:, 1].astype(np.int64)
    order = np.argsort(t, kind="stable")
    tag, t = tag[order], t[order]
    times = {}
    for tg, ts in zip(tag, t):
        times.setdefault((int(tg >> 8) & 255, int(tg & 255)), []).append(int(ts))

    def mean_dur(kern, a, b):
        x, y = times.get((kern, a), []), times.get((kern, b), [])
        m = min(len(x), len(y))
        if m < 4:
            return None
        d = (np.array(y[-m:]) - np.array(x[-m:]))[2:]
        return float(np.mean(d)) / 1e3
    out = {"update_wait_for_alpha": mean_dur(1, 1, 2), "update_push_chunk0": mean_dur(1, 2, 3), "update_kernel": mean_dur(1, 1, 4)}
    passes = sorted({kern for kern, _ in times if kern >= 0x10})
    for kern in passes:
        b = kern - 0x10
        out[f"spmv_pass{b}_wait_for_chunk"] = mean_dur(kern, 1, 2)
        out[f"spmv_pass{b}_gather"] = mean_dur(kern, 2, 4)
        out[f"spmv_pass{b}_senders_next_chunk"] = mean_dur(kern, 5, 6)
    out = {k_: (round(v, 1) if v is not None else None) for k_, v in out.items()}
    waits = [v for k_, v in out.items() if "wait" in k_ and v is not None]
    out["wait_total_max_over_ranks"] = round(max_over_ranks(sum(waits)), 1) if waits else None
    out["note"] = "rank 0; pass gather time of a non-final pass is that of its first gatherer CTA"
    return out


def workload_config(w, n, nnz, k, world):
    """The `config` object — identical in the `ours` and `reference` arms (same workload, same keys)."""
    n_loc, nnz_loc = n / world, nnz / world
    return {"workload": w["name"], "n": n, "nnz": nnz, "k": k, "reorth": "none", "x": "ones",
            "l2_policy": "inputs larger than L2 (CSR %.2f GB + basis %.2f GB per GPU)" % ((4.0 * nnz_loc + 4 * n_loc) / 1e9, 8.0 * n_loc * k / 1e9)}


def summary_fixture(w, scale_override, k):
    """Committed summary of the reference's (or, for sizes the CPU reference cannot reach, this library's 1-GPU) answer."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import fixture_parity as fp
    if w["kind"] != "rmat":
        return fp, None
    scale = scale_override or w["scale"]
    path = fp.fixture_path("rmat", scale, k, w["seed"], w["ef"])
    if path is None:
        own = os.path.join(fp.GOLDEN, f"own_rmat_s{scale}_k{k}_summary.npz")
        path = own if os.path.exists(own) else None
    return fp, path


def cpu_reference_sample(orc, csr_path, n, nnz, iters, reps=1):
    """Times the reference's own CPU pipeline (oracle/_ref/ref_final: lanczosDecomp<double>(A, m, ones, cuda=false) ->
    eigenDecomp -> multOut, parallel-final/main.cu:83-93; Lanczos single-threaded, multOut on the reference's 4 OpenBLAS
    threads) at Krylov dimension m = `iters` on the workload graph: a bounded sample of the k-step job with every stage present.
    Returns per-repetition iterations/s, seconds, the kind, and the reference's alpha/beta of the sample (the leading
    coefficients of the full run). Falls back to the C restatement (oracle/lanczos_oracle.c) when oracle/_ref is absent."""
    if orc.have_ref():
        r = orc.run_ref_final(None, None, iters, reps=reps, want_output=True, csr_path=csr_path)
        secs = [t["total_s"] for t in r["timings"]]
        vals = [iters / s for s in secs]
        return vals, secs, "reference", r["alpha"], r["beta"]
    with open(csr_path, "rb") as f:                      # LZCSR1 cache, read without the product library
        assert f.read(8) == b"LZCSR1\0\0"
        nn, mm = (int(v) for v in np.fromfile(f, np.uint64, 2))
        ro, ci = np.fromfile(f, np.uint32, nn + 1), np.fromfile(f, np.uint32, mm)
    vals, secs, a, b = [], [], None, None
    for _ in range(reps):
        t0 = time.perf_counter()
        _, a, b = orc.expv(ro, ci, iters, np.ones(n))
        dt = time.perf_counter() - t0
        vals.append(iters / dt); secs.append(dt)
    return vals, secs, "port", a, b


_MAKE_CSR = """
import sys
sys.path.insert(0, sys.argv[1])
import __graft_entry__ as g
lz = g.load_package()
kind, a, b, seed, path, dev = sys.argv[2], int(sys.argv[3]), int(sys.argv[4]), int(sys.argv[5]), sys.argv[6], int(sys.argv[7])
spec = {"rmat": lambda: lz.GraphSpec.rmat(a, b, seed), "er": lambda: lz.GraphSpec.er(a, b, seed), "band": lambda: lz.GraphSpec.band(a, seed)}[kind]()
try:
    with lz.Context(dev) as ctx:
        ctx.graph_generate(spec)
        ro, ci = ctx.csr_download()
except lz.LzError:
    _, ro, ci = lz.generate_host(spec)
lz.write_bin(path, ro, ci)
print(len(ro) - 1, int(ro[-1]))
"""


def make_csr_file(w, scale_override, n_override, path, device):
    """Writes the workload's CSR cache in a SEPARATE process, so the process that times the reference never loads liblzb200.so."""
    if w["kind"] == "rmat":
        a, b = scale_override or w["scale"], w["ef"]
    elif w["kind"] == "er":
        a, b = n_override or w["n"], w["m"]
    else:
        a, b = n_override or w["n"], 0
    r = subprocess.run([sys.executable, "-c", _MAKE_CSR, ROOT, w["kind"], str(a), str(b), str(w["seed"]), path, str(device)],
                       check=True, capture_output=True, text=True)
    n, nnz = (int(v) for v in r.stdout.split()[-2:])
    return n, nnz


DUMP_SAMPLE = 1 << 21   # entries of e^A x that --dump-outputs writes at most: 16 MB of values + 16 MB of vertex ids


def dump_outputs(ctx, out_dir, write):
    """--dump-outputs: what a caller of the timed step receives, e^A x (lz_get_ans) and the tridiagonal (lz_get_tridiag), as
    float64 .npy files. Above DUMP_SAMPLE vertices ans.npy is a fixed seeded sample and ans_index.npy holds its vertex ids.
    Collective on several GPUs (lz_get_ans gathers the vector); only a rank with `write` set touches the file system."""
    y = ctx.get_ans()
    alpha, beta = ctx.get_tridiag()
    if not write:
        return
    os.makedirs(out_dir, exist_ok=True)
    out = {"alpha": alpha, "beta": beta, "ans": y}
    if len(y) > DUMP_SAMPLE:
        idx = np.sort(np.random.default_rng(20261018).choice(len(y), DUMP_SAMPLE, replace=False))
        out["ans"], out["ans_index"] = y[idx], idx.astype(np.float64)
    for name, a in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def sample_iters_for(nnz):
    # ~1e-8 s per stored entry per CPU iteration at large n (measured: 108 ms/iter at nnz 1.68e7) -> aim for ~10-15 s
    per_iter = max(nnz * 1.2e-8, 1e-4)
    return int(min(50, max(2, round(12.0 / per_iter))))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--workload", default="c3", choices=sorted(WORKLOADS))
    ap.add_argument("--scale", type=int, default=None, help="override the R-MAT scale (debug)")
    ap.add_argument("--k", type=int, default=None)
    ap.add_argument("--vertices", dest="n", type=int, default=None, help="override n of the ER / banded workloads (debug)")
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-reorth-detail", action="store_true")
    ap.add_argument("--no-f32-detail", action="store_true")
    ap.add_argument("--save-summary", default=None, help="write a summary fixture (.npz) of this run's answer (rank 0)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the last step's e^A x (sampled on large graphs) and alpha/beta as DIR/*.npy")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the answer of --impl ours")

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if world != args.gpus and world > 1:
        args.gpus = world
    w = dict(WORKLOADS[args.workload])
    k = args.k or w["k"]
    overrides = [f"{a}={v}" for a, v in (("scale", args.scale), ("n", args.n), ("k", args.k)) if v]
    if overrides:                                  # debug overrides must not masquerade as the named config
        w["name"] += " [override: " + ", ".join(overrides) + "]"
    warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup

    # ---------------------------------------------------------------------------------------------- reference arm
    if args.impl == "reference":
        if rank != 0:
            return 0
        orc = graft.load_oracle()              # the oracle is only ever loaded for the reference / cpu_baseline legs
        csr_path = os.path.join(tempfile.gettempdir(), f"lz_bench_{args.workload}_{args.scale or ''}_{os.getpid()}.bin")
        n, nnz = make_csr_file(w, args.scale, args.n, csr_path, local_rank)     # input construction: separate process, untimed
        m = min(sample_iters_for(nnz), k)             # never more steps than the config's Krylov dimension
        total = args.steps + args.warmup
        vals, secs, kind, a_ref, b_ref = cpu_reference_sample(orc, csr_path, n, nnz, m, reps=total)
        os.unlink(csr_path)
        vals, secs = vals[args.warmup:], secs[args.warmup:]
        value = m * len(secs) / sum(secs)
        sample = (f"per step: the reference pipeline at Krylov dimension {m} on {w['name']} (lanczosDecomp<double>(A,{m},ones,cuda=false) -> "
                  f"eigenDecomp -> multOut; Lanczos on 1 thread, multOut on the reference's 4 OpenBLAS threads)")
        lead = {"alpha": [float(v) for v in a_ref[:m]], "beta": [float(v) for v in b_ref[:m - 1]]}
        fp, fix = summary_fixture(w, args.scale, k)
        if fix and "own_" not in os.path.basename(fix):       # the sample's coefficients are the leading ones of the committed k-step reference run
            g = np.load(fix)
            lead["max_rel_diff_vs_fixture"] = float(max(np.max(np.abs(a_ref[:m] - g["alpha"][:m]) / np.abs(g["alpha"][:m])),
                                                         np.max(np.abs(b_ref[:m - 1] - g["beta"][:m - 1]) / np.abs(g["beta"][:m - 1]))))
            lead["fixture"] = os.path.basename(fix)
        line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": 1e3 * sum(secs) / len(secs), "higher_is_better": True, "scaling": "strong",
                "vs_baseline": None, "dtype": "f64", "data": "synthetic",
                "config": workload_config(w, n, nnz, k, args.gpus),
                "cpu_baseline": {"value": value, "unit": UNIT, "cores": 1, "kind": kind, "sample": sample, "sample_iters": m,
                                 "host_cores_available": os.cpu_count()},
                "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                "tridiag_lead": lead}
        print(json.dumps(line), flush=True)
        return 0

    lz = graft.load_package()

    # ------------------------------------------------------------------------------------------------------ our arm
    import torch
    dist = None
    uid = None
    if world > 1:
        import torch.distributed as dist
        # torch.distributed is host-side plumbing only (unique-id broadcast, barriers, max over ranks): gloo suffices.
        # The data path's collectives are NCCL calls inside liblzb200.so on its own communicator.
        dist.init_process_group("gloo")
        box = [lz.nccl_unique_id() if rank == 0 else None]
        dist.broadcast_object_list(box, src=0)
        uid = box[0]

    def barrier():
        if dist:
            dist.barrier()

    def max_over_ranks(x):
        if not dist:
            return x
        t = torch.tensor([x], dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    ctx = lz.Context(local_rank, rank, world, uid)
    spec = make_spec(lz, w, args.scale, args.n)
    t0 = time.perf_counter()
    ctx.graph_generate(spec)
    ctx.sync()
    t_graph = time.perf_counter() - t0
    gi = ctx.graph_info()
    n, nnz = gi.n, gi.nnz
    ctx.set_start_vector(None)                     # x = ones resident in HBM (main.cu:79)
    ctx.lanczos_run(k)                             # allocates the basis
    ctx.sync()

    def step():
        ctx.lanczos_run(k)
        ctx.tridiag_expv()
        ctx.multout()

    # Per-kernel CUDA events (profiling) are recorded inside the timed region whenever the step loop is issued launch by
    # launch (the default workload). Small single-GPU workloads replay the loop as one CUDA graph, which cannot carry the
    # events: there the timed region runs un-instrumented and one extra instrumented step follows it for the breakdown.
    graph_replay = world == 1 and gi.n_local <= (4 << 20) and os.environ.get("LZ_CUDA_GRAPH", "1") != "0"
    for _ in range(warmup):
        step()
    ctx.sync()
    if not graph_replay:
        ctx.set_profiling(True)
        step(); ctx.sync()                         # one profiled warm-up so event creation is outside the timed region
    launches0 = ctx.timings().kernel_launches
    sampler = ClockSampler(local_rank)
    barrier(); ctx.sync()
    sampler.start()
    ctx.timer_start()
    for _ in range(args.steps):
        step()
    ms = ctx.timer_stop()
    ctx.sync(); barrier()
    clocks = sampler.stop()
    tm = ctx.timings()
    launches = tm.kernel_launches - launches0
    ms = max_over_ranks(ms)
    value = k * args.steps / (ms * 1e-3)
    if args.dump_outputs:
        dump_outputs(ctx, args.dump_outputs, rank == 0)
    if graph_replay:
        ctx.set_profiling(True)
        step(); ctx.sync(); step(); ctx.sync()
        tm = ctx.timings()
    ctx.set_profiling(False)

    # lanczos-only and multOut-only numbers of the last step
    detail = {"lanczos_ms": tm.lanczos_ms, "tridiag_ms": tm.tridiag_ms, "multout_ms": tm.multout_ms,
              "spmv_ms_avg": tm.spmv_ms_avg, "update_scale_ms_per_iter": tm.update_ms_avg, "comm_ms_per_iter": tm.comm_ms_avg,
              "lanczos_only_iters_per_s": k / (tm.lanczos_ms * 1e-3) if tm.lanczos_ms else None,
              "graph_build_s": t_graph, "max_degree": gi.max_degree, "empty_rows": gi.empty_rows}

    # roofline of the dominant kernel (the SpMV: k_spmv_sell by default, k_spmv_dot for the CSR variants): algorithmic bytes 4*nnz + 20*n per launch (SURVEY.md 8d), per GPU
    peak, peak_src = measured_peak()
    # x is "compulsory once": every entry this rank's rows reference = its own slice + the referenced remote entries (all of x
    # for R-MAT; a halo plus chords for band-like graphs, where the exchange reports the fraction)
    xmode_, xfrac_ = ctx.exchange_info()
    x_ref = n if xmode_ in (0, 1) else gi.n_local * (1.0 + xfrac_ * (world - 1))
    b_spmv = 4.0 * gi.nnz_local + 4.0 * gi.n_local + 8.0 * min(x_ref, n) + 8.0 * gi.n_local   # == 4 nnz + 20 n at world == 1
    spmv_gbs = b_spmv / (tm.spmv_ms_avg * 1e-3) / 1e9 if tm.spmv_ms_avg else None
    spmv_kernel = "k_spmv_sell" if os.environ.get("LZ_SPMV_VARIANT", "0") in ("", "0") else "k_spmv_dot"
    roofline = {"bound": "hbm", "kernel": spmv_kernel, "achieved": spmv_gbs, "peak": peak, "unit": "GB/s",
                "frac": (spmv_gbs / peak) if spmv_gbs else None, "traffic": ncu_traffic(args.workload, world),
                "algorithmic_bytes_per_launch": b_spmv, "peak_source": peak_src,
                # what actually binds this kernel on a random graph: the SM load path's line-lookup rate (DESIGN.md section 3)
                "gather": {"achieved_ggathers_s": gi.nnz_local / (tm.spmv_ms_avg * 1e-3) / 1e9 if tm.spmv_ms_avg else None,
                           "ceiling_ggathers_s": GATHER_CEILING, "frac": (gi.nnz_local / (tm.spmv_ms_avg * 1e-3) / 1e9 / GATHER_CEILING)
                           if tm.spmv_ms_avg else None, "ceiling_source": "profiles/microbench/gather_bench_r01.txt (L2-resident random 8-B gathers)"}}
    b_iter = 4.0 * gi.nnz_local + 68.0 * gi.n_local
    detail["iteration_roofline_iters_per_s"] = peak * 1e9 / b_iter
    detail["iteration_frac_of_roofline"] = (k / (tm.lanczos_ms * 1e-3)) / (peak * 1e9 / b_iter) if tm.lanczos_ms else None
    b_mult = 8.0 * gi.n_local * k + 8.0 * gi.n_local
    detail["multout_gbs"] = b_mult / (tm.multout_ms * 1e-3) / 1e9 if tm.multout_ms else None

    # several GPUs: where a step's time goes, from the device-side timeline of one extra (untimed) run — stream events cannot
    # tell waiting for a peer apart from work inside the fused kernels (tools/trace_step.py prints the full table)
    if world > 1:
        try:
            detail["step_breakdown_us"] = step_breakdown(ctx, k, max_over_ranks)
        except Exception as e:                        # measurement hook only: never fail the bench line over it
            detail["step_breakdown_us"] = {"error": str(e)[:200]}

    # the config's full-reorthogonalisation variant (BASELINE configs[2] "with full reorthogonalisation"): its own top-level
    # object with its own roofline (the Gram-Schmidt passes over the resident basis are HBM-bound GEMV-T + GEMV-N)
    reorth_variant = None
    if w.get("reorth") and not args.no_reorth_detail:
        ctx.lanczos_run(k, lz.REORTH_FULL); ctx.sync()
        barrier()
        ctx.timer_start()
        for _ in range(3):
            ctx.lanczos_run(k, lz.REORTH_FULL)
        ms_r = max_over_ranks(ctx.timer_stop()) / 3.0
        second = ctx.timings().reorth_second_passes
        # one classical Gram-Schmidt pass per step (SURVEY 8d: 8n*k(k+1) + 16nk), plus the repeated passes
        b_reorth = (8.0 * gi.n_local * k * (k + 1) + 16.0 * gi.n_local * k) * (1.0 + second / max(k - 1, 1))
        r_gbs = b_reorth / max((ms_r - tm.lanczos_ms) * 1e-3, 1e-9) / 1e9
        reorth_variant = {"metric": METRIC, "value": k / (ms_r * 1e-3), "unit": UNIT, "lanczos_ms": ms_r, "reorth": "full",
                          "scheme": "CGS every step, second pass when ||w'||^2 < ||w||^2 / 2 (DGKS)", "second_passes": second,
                          "roofline": {"bound": "hbm", "kernel": "k_multidot + k_combine", "achieved": r_gbs, "peak": peak, "unit": "GB/s",
                                       "frac": r_gbs / peak, "algorithmic_bytes": b_reorth,
                                       "note": "reorthogonalisation bytes over (reorth run - plain run) device time"}}
        detail["full_reorth"] = {"lanczos_ms": ms_r, "iters_per_s": k / (ms_r * 1e-3), "reorth_gbs": r_gbs}

    # SURVEY 8f-4: the same job with the basis stored in fp32 (LZ_BASIS_F32; one GPU): multOut and reorthogonalisation bytes halve
    basis_f32 = None
    if world == 1 and not args.no_f32_detail:
        ctx.set_basis_precision(lz.BASIS_F32)
        ctx.set_start_vector(None)
        ctx.set_profiling(False)
        for _ in range(2):
            step()
        ctx.timer_start()
        for _ in range(3):
            step()
        ms32 = ctx.timer_stop() / 3.0
        t32 = ctx.timings()
        y32 = ctx.get_ans()
        basis_f32 = {"value": k / (ms32 * 1e-3), "unit": UNIT, "ms_per_step": ms32, "multout_ms": t32.multout_ms,
                     "multout_gbs": (4.0 * gi.n_local * k + 8.0 * gi.n_local) / (t32.multout_ms * 1e-3) / 1e9 if t32.multout_ms else None,
                     "basis_bytes": 4.0 * gi.n_local * k}
        if w.get("reorth") and not args.no_reorth_detail:
            ctx.lanczos_run(k, lz.REORTH_FULL); ctx.sync()
            ctx.timer_start()
            for _ in range(3):
                ctx.lanczos_run(k, lz.REORTH_FULL)
            ms_r32 = ctx.timer_stop() / 3.0
            b_r32 = 4.0 * gi.n_local * k * (k + 1) + 16.0 * gi.n_local * k
            basis_f32["full_reorth"] = {"value": k / (ms_r32 * 1e-3), "unit": UNIT, "lanczos_ms": ms_r32, "reorth_algorithmic_gb": b_r32 / 1e9,
                                        "reorth_gbs": b_r32 / max((ms_r32 - tm.lanczos_ms) * 1e-3, 1e-9) / 1e9}
        ctx.set_basis_precision(lz.BASIS_F64)
        ctx.set_start_vector(None)

    # end to end through the reference-facing call with HOST buffers (pinned), H2D of x and D2H of the answer inside
    x_host = torch.ones(n, dtype=torch.float64).pin_memory().numpy()
    y_host = torch.empty(n, dtype=torch.float64).pin_memory().numpy()
    want = rank == 0                               # the caller (rank 0) holds x and receives e^A x; the other ranks only compute

    def e2e_call():
        if world > 1:
            ctx.expv_host_root(x_host, k, out=y_host, root=0)    # one PCIe upload, NVLink broadcast, one download
        else:
            ctx.expv_host(x_host, k, out=y_host)
    for _ in range(2):
        e2e_call()
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        e2e_call()                                 # synchronous: returns after the D2H copy of the answer
    e2e_s = max_over_ranks(time.perf_counter() - t0)
    e2e = {"value": k * args.steps / e2e_s, "unit": UNIT, "h2d_bytes_per_step": 8 * n, "d2h_bytes_per_step": 8 * n,
           "ms_per_step": 1e3 * e2e_s / args.steps,
           "call": "lz_expv_host (pinned host x -> pinned host e^A x)" if world == 1 else
                   "lz_expv_host_root (rank 0: pinned host x -> NVLink broadcast -> ... -> pinned host e^A x)"}
    finite = bool(np.isfinite(y_host).all()) if want else True
    alpha_g, beta_g = ctx.get_tridiag()

    # end to end when the caller wants the RANKING (BASELINE configs[1]: "e^A x + centrality ranking"): host x in, the 100 most
    # central vertices out — lz_top_k selects on the device, so 100 (id, value) pairs cross PCIe instead of n doubles
    def e2e_rank_call():
        ctx.set_start_vector_root(x_host if want else None, 0) if world > 1 else ctx.set_start_vector(x_host)
        ctx.lanczos_run(k); ctx.tridiag_expv(); ctx.multout()
        return ctx.top_k(100)
    for _ in range(2):
        top_idx, top_val = e2e_rank_call()
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        top_idx, top_val = e2e_rank_call()
    rank_s = max_over_ranks(time.perf_counter() - t0)
    e2e_rank = {"value": k * args.steps / rank_s, "unit": UNIT, "ms_per_step": 1e3 * rank_s / args.steps, "h2d_bytes_per_step": 8 * n,
                "d2h_bytes_per_step": 100 * 12, "call": "lz_set_start_vector(host x) + lz_lanczos_run + lz_tridiag_expv + lz_multout + lz_top_k(100)"}

    # parity of THIS run's answer (the vector the e2e call returned to rank 0) against the committed summary of the reference
    parity = None
    fp, fix = summary_fixture(w, args.scale, k)
    if rank == 0:
        if fix:
            parity = fp.compare(y_host, fix, alpha_g, beta_g, top_idx, top_val)
            if basis_f32 is not None:
                p32 = fp.compare(y32, fix)
                basis_f32["parity_vs_reference_double"] = {"rel_2norm": p32["rel_2norm"], "top100_identical": p32["top100_identical"],
                                                           "bar": "reference float vs double: 2.7e-7 .. 5.2e-6 (tests/golden/reference_float.npz)"}
            if "own_" in os.path.basename(fix):
                parity["source"] = "this library's 1-GPU answer (the CPU reference cannot reach this size); " + parity["source"]
        else:
            parity = {"fixture": None, "note": "no committed reference summary for this workload; see tests/ for its parity cases",
                      "top_k_api_identical_to_host_argsort": bool(np.array_equal(fp.top_order(y_host, 100), top_idx))}
        if args.save_summary:
            sys.path.insert(0, os.path.join(ROOT, "tests", "golden"))
            import make_golden_c3 as mg
            meta = {"graph": {k_: w[k_] for k_ in ("kind", "scale", "ef", "seed") if k_ in w}, "k": k, "x": "ones", "nnz": nnz,
                    "source": f"bench.py --save-summary on {world} GPU(s), liblzb200 (NOT the reference)"}
            np.savez_compressed(args.save_summary, **mg.summarize(np.array(y_host), alpha_g, beta_g, meta))

    xmode, xfrac = ctx.exchange_info()
    exchange = {0: "none (one GPU)", 1: "ncclAllGather", 2: "peer stores over NVLink, whole vector",
                3: "peer stores over NVLink, referenced entries only (%.3g of the vector)" % xfrac}[xmode]
    ctx.close()

    # CPU baseline: the reference's own pipeline on the same graph, bounded sample, rank 0, N == 1 only
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        orc = graft.load_oracle()
        csr_path = os.path.join(tempfile.gettempdir(), f"lz_bench_{args.workload}_{os.getpid()}.bin")
        make_csr_file(w, args.scale, args.n, csr_path, local_rank)
        m = min(sample_iters_for(nnz), k)             # never more steps than the config's Krylov dimension
        vals, secs, kind, a_ref, b_ref = cpu_reference_sample(orc, csr_path, n, nnz, m, reps=1)
        os.unlink(csr_path)
        cpu = {"value": vals[0], "unit": UNIT, "cores": 1, "kind": kind,
               "sample": f"the reference pipeline at Krylov dimension {m} on {w['name']} (lanczosDecomp<double>, cuda=false, 1 thread; "
                         f"eigenDecomp; multOut on 4 OpenBLAS threads), {secs[0]:.1f} s",
               "host_cores_available": os.cpu_count(),
               # the reference's coefficients from this very run vs the GPU run's (same graph, same start vector)
               "tridiag_lead_max_rel_diff_vs_gpu": float(max(np.max(np.abs(a_ref[:m] - alpha_g[:m]) / np.abs(a_ref[:m])),
                                                             np.max(np.abs(b_ref[:m - 1] - beta_g[:m - 1]) / np.abs(b_ref[:m - 1])))) if m > 1 else None}

    if rank == 0:
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": warmup,
                "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
                "dtype": "f64", "data": "synthetic",
                "config": workload_config(w, n, nnz, k, world),
                "impl_config": {"parallelism": f"row-sharded x{world}" if world > 1 else "single GPU", "exchange": exchange,
                                "launch": "CUDA graph replay of the k-step loop" if graph_replay else "stream launches"},
                "clocks": clocks, "e2e": e2e, "e2e_rank": e2e_rank, "gpu_launches": int(launches), "roofline": roofline, "cpu_baseline": cpu,
                "parity": parity, "result_finite": finite, "reorth_variant": reorth_variant, "basis_f32": basis_f32, "detail": detail}
        print(json.dumps(line), flush=True)
    if dist:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
