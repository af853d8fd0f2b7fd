"""Host-side logic that needs no GPU: the C++ mirror of the reference API builds and refuses to run without a device,
bench.py's reference arm follows the contract (also under a 2-rank launch, gloo / CPU only), and the sharding arithmetic
of the multi-GPU layout."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIBDIR = os.path.join(ROOT, "msc-hpc-final-project_b200", "lib")


def _have_gpu():
    try:
        return subprocess.run(["nvidia-smi", "-L"], capture_output=True).returncode == 0
    except OSError:
        return False


def test_cpp_api_mirror_builds_and_has_reference_surface(lz):
    subprocess.check_call(["make", "-s", "-C", LIBDIR])
    assert os.path.exists(os.path.join(LIBDIR, "final"))
    # the reference's public names (SURVEY.md section 8b) are present with the reference's signatures
    hdr = {f: open(os.path.join(LIBDIR, f)).read() for f in os.listdir(LIBDIR) if f.endswith(".h")}
    assert "adjMatrix(const unsigned N, const unsigned E, std::ifstream& f)" in hdr["adjMatrix.h"]
    assert "adjMatrix(const unsigned N, const unsigned m, const char c)" in hdr["adjMatrix.h"]
    assert "adjMatrix(const unsigned N, const unsigned E)" in hdr["adjMatrix.h"]
    assert "lanczosDecomp(adjMatrix& adj, const unsigned krylov, T* starting_vec, bool cuda" in hdr["cu_lanczos.h"]
    assert "eigenDecomp(lanczosDecomp<T>& _L)" in hdr["eigen.h"]
    assert "void multOut(lanczosDecomp<T>& L, eigenDecomp<T>& E, adjMatrix& A, bool Qtrans)" in hdr["multiplyOut.h"]
    assert "void check_ans(lanczosDecomp<T>& L1, lanczosDecomp<U>& L2)" in hdr["check_ans.h"]
    assert "void write_ans(std::string filename, lanczosDecomp<T>& L)" in hdr["write_ans.h"]
    assert '"k:f:b:n:e:v"' in hdr["helpers.h"]


def test_cpp_driver_fails_loudly_without_gpu(lz):
    if _have_gpu():
        pytest.skip("a GPU is present")
    subprocess.check_call(["make", "-s", "-C", LIBDIR])
    r = subprocess.run([os.path.join(LIBDIR, "final"), "--graph", "er", "-n", "500", "-e", "1500", "-k", "5"],
                       capture_output=True, text=True)
    assert r.returncode != 0
    assert "no CPU fallback" in r.stderr


def _run_bench(args, env_extra=None, timeout=300):
    env = dict(os.environ)
    env.update(env_extra or {})
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + args, capture_output=True, text=True, env=env,
                          timeout=timeout)


def test_bench_reference_arm_contract():
    r = _run_bench(["--impl", "reference", "--workload", "c1", "--steps", "2", "--warmup", "1"])
    assert r.returncode == 0, r.stderr[-2000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["metric"] == "lanczos_iterations_per_sec" and line["unit"] == "iterations/s"
    assert line["steps"] == 2 and line["warmup"] == 1 and line["value"] > 0 and line["higher_is_better"] is True
    assert line["e2e"] == {"value": line["value"], "unit": line["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert line["cpu_baseline"]["kind"] in ("reference", "port") and line["cpu_baseline"]["cores"] == 1
    assert line["config"]["workload"].startswith("C1")


def test_bench_reference_arm_two_ranks_only_rank0_works():
    """Under torchrun (N > 1) rank 0 alone runs and prints the reference line; the other ranks exit 0 without work."""
    procs = []
    for rank in (0, 1):
        env = {"RANK": str(rank), "LOCAL_RANK": str(rank), "WORLD_SIZE": "2", "MASTER_ADDR": "127.0.0.1", "MASTER_PORT": "29733"}
        procs.append(_run_bench(["--impl", "reference", "--gpus", "2", "--workload", "c1", "--steps", "1", "--warmup", "0"], env))
    assert procs[0].returncode == 0 and procs[1].returncode == 0
    assert json.loads(procs[0].stdout.strip().splitlines()[-1])["n_gpus"] == 2
    assert procs[1].stdout.strip() == ""


def _gloo_worker(rank, world, port, q):
    import torch.distributed as dist
    os.environ.update({"MASTER_ADDR": "127.0.0.1", "MASTER_PORT": str(port), "RANK": str(rank), "WORLD_SIZE": str(world)})
    dist.init_process_group("gloo", rank=rank, world_size=world)
    box = [b"uid-from-rank-0" if rank == 0 else None]
    dist.broadcast_object_list(box, src=0)                       # how bench.py / dist_check.py ship the NCCL unique id
    import torch
    t = torch.tensor([float(rank + 1)], dtype=torch.float64)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)                     # how bench.py takes the max over ranks
    q.put((rank, box[0], float(t.item())))
    dist.destroy_process_group()


def test_two_rank_plumbing_on_gloo():
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    ps = [ctx.Process(target=_gloo_worker, args=(r, 2, 29741, q)) for r in range(2)]
    for p in ps:
        p.start()
    got = sorted(q.get(timeout=120) for _ in ps)
    for p in ps:
        p.join(timeout=60)
        assert p.exitcode == 0
    assert got == [(0, b"uid-from-rank-0", 2.0), (1, b"uid-from-rank-0", 2.0)]


@pytest.mark.parametrize("n,world", [(257, 2), (10000, 4), (1 << 20, 8), (33, 8)])
def test_shard_layout_arithmetic(n, world):
    """The relabelling rule of lz_graph.cu (sorted position s -> rank s % world, local row s // world, new id
    rank * n_loc + local, n_loc = ceil(n / world) rounded up to 32) is a bijection onto disjoint, equal, aligned slices."""
    n_loc = ((n + world - 1) // world + 31) // 32 * 32
    s = np.arange(n)
    new = (s % world) * n_loc + s // world
    assert len(np.unique(new)) == n and new.max() < n_loc * world
    per_rank = np.bincount(new // n_loc, minlength=world)
    assert per_rank.max() - per_rank.min() <= 1
    assert (n_loc * 8) % 256 == 0
    # degree-sorted dealing keeps every rank's rows sorted by the same key
    for r in range(world):
        mine = np.sort(new[new // n_loc == r]) - r * n_loc
        assert np.array_equal(mine, np.arange(len(mine)))


def test_fixture_parity_checker_against_oracle_ranking(orc, golden):
    """tests/fixture_parity.py (the checker bench.py uses for its `parity` object): its host ranking equals the oracle's on
    vectors with ties, and a summary made from a vector compares clean with that vector and dirty with a perturbed one."""
    import fixture_parity as fp
    import sys
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden"))
    import make_golden_c3 as mg
    rng = np.random.default_rng(0)
    y = np.floor(rng.random(5000) * 50.0)                      # many ties
    for m in (1, 10, 100, 5000):
        assert np.array_equal(fp.top_order(y, m), orc.top_k(y, m))
    g = golden("c1_er_n10000_k20")
    y = g["ans"]
    import tempfile
    with tempfile.TemporaryDirectory() as td:
        path = os.path.join(td, "s.npz")
        np.savez_compressed(path, **mg.summarize(y, g["alpha"], g["beta"], {"source": "test"}))
        r = fp.compare(y, path, g["alpha"], g["beta"], orc.top_k(y, 100), y[orc.top_k(y, 100)])
        assert r["ok"] and r["rel_2norm"] == 0.0 and r["top_k_api_identical"] and r["alpha_lead_rel"] == 0.0
        y2 = y.copy()
        y2[int(g["n"]) // 2] *= 1.0 + 1e-6                    # one wrong entry anywhere must show up (block sums cover every entry)
        assert not fp.compare(y2, path)["ok"]
        y3 = y.copy()
        t = orc.top_k(y, 2)
        y3[t[0]], y3[t[1]] = y[t[1]], y[t[0]]                 # swapped ranking
        assert not fp.compare(y3, path)["top100_identical"]


def test_c3_and_c2_reference_summaries_are_committed():
    import fixture_parity as fp
    for scale, k in ((20, 30), (24, 50)):
        p = fp.fixture_path("rmat", scale, k)
        assert p, (scale, k)
        g = np.load(p)
        assert len(g["alpha"]) == k and len(g["beta"]) == k - 1 and int(g["n"]) == 1 << scale
        assert float(g["top_gap"]) > 1e-6 and "ref_final" in str(g["meta"])


def test_bench_step_breakdown_parses_a_device_timeline():
    """bench.step_breakdown turns (tag, ns) events of lz_debug_trace into per-phase means; checked on a synthetic timeline."""
    sys.path.insert(0, ROOT)
    import bench

    def tag(kern, phase):
        return (kern << 8) | phase
    ev, t = [], 1000
    for step in range(8):
        ev += [(tag(0x10, 1), t), (tag(0x10, 5), t), (tag(0x10, 2), t + 1000), (tag(0x10, 6), t + 90000), (tag(0x10, 4), t + 101000)]
        t += 120000
        ev += [(tag(0x11, 1), t), (tag(0x11, 2), t + 2000), (tag(0x11, 4), t + 60000)]
        t += 65000
        ev += [(tag(0x01, 1), t), (tag(0x01, 2), t + 9000), (tag(0x01, 3), t + 109000), (tag(0x01, 4), t + 130000)]
        t += 135000

    class FakeCtx:
        def trace_on(self, cap): pass
        def lanczos_run(self, k): pass
        def trace_read(self, cap): return np.array(ev, dtype=np.uint64)
    out = bench.step_breakdown(FakeCtx(), 8, lambda x: x)
    assert out["update_wait_for_alpha"] == 9.0 and out["update_push_chunk0"] == 100.0 and out["update_kernel"] == 130.0
    assert out["spmv_pass0_wait_for_chunk"] == 1.0 and out["spmv_pass0_gather"] == 100.0 and out["spmv_pass0_senders_next_chunk"] == 90.0
    assert out["spmv_pass1_wait_for_chunk"] == 2.0 and out["spmv_pass1_senders_next_chunk"] is None
    assert out["wait_total_max_over_ranks"] == 12.0


def test_bench_dump_outputs_writes_float_arrays_and_a_fixed_sample(tmp_path):
    """bench.dump_outputs (--dump-outputs): float64 .npy files of the answer and the tridiagonal; a vector longer than
    DUMP_SAMPLE becomes the same seeded sample on every run, with its vertex ids; a rank without `write` writes nothing."""
    sys.path.insert(0, ROOT)
    import bench

    class FakeCtx:
        def __init__(self, n):
            self.y = np.random.default_rng(n).random(n)

        def get_ans(self):
            return self.y

        def get_tridiag(self):
            return np.arange(1.0, 6.0), np.arange(1.0, 5.0)
    small, big = FakeCtx(1000), FakeCtx(bench.DUMP_SAMPLE + 12345)
    bench.dump_outputs(small, str(tmp_path / "small"), True)
    assert sorted(os.listdir(tmp_path / "small")) == ["alpha.npy", "ans.npy", "beta.npy"]
    assert np.array_equal(np.load(tmp_path / "small" / "ans.npy"), small.y)
    runs = []
    for d in ("big1", "big2"):
        bench.dump_outputs(big, str(tmp_path / d), True)
        runs.append({f: np.load(tmp_path / d / f) for f in os.listdir(tmp_path / d)})
    assert sorted(runs[0]) == ["alpha.npy", "ans.npy", "ans_index.npy", "beta.npy"]
    assert all(a.dtype == np.float64 for a in runs[0].values())
    assert all(np.array_equal(runs[0][f], runs[1][f]) for f in runs[0])
    idx = runs[0]["ans_index.npy"].astype(np.int64)
    assert len(idx) == bench.DUMP_SAMPLE and np.all(np.diff(idx) > 0) and idx[-1] < len(big.y)
    assert np.array_equal(runs[0]["ans.npy"], big.y[idx])
    assert np.array_equal(runs[0]["alpha.npy"], np.arange(1.0, 6.0))
    assert sum(os.path.getsize(tmp_path / "big1" / f) for f in runs[0]) <= 64 << 20
    bench.dump_outputs(big, str(tmp_path / "other_rank"), False)
    assert not os.path.exists(tmp_path / "other_rank")
