"""Multi-GPU check of lz_ritz, one process per GPU:  torchrun --nproc-per-node P tests/ritz_dist_check.py
Every rank computes the one-GPU answer on its own device first, then the row-sharded one: Ritz pairs, vectors and the
spectral-radius bracket must match to 1e-12, and lo / hi must be the same bits on every rank. Prints 'RITZ_DIST_OK <world>' on rank 0."""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import __graft_entry__ as g  # noqa: E402


def pairs(c, m, want):
    th, rho, res = c.ritz(m)
    Y = [c.ritz_vector(j, want_result=want) for j in range(m)]
    return th, rho, res, Y, c.spectral_radius_bounds()


def main():
    import torch.distributed as dist
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ.get("LOCAL_RANK", 0))
    dist.init_process_group("gloo")
    lz = g.load_package()
    gdir = os.path.join(ROOT, "tests", "golden")
    cases = []
    for name in ("rmat_s12_k30", "band_n4096_k40", "er_n257_k10_ragged"):
        gl = np.load(os.path.join(gdir, name + ".npz"))
        n = int(gl["n"])
        cases.append((name, gl["row_offset"], gl["col_idx"], None, 40, lz.REORTH_NONE, 1))
        cases.append((name, gl["row_offset"], gl["col_idx"], np.random.default_rng(7).standard_normal(n), 40, lz.REORTH_FULL, 4))
    ref = []
    with lz.Context(local) as c1:
        for name, ro, ci, x, k, reorth, m in cases:
            c1.csr_upload(ro, ci)
            c1.set_start_vector(x)
            c1.lanczos_run(min(k, len(ro) - 1), reorth)
            ref.append(pairs(c1, m, True))
    box = [lz.nccl_unique_id() if rank == 0 else None]
    dist.broadcast_object_list(box, src=0)
    ctx = lz.Context(local, rank, world, box[0])
    for (name, ro, ci, x, k, reorth, m), (th0, rho0, res0, Y0, b0) in zip(cases, ref):
        ctx.csr_upload(ro, ci)
        ctx.set_start_vector(x)
        ctx.lanczos_run(min(k, len(ro) - 1), reorth)
        want = rank == world - 1          # one rank downloads, the others only take part in the gathers
        th, rho, res, Y, b = pairs(ctx, m, want)
        tag = (name, reorth, m)
        assert np.allclose(th, th0, rtol=1e-12, atol=0) and np.allclose(rho, rho0, rtol=1e-12, atol=0), tag
        assert np.allclose(res, res0, rtol=1e-6, atol=1e-12 * th0[0]), tag
        assert abs(b[0] - b0[0]) <= 1e-12 * b0[0] and abs(b[1] - b0[1]) <= 1e-12 * b0[1], (tag, b, b0)
        if want:
            for j in range(m):
                assert np.abs(Y[j] - Y0[j]).max() < 1e-12, (tag, j, np.abs(Y[j] - Y0[j]).max())
        else:
            assert all(y is None for y in Y)
        allb = [None] * world
        dist.all_gather_object(allb, b)
        assert all(v == allb[0] for v in allb), (tag, allb)
        # eigenvector centrality through the product API after lz_ritz
        idx, val = ctx.top_k(100)
        if want:
            assert np.array_equal(val, Y[0][idx])
    ctx.close()
    dist.barrier()
    if rank == 0:
        print(f"RITZ_DIST_OK {world}", flush=True)
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
