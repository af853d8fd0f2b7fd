"""Top Ritz pairs of the Krylov basis (lz_ritz): certified eigenvalue intervals, eigenvector centrality, and the spectral-radius
bracket that makes a Katz parameter safe. All need a GPU.

References: dense eigh for small graphs, scipy's eigsh for larger ones, the CPU oracle's Lanczos alpha/beta/Q for Krylov-level
checks, scipy's sparse solver for Katz."""
import os
import subprocess
import sys

import numpy as np
import pytest
import scipy.sparse as sp
import scipy.sparse.csgraph as csg
import scipy.sparse.linalg as spl

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDENS = ["er_n2000_k20", "rmat_s12_k30", "band_n4096_k40"]
ALL_GOLDENS = ["er_n257_k10_ragged", "er_n2000_k20", "rmat_s12_k30", "band_n4096_k40", "c1_er_n10000_k20", "rmat_s14_k50"]
GRAPH500 = (.57, .19, .19)


def adjacency(ro, ci):
    n = len(ro) - 1
    return sp.csr_matrix((np.ones(len(ci)), ci.astype(np.int64), ro.astype(np.int64)), shape=(n, n))


def rel2(a, b):
    return np.linalg.norm(a - b) / np.linalg.norm(b)


def sign_fixed(v):
    v = v / np.linalg.norm(v)
    return -v if v.sum() < 0 else v


def vec_tol(th, base):
    """Per-vector tolerance: a Ritz vector moves by about eps * ||A|| / gap_j under rounding, gap_j = distance of theta_j to the other
    Ritz values returned."""
    th = np.asarray(th)
    gaps = np.array([np.min(np.abs(np.delete(th, j) - th[j])) if len(th) > 1 else np.inf for j in range(len(th))])
    return base * np.maximum(1.0, np.abs(th).max() / gaps)


def raises_code(lz, code, fn, *a):
    with pytest.raises(lz.LzError) as e:
        fn(*a)
    assert e.value.code == code, str(e.value)


@pytest.fixture(scope="module")
def ctx(lz):
    c = lz.Context(0)
    yield c
    c.close()


@pytest.fixture
def mctx(lz, ctx):
    yield ctx
    ctx.set_matfun(lz.MATFUN_EXP, 1.0)
    ctx.set_spmv_variant(lz.SPMV_AUTO)


def run(c, lz, ro, ci, k, x=None, reorth=None):
    c.csr_upload(ro, ci)
    c.set_start_vector(x)
    c.lanczos_run(k, lz.REORTH_NONE if reorth is None else reorth)


@pytest.mark.parametrize("name", GOLDENS)
def test_certified_intervals(lz, golden, mctx, name):
    """Full reorthogonalisation, random start, k = 60, m = 8: every [rho - r, rho + r] holds an eigenvalue of the dense A; rho and r
    are what numpy computes from the returned vectors; the vectors are orthonormal with non-negative sums."""
    g = golden(name)
    ro, ci, n = g["row_offset"], g["col_idx"], int(g["n"])
    A = adjacency(ro, ci)
    lam = np.linalg.eigvalsh(A.toarray())
    norm_a = np.abs(lam).max()
    run(mctx, lz, ro, ci, 60, np.random.default_rng(11).standard_normal(n), lz.REORTH_FULL)
    m = 8
    th, rho, res = mctx.ritz(m)
    assert np.all(np.diff(th) <= 0)
    Y = np.stack([mctx.ritz_vector(j) for j in range(m)], axis=1)
    for j in range(m):
        assert np.min(np.abs(lam - rho[j])) <= res[j] + 1e-12 * norm_a, (j, rho[j], res[j])
        y = Y[:, j]
        ay = A @ y
        r_np = np.linalg.norm(ay - (y @ ay) * y)
        assert abs(rho[j] - y @ ay) <= 1e-9 * abs(y @ ay), j
        assert abs(res[j] - r_np) <= 1e-12 * norm_a, (j, res[j], r_np)
        assert y.sum() >= 0
    assert np.abs(Y.T @ Y - np.eye(m)).max() < 1e-10


@pytest.mark.parametrize("name", GOLDENS)
def test_krylov_parity(lz, orc, golden, mctx, name):
    """theta_j and y_j against Q z_j / ||Q z_j|| built from the oracle's Lanczos alpha / beta / Q at the same k.
    Plain run from ones (lagged basis rows): the top pair, which has converged. Past it a plain run's T grows ghost copies of the
    converged eigenvalue at steps that depend on rounding, so the oracle's T and this one need not share their second Ritz value.
    Full reorthogonalisation from a random start: the top 4 pairs."""
    g = golden(name)
    ro, ci, k, n = g["row_offset"], g["col_idx"], int(g["k"]), int(g["n"])
    m = 4
    for x, reorth, checked in ((np.ones(n), lz.REORTH_NONE, 1), (np.random.default_rng(8).standard_normal(n), lz.REORTH_FULL, m)):
        a, b, Q = orc.lanczos(ro, ci, k, x, orc.FULL if reorth else orc.PLAIN)
        th_ref, Z = np.linalg.eigh(np.diag(a) + np.diag(b, 1) + np.diag(b, -1))
        run(mctx, lz, ro, ci, k, x, reorth)
        th, _, _ = mctx.ritz(m)
        tol = vec_tol(th_ref[::-1], 1e-9)
        for j in range(checked):
            assert abs(th[j] - th_ref[k - 1 - j]) <= 1e-9 * abs(th_ref[k - 1 - j]), (reorth, j)
            ref = sign_fixed(Q @ Z[:, k - 1 - j])
            y = mctx.ritz_vector(j)
            assert min(rel2(y, ref), rel2(-y, ref)) < tol[j], (name, reorth, j, rel2(y, ref), tol[j])


def perron_check(lz, orc, c, ro, ci, k):
    n = len(ro) - 1
    A = adjacency(ro, ci)
    run(c, lz, ro, ci, k)
    th, rho, res = c.ritz(1)
    y = c.get_ans()
    lam, vec = spl.eigsh(A, k=2, which="LA", tol=1e-14)
    v = sign_fixed(vec[:, np.argmax(lam)])
    gap = lam.max() - lam.min()
    bound = 2 * res[0] / gap + 1e-10
    assert np.linalg.norm(y - v) <= bound, (np.linalg.norm(y - v), bound)
    assert np.array_equal(y, c.ritz_vector(0))
    idx, val = c.top_k(100)
    assert np.array_equal(idx, orc.top_k(y)) and np.array_equal(val, y[idx])
    s = np.sort(v)[::-1][:101]
    if np.min(s[:-1] - s[1:]) > 2 * bound:          # the ranking is determined to within the vector's error bound
        assert np.array_equal(idx, orc.top_k(v))
    return y


def test_eigenvector_centrality_golden(lz, orc, golden, mctx):
    g = golden("rmat_s14_k50")
    perron_check(lz, orc, mctx, g["row_offset"], g["col_idx"], int(g["k"]))


def test_eigenvector_centrality_c2(lz, orc, mctx):
    """C2-sized R-MAT (2^20 vertices, k = 30)."""
    mctx.graph_generate(lz.GraphSpec.rmat(20, 8, 1))
    ro, ci = mctx.csr_download()
    perron_check(lz, orc, mctx, ro, ci, 30)


def graph500_small(lz):
    n, ro, ci = lz.generate_host(lz.GraphSpec.rmat(11, 8, 3, *GRAPH500))
    return ro, ci


def islands(lz):
    """Isolated vertices, a triangle, a path, a star and a denser block: several components of different spectral radius."""
    rng = np.random.default_rng(4)
    u, v = [0, 1, 2, 10, 11, 12, 20, 20, 20, 20], [1, 2, 0, 11, 12, 13, 21, 22, 23, 24]
    blk = rng.integers(30, 90, size=(400, 2))
    u = np.concatenate([u, blk[:, 0]]).astype(np.uint32)
    v = np.concatenate([v, blk[:, 1]]).astype(np.uint32)
    n, ro, ci = lz.csr_from_edges(120, u, v)
    return ro, ci


def bracket_cases(lz, golden):
    for name in ALL_GOLDENS:
        g = golden(name)
        yield name, g["row_offset"], g["col_idx"], int(g["k"])
    yield "graph500_s11", *graph500_small(lz), 30
    yield "islands", *islands(lz), 20


def test_bracket_holds(lz, golden, mctx):
    """lo <= lambda_max <= hi on every golden, a Graph500 graph and a graph with isolated vertices and several components."""
    for name, ro, ci, k in bracket_cases(lz, golden):
        A = adjacency(ro, ci)
        lmax = np.linalg.eigvalsh(A.toarray())[-1] if A.shape[0] <= 4096 else spl.eigsh(A, k=1, which="LA", tol=1e-14)[0][0]
        for reorth in (lz.REORTH_NONE, lz.REORTH_FULL):
            run(mctx, lz, ro, ci, min(k, A.shape[0]), None, reorth)
            mctx.ritz(1)
            lo, hi = mctx.spectral_radius_bounds()
            assert lo <= lmax * (1 + 1e-12) and lmax <= hi, (name, reorth, lo, lmax, hi)


def test_bracket_tight_when_converged(lz, golden, mctx):
    """(hi - lo) / lo <= 1e-6 where y_0 has converged: the connected ER golden at k = 50, and the band golden (relative gap 7e-3,
    not converged at k = 50) at k = 150 with full reorthogonalisation."""
    for name, k, reorth in (("er_n2000_k20", 50, lz.REORTH_NONE), ("band_n4096_k40", 150, lz.REORTH_FULL)):
        g = golden(name)
        ro, ci = g["row_offset"], g["col_idx"]
        assert csg.connected_components(adjacency(ro, ci), directed=False)[0] == 1
        run(mctx, lz, ro, ci, k, None, reorth)
        mctx.ritz(1)
        lo, hi = mctx.spectral_radius_bounds()
        assert (hi - lo) / lo <= 1e-6, (name, lo, hi)
    for name in ("rmat_s12_k30", "rmat_s14_k50"):     # disconnected, but the small components are far below lambda_max
        g = golden(name)
        run(mctx, lz, g["row_offset"], g["col_idx"], 50)
        mctx.ritz(1)
        lo, hi = mctx.spectral_radius_bounds()
        assert (hi - lo) / lo <= 1e-6, (name, lo, hi)


@pytest.mark.parametrize("name", GOLDENS)
def test_katz_through_bracket(lz, golden, mctx, name):
    """alpha = 0.9 / hi is certified below 1 / lambda_max: the resolvent solve succeeds and is Katz."""
    g = golden(name)
    ro, ci, n = g["row_offset"], g["col_idx"], int(g["n"])
    A = adjacency(ro, ci)
    run(mctx, lz, ro, ci, 60)
    mctx.ritz(1)
    lo, hi = mctx.spectral_radius_bounds()
    alpha = 0.9 / hi
    mctx.set_matfun(lz.MATFUN_RESOLVENT, alpha)
    assert mctx.spectral_radius_bounds() == (lo, hi)          # lz_set_matfun keeps the pairs
    mctx.tridiag_expv()
    mctx.multout()
    y = mctx.get_ans()
    assert rel2(y, spl.spsolve((sp.identity(n) - alpha * A).tocsc(), np.ones(n))) < 1e-9


def test_independent_of_existing_path(lz, golden):
    """After lz_ritz the coefficients, a following multOut and the answer are bit-identical to a context that never called it."""
    g = golden("rmat_s14_k50")
    ro, ci, k = g["row_offset"], g["col_idx"], int(g["k"])
    with lz.Context(0) as c0, lz.Context(0) as c1:
        out = []
        for c, with_ritz in ((c0, False), (c1, True)):
            run(c, lz, ro, ci, k)
            c.tridiag_expv()
            if with_ritz:
                c.ritz(8)
            w, z, coef = c.get_eigen()
            c.multout()
            out.append((w, z, coef, c.get_ans(), c.get_tridiag()))
        for a, b in zip(*out):
            if isinstance(a, tuple):
                assert all(np.array_equal(x, y) for x, y in zip(a, b))
            else:
                assert np.array_equal(a, b)


def test_after_overflow_and_state(lz, mctx):
    """lz_ritz works after an EXP solve that overflowed (t * lambda_max = 800); a new run or start vector drops the pairs."""
    ro, ci = graph500_small(lz)
    lmax = np.linalg.eigvalsh(adjacency(ro, ci).toarray())[-1]
    run(mctx, lz, ro, ci, 30)
    mctx.set_matfun(lz.MATFUN_EXP, 800.0 / lmax)
    mctx.tridiag_expv()
    raises_code(lz, -6, mctx.get_eigen)
    th, rho, res = mctx.ritz(2)
    assert abs(th[0] - lmax) <= 1e-9 * lmax and abs(rho[0] - lmax) <= res[0] + 1e-12 * lmax
    lo, hi = mctx.spectral_radius_bounds()
    assert lo <= lmax * (1 + 1e-12) <= hi * (1 + 1e-12)
    mctx.set_matfun(lz.MATFUN_EXP_SCALED, 1.0)
    assert mctx.spectral_radius_bounds() == (lo, hi)
    mctx.lanczos_run(30)
    raises_code(lz, -1, mctx.spectral_radius_bounds)
    mctx.ritz(1)
    mctx.set_start_vector(None)
    raises_code(lz, -1, mctx.ritz_vector, 0)


def ritz_all(c, m):
    th, rho, res = c.ritz(m)
    return th, rho, res, np.stack([c.ritz_vector(j) for j in range(m)])


def test_variants(lz, golden, monkeypatch):
    """fp32 basis (vectors to 1e-6, same theta), unlagged loop (1e-12), CSR SpMV variants (same pairs), and m = 1 against the first
    vector of m = 4 (the block kernel against k_combine). Reorthogonalised runs from a random start, so every pair is well defined."""
    g = golden("rmat_s14_k50")
    ro, ci, k, n = g["row_offset"], g["col_idx"], int(g["k"]), int(g["n"])
    x = np.random.default_rng(3).standard_normal(n)
    m = 4

    def same(a, b, tol):
        assert np.allclose(a[0], b[0], rtol=1e-12, atol=0) and np.allclose(a[1], b[1], rtol=1e-12, atol=0)
        vt = vec_tol(a[0], tol)
        for j in range(m):
            assert np.abs(a[3][j] - b[3][j]).max() < vt[j], j
    with lz.Context(0) as c:
        run(c, lz, ro, ci, k, x, lz.REORTH_FULL)
        ref = ritz_all(c, m)
        th1, _, _, Y1 = ritz_all(c, 1)
        assert th1[0] == ref[0][0] and np.abs(Y1[0] - ref[3][0]).max() < 1e-13
        for v in (lz.SPMV_VECTOR, lz.SPMV_WARP):
            c.set_spmv_variant(v)
            run(c, lz, ro, ci, k, x, lz.REORTH_FULL)
            same(ritz_all(c, m), ref, 1e-12)
        c.set_spmv_variant(lz.SPMV_AUTO)
    with lz.Context(0) as c:
        c.set_basis_precision(lz.BASIS_F32)
        run(c, lz, ro, ci, k)
        th32, _, _, Y32 = ritz_all(c, m)
    with lz.Context(0) as c:
        run(c, lz, ro, ci, k)
        th64, _, _, Y64 = ritz_all(c, m)
    assert np.array_equal(th32, th64)                          # same alpha / beta: the fp32 basis only rounds V
    vt = vec_tol(th64, 1e-6)
    assert all(np.abs(Y32[j] - Y64[j]).max() < vt[j] for j in range(m))
    monkeypatch.setenv("LZ_LAGGED_NORM", "0")
    with lz.Context(0) as c:
        run(c, lz, ro, ci, k, x, lz.REORTH_FULL)
        same(ritz_all(c, m), ref, 1e-12)


def test_validation(lz, golden):
    g = golden("er_n2000_k20")
    ro, ci = g["row_offset"], g["col_idx"]
    with lz.Context(0) as c:
        raises_code(lz, -1, c.ritz, 1)
        c.csr_upload(ro, ci)
        raises_code(lz, -1, c.ritz, 1)                      # no run yet
        raises_code(lz, -1, c.spectral_radius_bounds)
        c.set_start_vector(None)
        c.lanczos_run(10)
        for m in (0, 17, 11):
            raises_code(lz, -1, c.ritz, m)
        raises_code(lz, -1, c.spectral_radius_bounds)       # before lz_ritz
        raises_code(lz, -1, c.ritz_vector, 0)
        c.ritz(3)
        raises_code(lz, -1, c.ritz_vector, 3)
        c.lanczos_run(20)
        c.ritz(16)
        assert c.ritz_vector(15).shape == (int(g["n"]),)


def _final(lz):
    libdir = os.path.join(os.path.dirname(lz.lib_path), "..", "lib")
    subprocess.check_call(["make", "-s", "-C", libdir])
    return os.path.join(libdir, "final")


def test_cpp_driver(lz, golden, tmp_path):
    """final --eigcent --top 10, --ritz 4 and --katz-frac 0.9 agree with the Python results; --katz-frac with --katz is refused."""
    final = _final(lz)
    g = golden("rmat_s12_k30")
    ro, ci, k = g["row_offset"], g["col_idx"], 50
    path = str(tmp_path / "g.mtx")
    lz.write_text(path, ro, ci)
    with lz.Context(0) as c:
        run(c, lz, ro, ci, k)
        th, rho, res = c.ritz(4)
        c.ritz(1)                                  # --eigcent and --katz-frac run m = 1
        idx, val = c.top_k(10)
        lo, hi = c.spectral_radius_bounds()
        c.set_matfun(lz.MATFUN_RESOLVENT, 0.9 / hi)
        c.tridiag_expv()
        c.multout()
        katz_top = c.top_k(10)[0]
    base = [final, "--path", path, "-k", str(k)]

    def go(*extra):
        r = subprocess.run(base + list(extra), capture_output=True, text=True, timeout=300)
        assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
        return r.stdout

    def bracket(out):
        line = next(l for l in out.splitlines() if l.startswith("spectral radius bracket: "))
        return float(line.split()[3]), float(line.split()[4])

    out = go("--eigcent", "--top", "10")
    assert "TOP 10 vertices by eigenvector centrality" in out
    assert [int(l.split()[2]) for l in out.splitlines() if l.startswith("rank ")] == list(idx)
    assert bracket(out) == pytest.approx((lo, hi), rel=1e-15)
    out = go("--ritz", "4")
    rows = [l.split() for l in out.splitlines() if l.startswith("ritz ")]
    assert len(rows) == 4
    for j, r in enumerate(rows):
        assert float(r[2]) == pytest.approx(th[j], rel=1e-15)
        assert float(r[3]) == pytest.approx(rho[j], rel=1e-15)
        assert float(r[4]) == pytest.approx(res[j], rel=1e-12, abs=1e-15 * th[0])
    out = go("--katz-frac", "0.9", "--top", "10")
    assert "Katz centrality" in out and "result finite: yes" in out
    assert bracket(out) == pytest.approx((lo, hi), rel=1e-15)
    alpha = float(next(l for l in out.splitlines() if l.startswith("katz alpha: ")).split()[2])
    assert alpha == pytest.approx(0.9 / hi, rel=1e-15)
    assert [int(l.split()[2]) for l in out.splitlines() if l.startswith("rank ")] == list(katz_top)
    r = subprocess.run(base + ["--katz-frac", "0.9", "--katz", "0.01"], capture_output=True, text=True, timeout=60)
    assert r.returncode == 2
    if lz.device_count() >= 2:
        out = go("--katz-frac", "0.9", "--gpus", "2")
        assert bracket(out) == pytest.approx((lo, hi), rel=1e-12)


@pytest.mark.parametrize("world", [2, 4, 8])
def test_ritz_several_gpus(lz, world):
    if lz.device_count() < world:
        pytest.skip(f"needs {world} GPUs")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={world}", "--master-addr", "127.0.0.1",
           "--master-port", str(29600 + world), os.path.join(ROOT, "tests", "ritz_dist_check.py")]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    assert f"RITZ_DIST_OK {world}" in r.stdout
