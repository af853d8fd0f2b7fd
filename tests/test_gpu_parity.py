"""Parity of the CUDA path (through the C ABI) with the oracle and with the reference's golden output. All need a GPU.

Tolerances (BASELINE.json north_star): e^A·x within 1e-9 relative 2-norm in fp64; top-100 ranking identical
(argsort(-y), stable index tie-break on both sides). Integer-valued SpMV inputs must be bit-exact."""
import json

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

TOL = 1e-9
CASES = ["c1_er_n10000_k20", "er_n2000_k20", "rmat_s12_k30", "rmat_s14_k50", "band_n4096_k40", "er_n257_k10_ragged"]


def rel2(a, b):
    return np.linalg.norm(a - b) / np.linalg.norm(b)


@pytest.fixture(scope="module")
def ctx(lz):
    c = lz.Context(0)
    yield c
    c.close()


@pytest.mark.parametrize("name", CASES)
def test_expv_matches_reference_golden(lz, orc, golden, ctx, name):
    g = golden(name)
    ro, ci, k, n = g["row_offset"], g["col_idx"], int(g["k"]), int(g["n"])
    ctx.csr_upload(ro, ci)
    y = ctx.expv_host(None, k)                      # x = ones, as every reference driver (main.cu:79)
    assert rel2(y, g["ans"]) < TOL
    assert orc.top_gap(g["ans"]) > 1e-6             # the ranking claim is meaningful
    assert np.array_equal(orc.top_k(y), orc.top_k(g["ans"]))
    # T itself is only comparable while the recurrence is still orthogonal: without reorthogonalisation rounding
    # differences (tree vs sequential sums) are amplified once Ritz values converge, in the reference's own
    # serial-vs-CUDA runs as well. e^A x above is the stable quantity; here we pin the leading coefficients.
    alpha, beta = ctx.get_tridiag()
    lead = min(6, k)
    np.testing.assert_allclose(alpha[:lead], g["alpha"][:lead], rtol=1e-8)
    np.testing.assert_allclose(beta[: lead - 1], g["beta"][: lead - 1], rtol=1e-8)
    # random start vector from host memory
    y2 = ctx.expv_host(g["x_random"], k)
    assert rel2(y2, g["ans_random"]) < TOL


@pytest.mark.parametrize("name", ["er_n2000_k20", "rmat_s12_k30", "rmat_s14_k50"])
def test_full_reorth_within_tolerance_of_plain_reference(lz, orc, golden, ctx, name):
    g = golden(name)
    ro, ci, k, n = g["row_offset"], g["col_idx"], int(g["k"]), int(g["n"])
    ctx.csr_upload(ro, ci)
    y = ctx.expv_host(None, k, lz.REORTH_FULL)
    assert rel2(y, g["ans"]) < TOL
    assert np.array_equal(orc.top_k(y), orc.top_k(g["ans"]))
    ans_o, alpha_o, _ = orc.expv(ro, ci, k, np.ones(n), reorth=orc.FULL)     # our CGS2 spec on the CPU
    assert rel2(y, ans_o) < TOL
    # basis is orthonormal to working precision
    Q = np.stack([ctx.get_basis(j) for j in range(k)])
    assert np.abs(Q @ Q.T - np.eye(k)).max() < 1e-12


@pytest.mark.parametrize("variant", ["auto", "vector", "warp"])
@pytest.mark.parametrize("spec_name", ["er", "rmat", "band", "tiny"])
def test_spmv_bit_exact_on_integer_data(lz, orc, ctx, spec_name, variant):
    spec = {"er": lz.GraphSpec.er(30011, 150000, 5), "rmat": lz.GraphSpec.rmat(15, 8, 3),
            "band": lz.GraphSpec.band(20000, 9), "tiny": lz.GraphSpec.er(33, 40, 1)}[spec_name]
    n, ro, ci = lz.generate_host(spec)
    ctx.set_spmv_variant({"auto": lz.SPMV_AUTO, "vector": lz.SPMV_VECTOR, "warp": lz.SPMV_WARP}[variant])
    try:
        ctx.csr_upload(ro, ci)
        rng = np.random.default_rng(7)
        x = rng.integers(-(1 << 20), 1 << 20, n).astype(np.float64)     # sums are exact in fp64 in any order
        assert np.array_equal(ctx.spmv_host(x), orc.spmv(ro, ci, x))
        assert np.array_equal(ctx.spmv_host(np.ones(n)), np.diff(ro).astype(np.float64))
        xr = rng.random(n)
        y, yo = ctx.spmv_host(xr), orc.spmv(ro, ci, xr)
        assert np.abs(y - yo).max() <= 64 * np.finfo(float).eps * max(1.0, np.abs(yo).max())
    finally:
        ctx.set_spmv_variant(lz.SPMV_AUTO)


@pytest.mark.parametrize("narrow", ["0", "1"])
@pytest.mark.parametrize("blocks", ["1", "3"])
def test_sliced_kernel_quad_paths_on_small_inputs(lz, orc, monkeypatch, narrow, blocks):
    """The batched-quad paths of the sliced kernel (4 slices per work unit; the NARROW instantiation handles slices up to 8
    wide 4 chunks x 4 slices at a time) normally switch on only at ~10^7 rows. Forced here on small ragged inputs, with one
    and with several column blocks, in both vertex orders: SpMV must stay bit-exact and e^A x within tolerance."""
    monkeypatch.setenv("LZ_SELL_GROUP", "4")
    monkeypatch.setenv("LZ_SELL_NARROW", narrow)
    monkeypatch.setenv("LZ_SPMV_COLBLOCKS", blocks)
    specs = [lz.GraphSpec.er(30011, 150000, 5), lz.GraphSpec.rmat(15, 8, 3), lz.GraphSpec.band(20000, 9), lz.GraphSpec.er(33, 40, 1),
             lz.GraphSpec.er(4099, 9000, 2)]
    for order in ("d", "n"):
        monkeypatch.setenv("LZ_ORDER", order)
        with lz.Context(0) as c:
            for spec in specs:
                n, ro, ci = lz.generate_host(spec)
                c.csr_upload(ro, ci)
                x = np.random.default_rng(7).integers(-(1 << 20), 1 << 20, n).astype(np.float64)
                assert np.array_equal(c.spmv_host(x), orc.spmv(ro, ci, x))
                assert np.array_equal(c.spmv_host(np.ones(n)), np.diff(ro).astype(np.float64))
            n, ro, ci = lz.generate_host(specs[1])
            c.csr_upload(ro, ci)
            y = c.expv_host(None, 20)
            ref, _, _ = orc.expv(ro, ci, 20, np.ones(n))
            assert rel2(y, ref) < TOL and np.array_equal(orc.top_k(y), orc.top_k(ref))


@pytest.mark.parametrize("spec_name", ["er", "rmat", "band"])
def test_device_generator_matches_host_generator(lz, ctx, spec_name):
    spec = {"er": lz.GraphSpec.er(50000, 300000, 11), "rmat": lz.GraphSpec.rmat(16, 8, 1),
            "band": lz.GraphSpec.band(70001, 5)}[spec_name]
    n, ro, ci = lz.generate_host(spec)
    ctx.graph_generate(spec)
    ro_d, ci_d = ctx.csr_download()
    assert np.array_equal(ro, ro_d) and np.array_equal(ci, ci_d)
    gi = ctx.graph_info()
    deg = np.diff(ro)
    assert (gi.n, gi.nnz, gi.max_degree, gi.empty_rows) == (n, len(ci), deg.max(), int((deg == 0).sum()))


def test_first_basis_vector_and_alpha0(lz, orc, golden, ctx):
    g = golden("rmat_s12_k30")
    ro, ci, n = g["row_offset"], g["col_idx"], int(g["n"])
    ctx.csr_upload(ro, ci)
    ctx.set_start_vector(g["x_random"])
    ctx.lanczos_run(3)
    q0 = ctx.get_basis(0)
    x = g["x_random"]
    np.testing.assert_allclose(q0, x / np.linalg.norm(x), rtol=1e-15)
    a_o, b_o, Q_o = orc.lanczos(ro, ci, 3, x)
    alpha, beta = ctx.get_tridiag()
    np.testing.assert_allclose(alpha, a_o, rtol=1e-12)
    np.testing.assert_allclose(beta, b_o, rtol=1e-12)
    for j in range(3):
        assert rel2(ctx.get_basis(j), Q_o[:, j]) < 1e-11


@pytest.mark.parametrize("k", [1, 2, 5, 64, 200])
def test_device_tridiag_solver_vs_oracle(lz, orc, ctx, k):
    """Runs Lanczos for k steps and compares the on-device eigen-solve + coefficient vector with the oracle's
    restatement of dstevd on the same (alpha, beta) — sign-free quantities only."""
    n, ro, ci = lz.generate_host(lz.GraphSpec.er(3000, 9000, 21))
    ctx.csr_upload(ro, ci)
    ctx.set_start_vector(None)
    ctx.lanczos_run(k, lz.REORTH_FULL if k > 30 else lz.REORTH_NONE)
    alpha, beta = ctx.get_tridiag()
    ctx.tridiag_expv()
    w, Z, c = ctx.get_eigen()
    w_o, Z_o = orc.tridiag_eig(alpha, beta)
    np.testing.assert_allclose(w, w_o, rtol=0, atol=1e-12 * max(1.0, np.abs(w_o).max()))
    T = np.diag(alpha) + (np.diag(beta, 1) + np.diag(beta, -1) if k > 1 else 0)
    assert np.abs(T @ Z - Z * w).max() < 1e-11 * max(1.0, np.abs(w).max())
    assert np.abs(Z.T @ Z - np.eye(k)).max() < 1e-12
    c_o = np.sqrt(n) * (Z_o @ (np.exp(w_o) * Z_o[0]))
    assert rel2(c, c_o) < 1e-11


def test_multout_is_idempotent_and_matches_manual_combination(lz, orc, golden, ctx):
    """The reference's multOut mutates E in place and cannot be called twice (SURVEY appendix A); ours can."""
    g = golden("er_n2000_k20")
    ro, ci, k, n = g["row_offset"], g["col_idx"], int(g["k"]), int(g["n"])
    ctx.csr_upload(ro, ci)
    ctx.set_start_vector(None)
    ctx.lanczos_run(k)
    ctx.tridiag_expv()
    ctx.multout()
    y1 = ctx.get_ans()
    ctx.multout()
    y2 = ctx.get_ans()
    assert np.array_equal(y1, y2)
    _, _, c = ctx.get_eigen()
    Q = np.stack([ctx.get_basis(j) for j in range(k)])
    assert rel2(y1, c @ Q) < 1e-14
    assert rel2(y1, g["ans"]) < TOL


def test_krylov_dimension_edge_cases(lz, orc, ctx):
    n, ro, ci = lz.generate_host(lz.GraphSpec.er(500, 2000, 2))
    ctx.csr_upload(ro, ci)
    x = np.ones(n)
    for k in (1, 2, 3):
        y = ctx.expv_host(x, k)
        yo, _, _ = orc.expv(ro, ci, k, x)
        assert rel2(y, yo) < 1e-12, k
    with pytest.raises(lz.LzError):
        ctx.lanczos_run(0)
    with pytest.raises(lz.LzError):
        ctx.lanczos_run(5, 7)


def test_call_order_errors(lz):
    with lz.Context(0) as c:
        with pytest.raises(lz.LzError):
            c.set_start_vector(None)          # no graph
        n, ro, ci = lz.generate_host(lz.GraphSpec.er(100, 300, 2))
        c.csr_upload(ro, ci)
        with pytest.raises(lz.LzError):
            c.lanczos_run(5)                  # no start vector
        c.set_start_vector(None)
        with pytest.raises(lz.LzError):
            c.tridiag_expv()                  # no decomposition
        c.lanczos_run(5)
        with pytest.raises(lz.LzError):
            c.multout()                       # no coefficients


def test_breakdown_is_reported_not_silent(lz, ctx):
    """Regular graph + constant x: A.1 = d.1 so beta_0 = 0 — the reference divides by zero and returns NaN
    (SURVEY 7.3-2). We must surface it as an error, not hand back NaNs as if they were a result."""
    n = 64
    ro = np.arange(0, 2 * n + 1, 2, dtype=np.uint32)
    ci = np.empty(2 * n, np.uint32)
    for i in range(n):
        ci[2 * i: 2 * i + 2] = sorted(((i - 1) % n, (i + 1) % n))
    ctx.csr_upload(ro, ci)
    with pytest.raises(lz.LzError) as e:
        ctx.expv_host(None, 5)
    assert e.value.code == -6
    y = ctx.expv_host(None, 1)                # k = 1 never divides: e^2 * 1
    np.testing.assert_allclose(y, np.exp(2.0), rtol=1e-14)


@pytest.mark.parametrize("scale,k", [(20, 30)])
def test_c2_size_against_oracle(lz, orc, ctx, scale, k):
    """BASELINE.json configs[1]: R-MAT 2^20, ~16 nnz/row, k=30, fp64 e^A·x + top-100 ranking, vs the CPU oracle
    (and vs the compiled reference itself when oracle/_ref is present)."""
    spec = lz.GraphSpec.rmat(scale, 8, 1)
    ctx.graph_generate(spec)
    ro, ci = ctx.csr_download()
    n = len(ro) - 1
    y = ctx.expv_host(None, k)
    if orc.have_ref():
        ref = orc.run_ref_final(ro, ci, k)["ans"]
    else:
        ref, _, _ = orc.expv(ro, ci, k, np.ones(n))
    assert np.isfinite(ref).all()
    assert rel2(y, ref) < TOL
    assert orc.top_gap(ref) > 1e-7
    assert np.array_equal(orc.top_k(y), orc.top_k(ref))
    yr = ctx.expv_host(None, k, lz.REORTH_FULL)
    assert rel2(yr, ref) < TOL and np.array_equal(orc.top_k(yr), orc.top_k(ref))


def test_full_size_properties_c3(lz, orc, ctx):
    """BASELINE.json configs[2] size (R-MAT 2^24, k=50): too big for the CPU oracle inside a test, so check
    size-independent properties: SpMV of ones = degree vector (exact), linearity of SpMV on integer data (exact),
    Lanczos basis orthonormality under full reorth, T = Q^T A Q consistency (alpha_j = q_j.A.q_j), k-convergence
    (k=40 vs k=50 agree), and determinism (two runs bit-identical)."""
    spec = lz.GraphSpec.rmat(24, 8, 1)
    ctx.graph_generate(spec)
    gi = ctx.graph_info()
    n = gi.n
    assert n == 1 << 24 and 15.5 < gi.nnz / n < 16.0
    ro, ci = ctx.csr_download()
    deg = np.diff(ro).astype(np.float64)
    assert np.array_equal(ctx.spmv_host(np.ones(n)), deg)
    rng = np.random.default_rng(3)
    a = rng.integers(-1000, 1000, n).astype(np.float64)
    b = rng.integers(-1000, 1000, n).astype(np.float64)
    ya, yb, yab = ctx.spmv_host(a), ctx.spmv_host(b), ctx.spmv_host(2 * a - 3 * b)
    assert np.array_equal(yab, 2 * ya - 3 * yb)
    # spot-check rows against a direct gather-sum
    rows = rng.integers(0, n, 2000)
    for r in rows[:200]:
        assert ya[r] == a[ci[ro[r]:ro[r + 1]]].sum()
    y50 = ctx.expv_host(None, 50)
    alpha, beta = ctx.get_tridiag()
    assert np.isfinite(y50).all() and np.all(beta > 0)
    q0, q1 = ctx.get_basis(0), ctx.get_basis(1)
    assert abs(q0 @ q1) < 1e-12 and abs(q1 @ q1 - 1) < 1e-12
    assert abs(q1 @ ctx.spmv_host(q1) - alpha[1]) < 1e-9 * abs(alpha[1])
    y50b = ctx.expv_host(None, 50)
    assert np.array_equal(y50, y50b)                               # deterministic reductions
    y40 = ctx.expv_host(None, 40)
    assert rel2(y40, y50) < 1e-9
    assert np.array_equal(orc.top_k(y40), orc.top_k(y50))
    y50r = ctx.expv_host(None, 50, lz.REORTH_FULL)
    assert rel2(y50r, y50) < TOL and np.array_equal(orc.top_k(y50r), orc.top_k(y50))
    qa, qb = ctx.get_basis(49), ctx.get_basis(3)
    assert abs(qa @ qb) < 1e-12 and abs(qa @ qa - 1) < 1e-12


@pytest.mark.parametrize("scale,k", [(20, 30), (24, 50)])
def test_named_configs_against_reference_summary(lz, ctx, scale, k):
    """BASELINE.json configs[1] (C2: R-MAT 2^20, k=30) and configs[2] (C3: R-MAT 2^24, k=50) against the committed summary of the
    UNMODIFIED reference's answer on the same graph (tests/golden/rmat_s*_summary.npz, made by make_golden_c3.py from
    oracle/_ref/ref_final): sampled + top entries and block sums to 1e-9 relative 2-norm, ||y||, top-100 ranking bit-identical
    (host argsort AND the product's lz_top_k), leading alpha/beta to 1e-8. Plain Lanczos and full reorthogonalisation."""
    import fixture_parity as fp
    path = fp.fixture_path("rmat", scale, k)
    assert path, "summary fixture missing"
    ctx.graph_generate(lz.GraphSpec.rmat(scale, 8, 1))
    for reorth in (lz.REORTH_NONE, lz.REORTH_FULL):
        y = ctx.expv_host(None, k, reorth)
        alpha, beta = ctx.get_tridiag()
        idx, val = ctx.top_k(100)
        r = fp.compare(y, path, alpha, beta, idx, val)
        assert r["top_gap"] > 1e-6                    # the ranking claim is meaningful on this graph
        assert r["rel_2norm"] < TOL and r["rel_2norm_block_sums"] < TOL and r["rel_norm2"] < TOL, r
        assert r["top100_identical"] and r["top256_identical"] and r["top_k_api_identical"], r
        assert r["top_k_api_rel_values"] < TOL
        assert r["alpha_lead_rel"] < 1e-8 and r["beta_lead_rel"] < 1e-8, r


@pytest.mark.parametrize("name", CASES)
def test_top_k_is_the_oracle_ranking(lz, orc, golden, ctx, name):
    """lz_top_k (device radix select) == argsort(-y) with ties towards the lower vertex id, for several m, incl. m > n."""
    g = golden(name)
    n, k = int(g["n"]), int(g["k"])
    ctx.csr_upload(g["row_offset"], g["col_idx"])
    y = ctx.expv_host(None, k)
    for m in (1, 7, 100, 1024):
        idx, val = ctx.top_k(m)
        assert len(idx) == min(m, n)
        assert np.array_equal(idx, orc.top_k(y, m))
        assert np.array_equal(val, y[idx])
    with pytest.raises(lz.LzError):
        ctx.top_k(0)
    with pytest.raises(lz.LzError):
        ctx.top_k(4096)


def test_top_k_ties_and_signs(lz, orc, ctx):
    """Ties go to the lower vertex id (k = 1 on a regular graph: every entry of e^A x is the same number), and the order is
    right for mixed signs, +-0 and tiny graphs (m > n)."""
    n = 4099
    ro = np.arange(0, 2 * n + 1, 2, dtype=np.uint32)
    ci = np.empty(2 * n, np.uint32)
    for i in range(n):
        ci[2 * i: 2 * i + 2] = sorted(((i - 1) % n, (i + 1) % n))
    ctx.csr_upload(ro, ci)
    y = ctx.expv_host(None, 1)
    assert np.all(y == y[0])
    idx, val = ctx.top_k(300)
    assert np.array_equal(idx, np.arange(300, dtype=np.uint32)) and np.all(val == y[0])
    # signed start vector with exact zeros: k = 1 gives y = e^2 * x (cycle: A x . x / x . x ... use the closed form check below)
    nn, ro2, ci2 = lz.generate_host(lz.GraphSpec.er(33, 40, 1))
    ctx.csr_upload(ro2, ci2)
    x = np.random.default_rng(3).integers(-3, 4, nn).astype(np.float64)
    y = ctx.expv_host(x, 6)
    idx, val = ctx.top_k(100)
    assert len(idx) == nn and np.array_equal(idx, orc.top_k(y, 100)) and np.array_equal(val, y[idx])


@pytest.mark.parametrize("name", ["rmat_s14_k50", "c1_er_n10000_k20", "band_n4096_k40"])
def test_fp32_basis_mode_against_reference_float_and_double(lz, orc, golden, name):
    """SURVEY 8f-4: LZ_BASIS_F32 stores V as floats (arithmetic fp64). Held to the reference's OWN single-precision agreement:
    the reference's float build differs from its double build by `ref_f32_vs_f64` (2.7e-7 .. 5.2e-6 on these graphs, committed in
    tests/golden/reference_float.npz from lanczosDecomp<float>); ours must be at least 10x closer to the double answer than that,
    no farther from the reference's float answer than the reference is from itself, and keep alpha/beta of the plain run equal to
    the fp64 run's (the recurrence runs on fp64 copies). Plain, full reorthogonalisation, ranking, get_basis, and switching back."""
    g = golden(name)
    fl = np.load(__import__("os").path.join(__import__("os").path.dirname(__file__), "golden", "reference_float.npz"))
    ref32, d_ref = fl[name + "__ans_f32"].astype(np.float64), float(fl[name + "__ref_f32_vs_f64"])
    ro, ci, k, n = g["row_offset"], g["col_idx"], int(g["k"]), int(g["n"])
    with lz.Context(0) as c:
        c.csr_upload(ro, ci)
        y64 = c.expv_host(None, k)
        a64, b64 = c.get_tridiag()
        c.set_basis_precision(lz.BASIS_F32)
        with pytest.raises(lz.LzError):
            c.lanczos_run(k)                              # the start vector went with the old basis
        y32 = c.expv_host(None, k)
        a32, b32 = c.get_tridiag()
        assert np.array_equal(a32, a64) and np.array_equal(b32, b64)
        assert rel2(y32, g["ans"]) < min(0.1 * d_ref, 1e-6), (rel2(y32, g["ans"]), d_ref)
        assert rel2(y32, ref32) < 1.5 * d_ref
        assert np.array_equal(c.top_k(100)[0], orc.top_k(y32))
        q = np.stack([c.get_basis(j) for j in (0, 1, k - 1)])
        gram = q @ q.T
        assert np.abs(np.diag(gram) - 1).max() < 1e-6 and abs(gram[0, 1]) < 1e-6   # (plain Lanczos: q_{k-1} need not be orthogonal to q_0)
        yr = c.expv_host(None, k, lz.REORTH_FULL)
        assert rel2(yr, g["ans"]) < 1e-6
        Q = np.stack([c.get_basis(j) for j in range(k)])
        assert np.abs(Q @ Q.T - np.eye(k)).max() < 1e-5    # orthonormal to fp32 rounding of the stored vectors
        y2 = c.expv_host(g["x_random"], k)
        assert rel2(y2, g["ans_random"]) < 1e-6
        c.set_basis_precision(lz.BASIS_F64)
        assert np.array_equal(c.expv_host(None, k), y64)  # back to the graded precision: same bits as before


@pytest.mark.parametrize("basis", ["f64", "f32"])
def test_unlagged_loop_still_matches(lz, orc, golden, monkeypatch, basis):
    """LZ_LAGGED_NORM=0 selects the reference-shaped loop (separate normalisation kernel, normalised basis rows) that the lagged
    loops replaced as the default; it stays in the library (and is what multi-GPU reorthogonalised runs use), so it stays tested:
    plain and reorthogonalised, both basis precisions, same answers as the default loop to rounding."""
    monkeypatch.setenv("LZ_LAGGED_NORM", "0")
    g = golden("rmat_s14_k50")
    ro, ci, k = g["row_offset"], g["col_idx"], int(g["k"])
    tol = TOL if basis == "f64" else 1e-6
    with lz.Context(0) as c:
        if basis == "f32":
            c.set_basis_precision(lz.BASIS_F32)
        c.csr_upload(ro, ci)
        for reorth in (lz.REORTH_NONE, lz.REORTH_FULL):
            y = c.expv_host(None, k, reorth)
            assert rel2(y, g["ans"]) < tol, (basis, reorth, rel2(y, g["ans"]))
            assert np.array_equal(c.top_k(100)[0], orc.top_k(y))
            q = np.stack([c.get_basis(j) for j in (0, 1, k - 1)])
            gram = q @ q.T
            unit = 1e-12 if basis == "f64" else 1e-6
            assert np.abs(np.diag(gram) - 1).max() < unit and abs(gram[0, 1]) < unit     # read-out is normalised
            if reorth:                                   # plain Lanczos loses orthogonality by step 50 (5e-4 here); reorth keeps it
                assert np.abs(gram - np.eye(3)).max() < (1e-12 if basis == "f64" else 1e-5)
        alpha, beta = c.get_tridiag()
        assert np.all(np.isfinite(alpha)) and np.all(beta > 0)


def test_analytic_eigen_combination(lz, orc, ctx):
    """The reference's analytic test method (serial/tests/numerical_test.cc:74-116; tests/test_oracle.py builds the same problem
    for the oracle): x is a combination of 100 eigenvectors of A, so e^A x is known in closed form. Recorded behaviour of the
    reference (serial/output/numerical_test_output.txt): useless at k = 5, 3.5e-11 at k = 20, 4e-15 at k = 25."""
    from test_oracle import analytic_eigen_combination
    n, ro, ci = lz.generate_host(lz.GraphSpec.er(1500, 6000, 17))
    x, y = analytic_eigen_combination(ro, ci)
    ctx.csr_upload(ro, ci)
    rel = {}
    for k in (5, 10, 20, 30):
        rel[k] = rel2(ctx.expv_host(x, k), y)
        ans_o, _, _ = orc.expv(ro, ci, k, x)
        assert rel2(ctx.expv_host(x, k), ans_o) < TOL
    assert rel[5] > 1e-3 and 1e-8 < rel[10] < 1e-4 and rel[20] < 1e-11 and rel[30] < 1e-11, rel
    assert rel2(ctx.expv_host(x, 30, lz.REORTH_FULL), y) < 1e-11


def test_cpp_api_driver_matches_reference_golden(lz, golden, tmp_path):
    """The C++ mirror of the reference API (lib/final: adjMatrix -> lanczosDecomp -> eigenDecomp -> multOut) reproduces the
    reference's answer through the reference's own text format."""
    import os
    import subprocess
    libdir = os.path.join(os.path.dirname(lz.lib_path), "..", "lib")
    subprocess.check_call(["make", "-s", "-C", libdir])
    g = golden("rmat_s12_k30")
    mtx, ans, out = str(tmp_path / "g.mtx"), str(tmp_path / "ans.f64"), str(tmp_path / "out.txt")
    lz.write_text(mtx, g["row_offset"], g["col_idx"])
    g["ans"].astype(np.float64).tofile(ans)
    r = subprocess.run([os.path.join(libdir, "final"), "--path", mtx, "-k", str(int(g["k"])), "--check", ans, "--write", out, "--top", "100"],
                       capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    assert "Relative norm of differences" in r.stdout
    y = np.loadtxt(out)
    assert np.linalg.norm(y - g["ans"]) / np.linalg.norm(g["ans"]) < TOL
    import oracle as orc_
    ranked = [int(l.split()[2]) for l in r.stdout.splitlines() if l.startswith("rank ")]
    assert ranked == list(orc_.top_k(g["ans"], 100))          # lanczosDecomp::top_k through the C++ mirror
    # generated graph + reorth + Barabasi-Albert constructor paths run and give finite answers
    for extra in (["--graph", "rmat", "--scale", "14", "-k", "20", "--reorth"], ["--graph", "ba", "-n", "5000", "-b", "4", "-k", "8"]):
        r = subprocess.run([os.path.join(libdir, "final")] + extra, capture_output=True, text=True, timeout=300)
        assert r.returncode == 0 and "result finite: yes" in r.stdout, r.stdout[-1500:] + r.stderr[-1500:]


@pytest.mark.parametrize("order", ["natural", "degree"])
def test_vertex_order_modes_give_the_same_answer(lz, orc, order, monkeypatch):
    """The internal vertex order (degree-sorted, or natural for band-like graphs) is invisible to the caller: both
    orders, forced through LZ_ORDER, reproduce the oracle on a banded and on a skewed graph."""
    monkeypatch.setenv("LZ_ORDER", order[0])
    with lz.Context(0) as c:
        for spec, k in ((lz.GraphSpec.band(1 << 16, 5), 25), (lz.GraphSpec.rmat(13, 8, 4), 25)):
            n, ro, ci = lz.generate_host(spec)
            c.csr_upload(ro, ci)
            y = c.expv_host(None, k)
            ref, _, _ = orc.expv(ro, ci, k, np.ones(n))
            assert rel2(y, ref) < TOL
            assert np.array_equal(orc.top_k(y), orc.top_k(ref))
            x = np.random.default_rng(1).integers(-99, 99, n).astype(np.float64)
            assert np.array_equal(c.spmv_host(x), orc.spmv(ro, ci, x))


def test_band_like_graph_keeps_natural_order_and_is_fast_path(lz, orc):
    """Large banded graph: the loader must pick the natural order by itself (max degree small, entries near the diagonal),
    and the answer must match the oracle."""
    spec = lz.GraphSpec.band(1 << 20, 5)
    with lz.Context(0) as c:
        c.graph_generate(spec)
        ro, ci = c.csr_download()
        n = len(ro) - 1
        y = c.expv_host(None, 30)
    ref, _, _ = orc.expv(ro, ci, 30, np.ones(n))
    assert rel2(y, ref) < TOL


def test_convergence_estimate_matches_actual_change(lz, orc, golden, ctx):
    """lz_estimate_change(k') = ||y_k - y_k'|| / ||y_k|| from the tridiagonal alone; compare with the change actually
    observed between two full runs (oracle-side check: the same quantity from the CPU restatement)."""
    g = golden("c1_er_n10000_k20")
    ro, ci, n = g["row_offset"], g["col_idx"], int(g["n"])
    ctx.csr_upload(ro, ci)
    y20 = ctx.expv_host(None, 20)
    est = {kp: ctx.estimate_change(kp) for kp in (8, 12, 16)}
    for kp, e in est.items():
        ykp, _, _ = orc.expv(ro, ci, kp, np.ones(n))
        actual = rel2(ykp, y20)
        assert e == pytest.approx(actual, rel=1e-3, abs=1e-13), (kp, e, actual)
    assert est[8] > est[12] > est[16]
    with pytest.raises(lz.LzError):
        ctx.estimate_change(20)
    # lz_choose_k: the smallest k' whose whole tail [k', k) meets the tolerance, consistent with the point estimates
    for tol in (1e-6, 1e-10, 1e-13):
        kc, e = ctx.choose_k(tol)
        assert 1 <= kc <= 20
        if kc < 20:
            assert e <= tol and all(ctx.estimate_change(kp) <= tol for kp in range(kc, 20))
            if kc > 1:
                assert ctx.estimate_change(kc - 1) > tol
            yk, _, _ = orc.expv(ro, ci, kc, np.ones(n))
            assert rel2(yk, y20) <= max(10 * tol, 1e-12)
    assert ctx.choose_k(1e-6)[0] <= ctx.choose_k(1e-10)[0] <= ctx.choose_k(1e-13)[0]
    assert ctx.choose_k(1e-300)[0] == 20            # nothing short of k reproduces the k-step answer that closely
    with pytest.raises(lz.LzError):
        ctx.choose_k(0.0)


@pytest.mark.parametrize("always", ["0", "1"])
def test_reorth_second_pass_path(always):
    """LZ_REORTH_FULL repeats the Gram-Schmidt pass only when needed; force it every step to exercise that path too."""
    import json
    import os
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    env = dict(os.environ, LZ_REORTH_ALWAYS_TWICE=always)
    r = subprocess.run([sys.executable, os.path.join(root, "tests", "reorth_twice_check.py")], capture_output=True, text=True, env=env, timeout=300)
    assert r.returncode == 0, r.stderr[-2000:]
    out = json.loads(r.stdout.strip().splitlines()[-1])
    assert out["rel"] < TOL and out["orth"] < 1e-12
    assert out["second_passes"] == (29 if always == "1" else out["second_passes"])
    if always == "0":
        assert out["second_passes"] <= 29


def test_bench_dump_outputs_match_reference_golden(lz, orc, golden, tmp_path):
    """bench.py --dump-outputs on C1 (the graph of c1_er_n10000_k20) writes the last timed step's e^A x and tridiagonal: the
    reference's answer to the same tolerances as above, next to the usual result line."""
    import json
    import os
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--workload", "c1", "--steps", "2", "--warmup", "1",
                        "--no-cpu-baseline", "--no-f32-detail", "--dump-outputs", str(tmp_path)], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    assert json.loads(r.stdout.strip().splitlines()[-1])["steps"] == 2
    g = golden("c1_er_n10000_k20")
    y, alpha, beta = (np.load(tmp_path / f"{f}.npy") for f in ("ans", "alpha", "beta"))
    assert rel2(y, g["ans"]) < TOL and np.array_equal(orc.top_k(y), orc.top_k(g["ans"]))
    np.testing.assert_allclose(alpha[:6], g["alpha"][:6], rtol=1e-8)
    np.testing.assert_allclose(beta[:5], g["beta"][:5], rtol=1e-8)
