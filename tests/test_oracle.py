"""Pins the CPU oracle (oracle/lanczos_oracle.c) against the reference's own output.

Golden vectors in tests/golden/*.npz were produced by the UNMODIFIED reference compiled into oracle/_ref (see
tests/golden/make_golden.py). Where oracle/_ref exists (build container, and the GPU box via gpurun) the reference is also
re-run live on a fresh seed. No GPU needed."""
import json

import numpy as np
import pytest

CASES = ["c1_er_n10000_k20", "er_n2000_k20", "rmat_s12_k30", "rmat_s14_k50", "band_n4096_k40", "er_n257_k10_ragged"]


def rel2(a, b):
    return np.linalg.norm(a - b) / np.linalg.norm(b)


@pytest.mark.parametrize("name", CASES)
def test_generator_reproduces_golden_graph(lz, golden, name):
    g = golden(name)
    s = json.loads(str(g["spec"]))
    spec = lz.GraphSpec(**s)
    n, ro, ci = lz.generate_host(spec)
    assert n == int(g["n"])
    assert np.array_equal(ro, g["row_offset"]) and np.array_equal(ci, g["col_idx"])
    # simple undirected graph: symmetric, no self loops, sorted unique columns, last vertex not isolated
    rows = np.repeat(np.arange(n, dtype=np.uint32), np.diff(ro))
    assert not np.any(rows == ci)
    fwd = set(zip(rows.tolist(), ci.tolist()))
    assert len(fwd) == len(ci) and all((c, r) in fwd for r, c in list(fwd)[:2000])
    assert ro[n] > ro[n - 1]


@pytest.mark.parametrize("name", CASES)
def test_oracle_matches_reference_golden(orc, golden, name):
    g = golden(name)
    ro, ci, k, n = g["row_offset"], g["col_idx"], int(g["k"]), int(g["n"])
    ans, alpha, beta = orc.expv(ro, ci, k, np.ones(n))
    # the recurrence is restated operation by operation: alpha/beta must match the reference to the last bits
    np.testing.assert_allclose(alpha, g["alpha"], rtol=1e-13, atol=0)
    np.testing.assert_allclose(beta, g["beta"], rtol=1e-13, atol=0)
    assert rel2(ans, g["ans"]) < 1e-12
    assert np.array_equal(orc.top_k(ans), orc.top_k(g["ans"]))
    # the reference's own serial/ tree agrees with its parallel-final host path
    assert rel2(g["ans_serial"], g["ans"]) < 1e-14
    # random start vector
    ans_r, alpha_r, _ = orc.expv(ro, ci, k, g["x_random"])
    np.testing.assert_allclose(alpha_r, g["alpha_random"], rtol=1e-13, atol=0)
    assert rel2(ans_r, g["ans_random"]) < 1e-12


@pytest.mark.parametrize("name", ["er_n2000_k20", "rmat_s12_k30", "band_n4096_k40"])
def test_oracle_arnoldi_variant_matches_serial_reference(orc, golden, name):
    g = golden(name)
    ro, ci, k, n = g["row_offset"], g["col_idx"], int(g["k"]), int(g["n"])
    ans, alpha, _ = orc.expv(ro, ci, k, np.ones(n), reorth=orc.ARNOLDI)
    np.testing.assert_allclose(alpha, g["alpha_arnoldi"], rtol=1e-12, atol=1e-12)
    assert rel2(ans, g["ans_arnoldi"]) < 1e-12


@pytest.mark.parametrize("name", ["er_n2000_k20", "rmat_s12_k30"])
def test_full_reorth_spec_agrees_with_plain_reference(orc, golden, name):
    """LZ_REORTH_FULL's specification (CGS2 every step) stays within the 1e-9 bar of the reference's plain answer."""
    g = golden(name)
    ro, ci, k, n = g["row_offset"], g["col_idx"], int(g["k"]), int(g["n"])
    ans, _, _ = orc.expv(ro, ci, k, np.ones(n), reorth=orc.FULL)
    assert rel2(ans, g["ans"]) < 1e-9
    assert np.array_equal(orc.top_k(ans), orc.top_k(g["ans"]))
    # and the basis really is orthonormal
    _, _, Q = orc.lanczos(ro, ci, k, np.ones(n), reorth=orc.FULL)
    assert np.abs(Q.T @ Q - np.eye(k)).max() < 1e-13


def test_spmv_restatement(orc, golden):
    g = golden("rmat_s12_k30")
    ro, ci, n = g["row_offset"], g["col_idx"], int(g["n"])
    assert np.array_equal(orc.spmv(ro, ci, np.ones(n)), np.diff(ro).astype(np.float64))   # A.1 = degrees, exact
    rng = np.random.default_rng(0)
    x = rng.integers(-1000, 1000, n).astype(np.float64)                                    # integer data: exact sums
    import scipy.sparse as sp
    A = sp.csr_matrix((np.ones(len(ci)), ci, ro), shape=(n, n))
    assert np.array_equal(orc.spmv(ro, ci, x), A @ x)


@pytest.mark.parametrize("k", [1, 2, 3, 17, 50, 100])
def test_tridiag_restatement_vs_lapack(orc, k):
    """lzo_tridiag_eig states dstevd's contract; LAPACK (via SciPy) is the third-party arithmetic the reference calls."""
    from scipy.linalg import eigh_tridiagonal
    rng = np.random.default_rng(k)
    a, b = rng.normal(size=k) * 5, np.abs(rng.normal(size=max(k - 1, 0))) + 0.1
    w, Z = orc.tridiag_eig(a, b)
    if k == 1:
        assert w[0] == a[0] and abs(Z[0, 0]) == 1.0
        return
    w_ref, Z_ref = eigh_tridiagonal(a, b)
    np.testing.assert_allclose(w, w_ref, rtol=0, atol=1e-13 * max(1.0, np.abs(w_ref).max()))
    T = np.diag(a) + np.diag(b, 1) + np.diag(b, -1)
    assert np.abs(T @ Z - Z * w).max() < 1e-12 * max(1.0, np.abs(w).max())
    assert np.abs(Z.T @ Z - np.eye(k)).max() < 1e-13
    # sign-free functional used by multOut: Z (e^w . Z[0,:])
    c, c_ref = Z @ (np.exp(w) * Z[0]), Z_ref @ (np.exp(w_ref) * Z_ref[0])
    assert rel2(c, c_ref) < 1e-12


def test_multout_layouts_agree(orc, golden):
    g = golden("er_n257_k10_ragged")
    ro, ci, k, n = g["row_offset"], g["col_idx"], int(g["k"]), int(g["n"])
    a, b, Q = orc.lanczos(ro, ci, k, np.ones(n))
    w, Z = orc.tridiag_eig(a, b)
    y0, c0 = orc.multout(w, Z, Q, np.sqrt(n), qtrans=False)
    y1, c1 = orc.multout(w, Z, np.ascontiguousarray(Q.T), np.sqrt(n), qtrans=True)
    assert np.array_equal(c0, c1) and rel2(y1, y0) < 1e-15
    assert rel2(y0, g["ans"]) < 1e-12


def test_oracle_vs_scipy_expm_multiply(orc, golden):
    """Independent check of the whole method (SURVEY.md section 6: 5.7e-13 on C1)."""
    from scipy.sparse import csr_matrix
    from scipy.sparse.linalg import expm_multiply
    g = golden("c1_er_n10000_k20")
    ro, ci, n = g["row_offset"], g["col_idx"], int(g["n"])
    A = csr_matrix((np.ones(len(ci)), ci, ro), shape=(n, n))
    y = expm_multiply(A, np.ones(n))
    assert rel2(g["ans"], y) < 1e-11
    assert np.array_equal(orc.top_k(g["ans"]), orc.top_k(y))


def test_check_ans_and_ranking_helpers(orc):
    a = np.array([1.0, 5.0, 5.0, 2.0, -3.0])
    b = np.array([1.0, 5.0, 4.0, 2.0, -3.0])
    mx, mi, nd, rel = orc.check_ans(a, b)
    assert (mx, mi) == (1.0, 2) and nd == 1.0 and rel == pytest.approx(1.0 / np.linalg.norm(b))
    assert orc.top_k(a, 3).tolist() == [1, 2, 3]          # tie -> lower index first


def test_live_reference_on_fresh_seed(lz, orc):
    """Re-runs the compiled reference (oracle/_ref) when present: fresh seed, CSR injection."""
    if not orc.have_ref():
        pytest.skip("oracle/_ref not built here (needs /root/reference)")
    n, ro, ci = lz.generate_host(lz.GraphSpec.rmat(13, 8, 99))
    r = orc.run_ref_final(ro, ci, 30)
    ans, alpha, beta = orc.expv(ro, ci, 30, np.ones(n))
    np.testing.assert_allclose(alpha, r["alpha"], rtol=1e-13)
    np.testing.assert_allclose(beta, r["beta"], rtol=1e-13)
    assert rel2(ans, r["ans"]) < 1e-12
    assert np.array_equal(orc.top_k(ans), orc.top_k(r["ans"]))


def _csr_from_dense(A):
    n = A.shape[0]
    ro = np.zeros(n + 1, dtype=np.uint32)
    ro[1:] = np.cumsum((A != 0).sum(axis=1))
    ci = np.concatenate([np.nonzero(A[i])[0] for i in range(n)]).astype(np.uint32)
    return ro, ci


def test_oracle_closed_forms(orc):
    """Pins the restatement independently of the reference (SURVEY.md section 8c): graphs whose e^A x is known in closed form.
    K_n and the star have 2 resp. 3 distinct eigenvalues, so Lanczos is exact after 2 resp. 3 steps for a generic x."""
    rng = np.random.default_rng(11)
    # complete graph: A = J - I  =>  e^A x = e^-1 (x + (e^n - 1)/n (1.x) 1)
    n = 40
    A = np.ones((n, n)) - np.eye(n)
    ro, ci = _csr_from_dense(A)
    x = 1.0 + rng.random(n)
    y, alpha, beta = orc.expv(ro, ci, 2, x)
    exact = np.exp(-1.0) * (x + (np.expm1(float(n)) / n) * x.sum())
    assert rel2(y, exact) < 1e-12
    # star: centre 0, eigenvalues +-sqrt(n-1) and 0
    n = 50
    A = np.zeros((n, n)); A[0, 1:] = 1; A[1:, 0] = 1
    ro, ci = _csr_from_dense(A)
    x = 1.0 + rng.random(n)
    y, _, _ = orc.expv(ro, ci, 3, x)
    w, V = np.linalg.eigh(A)
    assert rel2(y, V @ (np.exp(w) * (V.T @ x))) < 1e-12
    # cycle (circulant: e^A x by FFT, eigenvalues 2 cos(2 pi j / n)) and path (eigenvalues 2 cos(pi j / (n + 1)))
    n = 64
    A = np.zeros((n, n))
    for i in range(n):
        A[i, (i + 1) % n] = A[(i + 1) % n, i] = 1
    ro, ci = _csr_from_dense(A)
    x = rng.random(n)
    y, _, _ = orc.expv(ro, ci, 30, x)
    lam = 2.0 * np.cos(2.0 * np.pi * np.arange(n) / n)
    exact = np.real(np.fft.ifft(np.exp(lam) * np.fft.fft(x)))
    assert rel2(y, exact) < 1e-10
    A[0, n - 1] = A[n - 1, 0] = 0                       # open the cycle: path
    ro, ci = _csr_from_dense(A)
    y, _, _ = orc.expv(ro, ci, 30, x)
    j = np.arange(1, n + 1)
    S = np.sqrt(2.0 / (n + 1)) * np.sin(np.pi * np.outer(j, j) / (n + 1))
    exact = S @ (np.exp(2.0 * np.cos(np.pi * j / (n + 1))) * (S @ x))
    assert rel2(y, exact) < 1e-10


def test_oracle_regular_graph_with_nonconstant_x(orc):
    """d-regular graph: with x = ones the reference breaks down (beta_0 = 0, NaN); a non-constant x must work and agree with
    the dense eigendecomposition. Circulant 4-regular graph on 101 vertices."""
    n = 101
    A = np.zeros((n, n))
    for i in range(n):
        for s in (1, 7):
            A[i, (i + s) % n] = A[(i + s) % n, i] = 1
    ro, ci = _csr_from_dense(A)
    assert np.all(np.diff(ro) == 4)
    x = 1.0 + np.random.default_rng(3).random(n)
    y, _, _ = orc.expv(ro, ci, 35, x)
    w, V = np.linalg.eigh(A)
    assert rel2(y, V @ (np.exp(w) * (V.T @ x))) < 1e-10
    y1, _, _ = orc.expv(ro, ci, 5, np.ones(n))          # the documented breakdown: not finite, and not silently "fixed"
    assert not np.all(np.isfinite(y1))


def analytic_eigen_combination(ro, ci, n_pairs=100, seed=1234):
    """The reference's own analytic test method (serial/tests/numerical_test.cc:74-116): x = sum_i c_i v_i over `n_pairs`
    eigenpairs of A with c_i ~ U(0,1), so that e^A x = sum_i c_i e^{lambda_i} v_i exactly. The reference read MATLAB-computed
    eigenpairs from data files that are not in the repository; here they come from a dense symmetric eigensolver."""
    n = len(ro) - 1
    A = np.zeros((n, n))
    rows = np.repeat(np.arange(n), np.diff(ro))
    A[rows, ci] = 1.0
    w, V = np.linalg.eigh(A)
    pick = np.argsort(-np.abs(w))[:n_pairs]                   # "the first 100 eigenpairs": largest magnitude, as MATLAB's eigs returns
    c = np.random.default_rng(seed).random(n_pairs)
    x = V[:, pick] @ c
    y = V[:, pick] @ (c * np.exp(w[pick]))
    return x, y


def test_oracle_analytic_eigen_combination(lz, orc):
    """Same construction and the same behaviour as the reference's recorded outcomes (serial/output/numerical_test_output.txt:
    useless at k = 5, 3.5e-11 at k = 20, 4e-15 at k = 25 on its 2114-vertex graph): the error falls steeply with k."""
    n, ro, ci = lz.generate_host(lz.GraphSpec.er(1500, 6000, 17))
    x, y = analytic_eigen_combination(ro, ci)
    rel = {}
    for k in (5, 10, 20, 30, 45):
        ans, _, _ = orc.expv(ro, ci, k, x)
        rel[k] = np.linalg.norm(ans - y) / np.linalg.norm(y)
    assert rel[5] > 1e-3 and 1e-8 < rel[10] < 1e-4 and rel[20] < 1e-11 and rel[30] < 1e-10 and rel[45] < 1e-11, rel
    # from k = 20 on the error sits at rounding level (5e-15 .. 1e-14, depending on the host's LAPACK), where the order of
    # two k's is noise: past that point a larger k may only stay at that level
    assert rel[5] > rel[10] > rel[20] and rel[30] <= max(rel[20], 1e-14), rel
