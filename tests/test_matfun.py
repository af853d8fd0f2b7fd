"""Matrix functions on the Krylov basis (lz_set_matfun): e^{tA} x at any inverse temperature t, the shifted e^{t(A - sI)} x
that never overflows, and the resolvent (I - alpha A)^{-1} x (Katz centrality). All need a GPU.

References: dense eigh for small graphs, f(T) on the CPU oracle's Lanczos alpha/beta/Q for Krylov-level checks, scipy's sparse
solver for the resolvent. TOL is the suite's 1e-9 relative 2-norm."""
import functools
import os
import subprocess

import numpy as np
import pytest
import scipy.sparse as sp
import scipy.sparse.linalg as spl

pytestmark = pytest.mark.gpu

TOL = 1e-9
GOLDENS = ["er_n2000_k20", "rmat_s12_k30", "band_n4096_k40"]
GRAPH500 = (.57, .19, .19)   # Graph500 R-MAT quadrant probabilities: lambda_max grows past exp's range with the scale


def rel2(a, b):
    return np.linalg.norm(a - b) / np.linalg.norm(b)


@pytest.fixture(scope="module")
def ctx(lz):
    c = lz.Context(0)
    yield c
    c.close()


@pytest.fixture
def mctx(lz, ctx):
    """The module context, back on the default function whatever the test left behind."""
    yield ctx
    ctx.set_matfun(lz.MATFUN_EXP, 1.0)


def adjacency(ro, ci):
    n = len(ro) - 1
    return sp.csr_matrix((np.ones(len(ci)), ci.astype(np.int64), ro.astype(np.int64)), shape=(n, n))


@functools.lru_cache(maxsize=4)
def dense_eigh(name):
    g = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", name + ".npz"))
    return np.linalg.eigh(adjacency(g["row_offset"], g["col_idx"]).toarray())


def krylov_f(orc, ro, ci, k, x, f):
    """||x|| Q f(T) e1 from the oracle's Lanczos at dimension k -> (vector, Ritz values)."""
    a, b, Q = orc.lanczos(ro, ci, k, x)
    th, Z = np.linalg.eigh(np.diag(a) + np.diag(b, 1) + np.diag(b, -1))
    return np.linalg.norm(x) * (Q @ (Z @ (f(th) * Z[0]))), th


def raises_code(lz, code, fn, *a):
    with pytest.raises(lz.LzError) as e:
        fn(*a)
    assert e.value.code == code, str(e.value)
    return str(e.value)


def graph500_small(lz):
    """Graph500 R-MAT small enough for a dense eigensolver; t chosen so that t * lambda_max = 800 > log(DBL_MAX)."""
    n, ro, ci = lz.generate_host(lz.GraphSpec.rmat(11, 8, 3, *GRAPH500))
    lam, V = np.linalg.eigh(adjacency(ro, ci).toarray())
    return ro, ci, lam, V, 800.0 / lam[-1]


def test_default_function_is_bit_identical(lz, golden):
    """(EXP, 1.0) is the default: selecting it, and coming back to it from the other kinds, changes no bit of the answer or
    of the coefficients."""
    with lz.Context(0) as c0, lz.Context(0) as c1:
        for name in ("rmat_s12_k30", "er_n2000_k20"):
            g = golden(name)
            k = int(g["k"])
            c0.csr_upload(g["row_offset"], g["col_idx"])
            c1.csr_upload(g["row_offset"], g["col_idx"])
            y0 = c0.expv_host(None, k)
            _, _, coef0 = c0.get_eigen()
            c1.set_matfun(lz.MATFUN_EXP, 1.0)
            assert np.array_equal(c1.expv_host(None, k), y0)
            for kind, p in ((lz.MATFUN_EXP_SCALED, 2.0), (lz.MATFUN_RESOLVENT, 0.01), (lz.MATFUN_EXP, 0.5)):
                c1.set_matfun(kind, p)
                c1.expv_host(None, k)
            c1.set_matfun(lz.MATFUN_EXP, 1.0)
            assert np.array_equal(c1.expv_host(None, k), y0)
            assert np.array_equal(c1.get_eigen()[2], coef0)
            assert c1.matfun_scale() == 0.0


@pytest.mark.parametrize("name", GOLDENS)
@pytest.mark.parametrize("t", [0.25, 0.5, 2.0])
def test_exp_inverse_temperature(lz, orc, golden, mctx, name, t):
    """e^{tA} x against ||x|| Q e^{tT} e1 of the oracle's Lanczos at the same k, and against the dense e^{tA} x where the
    convergence estimate shows the Krylov answer has converged."""
    g = golden(name)
    ro, ci, k, n = g["row_offset"], g["col_idx"], int(g["k"]), int(g["n"])
    mctx.csr_upload(ro, ci)
    mctx.set_matfun(lz.MATFUN_EXP, t)
    y = mctx.expv_host(None, k)
    assert mctx.matfun_scale() == 0.0
    ref, _ = krylov_f(orc, ro, ci, k, np.ones(n), lambda th: np.exp(t * th))
    assert rel2(y, ref) < TOL
    kc, _ = mctx.choose_k(1e-12)
    if kc < k:
        lam, V = dense_eigh(name)
        assert rel2(y, V @ (np.exp(t * lam) * V.sum(axis=0))) < TOL


def test_scaled_exp_never_overflows(lz, orc, mctx):
    """t * lambda_max = 800: EXP overflows and fails; EXP_SCALED gives e^{t(A - sI)} x, which in log domain is the dense
    e^{tA} x, with the dense answer's ranking."""
    ro, ci, lam, V, t = graph500_small(lz)
    n, k = len(ro) - 1, 30
    mctx.csr_upload(ro, ci)
    mctx.set_matfun(lz.MATFUN_EXP, t)
    raises_code(lz, -6, mctx.expv_host, None, k)
    mctx.set_matfun(lz.MATFUN_EXP_SCALED, t)
    y = mctx.expv_host(None, k)
    ls = mctx.matfun_scale()
    assert np.all(np.isfinite(y)) and ls > 709
    ref = V @ (np.exp(t * (lam - lam[-1])) * V.sum(axis=0))          # e^{t(A - lambda_max I)} x
    assert rel2(y * np.exp(ls - t * lam[-1]), ref) < TOL
    assert orc.top_gap(ref) > 1e-6
    assert np.array_equal(mctx.top_k(100)[0], orc.top_k(ref))


@pytest.mark.parametrize("name", GOLDENS)
def test_scaled_exp_equals_exp_where_finite(lz, orc, golden, mctx, name):
    g = golden(name)
    k = int(g["k"])
    mctx.csr_upload(g["row_offset"], g["col_idx"])
    y = mctx.expv_host(None, k)
    top = mctx.top_k(100)[0]
    mctx.set_matfun(lz.MATFUN_EXP_SCALED, 1.0)
    ys = mctx.expv_host(None, k)
    ls = mctx.matfun_scale()
    w, _, _ = mctx.get_eigen()
    assert ls == w[-1]
    assert rel2(ys * np.exp(ls), y) < 1e-13
    assert np.array_equal(orc.top_k(ys), orc.top_k(y))
    assert np.array_equal(mctx.top_k(100)[0], top)


def test_graph500_scale20_where_exp_overflows(lz, orc, mctx):
    """Graph500 R-MAT at scale 20, edge factor 8 (lambda_max ~ 839): the unshifted exponential has no finite answer, the
    shifted one matches the oracle's Krylov answer in log domain, ranking included."""
    k = 30
    mctx.graph_generate(lz.GraphSpec.rmat(20, 8, 1, *GRAPH500))
    ro, ci = mctx.csr_download()
    n = len(ro) - 1
    msg = raises_code(lz, -6, mctx.expv_host, None, k)
    assert "not finite" in msg
    mctx.set_matfun(lz.MATFUN_EXP_SCALED, 1.0)
    y = mctx.expv_host(None, k)
    ls = mctx.matfun_scale()
    ref, th = krylov_f(orc, ro, ci, k, np.ones(n), lambda th: np.exp(th - th.max()))
    assert th.max() > 709
    assert rel2(y * np.exp(ls - th.max()), ref) < TOL
    assert np.array_equal(orc.top_k(y), orc.top_k(ref))
    assert np.array_equal(mctx.top_k(100)[0], orc.top_k(ref))


@pytest.mark.parametrize("name", GOLDENS)
def test_resolvent_is_katz(lz, orc, golden, mctx, name):
    """(I - alpha A)^{-1} x against a sparse direct solve for alpha = 0.5 / lambda_max and 0.9 / lambda_max at a Krylov dimension
    the convergence estimate accepts; alpha past 1 / theta_max fails with its own message; alpha = 0 gives x back."""
    g = golden(name)
    ro, ci, n = g["row_offset"], g["col_idx"], int(g["n"])
    A = adjacency(ro, ci)
    lmax = spl.eigsh(A, k=1, which="LA")[0][0]
    x = np.ones(n)
    k = 60
    mctx.csr_upload(ro, ci)
    for frac in (0.5, 0.9):
        alpha = frac / lmax
        mctx.set_matfun(lz.MATFUN_RESOLVENT, alpha)
        y = mctx.expv_host(None, k)
        assert mctx.choose_k(1e-10)[0] < k
        assert rel2(y, spl.spsolve((sp.identity(n) - alpha * A).tocsc(), x)) < TOL
        assert mctx.matfun_scale() == 0.0
    mctx.set_matfun(lz.MATFUN_EXP_SCALED, 1.0)
    mctx.expv_host(None, k)
    theta_max = mctx.get_eigen()[0][-1]
    mctx.set_matfun(lz.MATFUN_RESOLVENT, 1.01 / theta_max)
    msg = raises_code(lz, -6, mctx.expv_host, None, k)
    assert "resolvent" in msg and "did not converge" not in msg
    raises_code(lz, -6, mctx.get_eigen)
    raises_code(lz, -6, mctx.estimate_change, k // 2)
    mctx.set_matfun(lz.MATFUN_RESOLVENT, 0.0)
    xr = np.random.default_rng(5).standard_normal(n)
    assert rel2(mctx.expv_host(xr, k), xr) < 1e-13


def test_convergence_estimate_per_function(lz, orc, golden, mctx):
    """lz_estimate_change / lz_choose_k follow the function: at t = 2 the estimate is the change between the oracle's answers at
    k' and k; more steps are needed as t grows; the shifted estimate is the unshifted one (and exists where that one fails)."""
    g = golden("c1_er_n10000_k20")
    ro, ci, n = g["row_offset"], g["col_idx"], int(g["n"])
    mctx.csr_upload(ro, ci)
    mctx.set_matfun(lz.MATFUN_EXP, 2.0)
    y20 = mctx.expv_host(None, 20)
    for kp in (8, 12, 16):
        ykp, _ = krylov_f(orc, ro, ci, kp, np.ones(n), lambda th: np.exp(2.0 * th))
        assert mctx.estimate_change(kp) == pytest.approx(rel2(ykp, y20), rel=1e-3, abs=1e-13), kp
    chosen = []
    for t in (0.5, 1.0, 2.0):                      # no new run: the estimate works on the kept tridiagonal
        mctx.set_matfun(lz.MATFUN_EXP, t)
        chosen.append(mctx.choose_k(1e-10)[0])
    assert chosen[0] <= chosen[1] <= chosen[2], chosen
    # Shifted and unshifted coefficients differ by e^{-ls} up to one rounding each, so the two estimates agree to 1e-12 relative
    # above the estimate's own rounding floor (~1e-16 * sqrt(k)).
    for t in (1.0, 2.0):
        mctx.set_matfun(lz.MATFUN_EXP, t)
        eu = [mctx.estimate_change(kp) for kp in range(4, 20)]
        ku = mctx.choose_k(1e-10)
        mctx.set_matfun(lz.MATFUN_EXP_SCALED, t)
        es = [mctx.estimate_change(kp) for kp in range(4, 20)]
        assert all(abs(a - b) <= 1e-12 * a + 1e-14 for a, b in zip(eu, es)), (t, eu, es)
        assert mctx.choose_k(1e-10)[0] == ku[0]
    ro, ci, lam, V, t = graph500_small(lz)
    mctx.csr_upload(ro, ci)
    mctx.set_start_vector(None)
    mctx.lanczos_run(30)
    mctx.set_matfun(lz.MATFUN_EXP, t)
    raises_code(lz, -6, mctx.estimate_change, 20)
    mctx.set_matfun(lz.MATFUN_EXP_SCALED, t)
    e = mctx.estimate_change(20)
    assert np.isfinite(e) and e < 1e-6


def test_one_basis_many_functions(lz, golden, mctx):
    """After one lz_lanczos_run each function is a coefficient solve + multOut: the same bits as a fresh pipeline under that
    setting, and no Lanczos step runs again."""
    g = golden("rmat_s12_k30")
    k, n = int(g["k"]), int(g["n"])
    funs = [(lz.MATFUN_EXP, 1.0), (lz.MATFUN_EXP, 0.5), (lz.MATFUN_EXP_SCALED, 3.0), (lz.MATFUN_RESOLVENT, 0.015),
            (lz.MATFUN_EXP, 2.0)]
    mctx.csr_upload(g["row_offset"], g["col_idx"])
    mctx.set_start_vector(None)
    mctx.lanczos_run(k)
    launches = [mctx.timings().kernel_launches]
    ys = []
    for kind, p in funs:
        mctx.set_matfun(kind, p)
        mctx.tridiag_expv()
        mctx.multout()
        ys.append(mctx.get_ans())
        launches.append(mctx.timings().kernel_launches)
    per_fun = np.diff(launches)
    assert np.all(per_fun == per_fun[0]) and per_fun[0] < 8, per_fun   # a coefficient solve and a multOut, never k steps
    for (kind, p), y in zip(funs, ys):
        mctx.set_matfun(kind, p)
        assert np.array_equal(mctx.expv_host(None, k), y), (kind, p)
        assert np.all(np.isfinite(y)) and y.shape == (n,)


@pytest.mark.parametrize("mode", ["f32", "reorth", "unlagged"])
def test_other_paths(lz, golden, monkeypatch, mode):
    """EXP_SCALED and RESOLVENT on the fp32 basis, with full reorthogonalisation and with the unlagged loop agree with the plain
    fp64 answer to the tolerances those modes are held to elsewhere."""
    g = golden("rmat_s14_k50")
    ro, ci, k = g["row_offset"], g["col_idx"], int(g["k"])
    funs = ((lz.MATFUN_EXP_SCALED, 4.0), (lz.MATFUN_RESOLVENT, 0.5 / 40.0))
    ref = {}
    with lz.Context(0) as c:
        c.csr_upload(ro, ci)
        for f in funs:
            c.set_matfun(*f)
            ref[f] = (c.expv_host(None, k), c.matfun_scale())
    if mode == "unlagged":
        monkeypatch.setenv("LZ_LAGGED_NORM", "0")
    tol = 1e-6 if mode == "f32" else TOL
    with lz.Context(0) as c:
        if mode == "f32":
            c.set_basis_precision(lz.BASIS_F32)
        c.csr_upload(ro, ci)
        for f in funs:
            c.set_matfun(*f)
            y = c.expv_host(None, k, lz.REORTH_FULL if mode == "reorth" else lz.REORTH_NONE)
            y0, ls0 = ref[f]
            assert rel2(y * np.exp(c.matfun_scale() - ls0), y0) < tol, (mode, f)


def test_validation(lz, orc, golden):
    g = golden("er_n2000_k20")
    ro, ci, k, n = g["row_offset"], g["col_idx"], int(g["k"]), int(g["n"])
    with lz.Context(0) as c:
        for kind, p in ((3, 1.0), (-1, 1.0), (lz.MATFUN_EXP, np.nan), (lz.MATFUN_EXP_SCALED, np.inf),
                        (lz.MATFUN_RESOLVENT, -np.inf)):
            raises_code(lz, -1, c.set_matfun, kind, p)
        raises_code(lz, -1, c.matfun_scale)
        c.csr_upload(ro, ci)
        c.set_matfun(lz.MATFUN_EXP, 0.5)
        c.set_start_vector(None)
        c.lanczos_run(k)
        raises_code(lz, -1, c.matfun_scale)                 # before lz_tridiag_expv
        c.tridiag_expv()
        c.multout()
        y = c.get_ans()
        ref, _ = krylov_f(orc, ro, ci, k, np.ones(n), lambda th: np.exp(0.5 * th))
        assert rel2(y, ref) < TOL                            # the setting survived lz_set_start_vector
        c.set_matfun(lz.MATFUN_EXP_SCALED, 0.5)              # drops coefficients and answer, keeps the run
        raises_code(lz, -1, c.get_ans)
        raises_code(lz, -1, c.top_k, 10)
        raises_code(lz, -1, c.matfun_scale)
        c.tridiag_expv()
        c.multout()
        assert rel2(c.get_ans() * np.exp(c.matfun_scale()), y) < 1e-13
        x = np.random.default_rng(2).standard_normal(n)
        c.set_start_vector(x)
        c.lanczos_run(k)
        c.tridiag_expv()
        c.multout()
        ref, th = krylov_f(orc, ro, ci, k, x, lambda th: np.exp(0.5 * (th - th.max())))
        assert rel2(c.get_ans(), ref) < TOL


def _final(lz):
    libdir = os.path.join(os.path.dirname(lz.lib_path), "..", "lib")
    subprocess.check_call(["make", "-s", "-C", libdir])
    return os.path.join(libdir, "final")


def test_cpp_driver_scaled_and_katz(lz, orc, tmp_path):
    """final --t T --scaled on an R-MAT whose e^{TA} overflows: exit 0, a finite answer, and the ranking the C ABI gives for the
    same setting; without --scaled the run fails. --katz runs too. With two or more GPUs, --gpus 2 gives the one-GPU answer."""
    final = _final(lz)
    k = 30
    with lz.Context(0) as c:
        c.graph_generate(lz.GraphSpec.rmat(14, 8, 1))
        c.set_matfun(lz.MATFUN_EXP_SCALED, 1.0)
        c.expv_host(None, k)
        t = 800.0 / float(c.get_eigen()[0][-1])
        c.set_matfun(lz.MATFUN_EXP_SCALED, t)
        c.expv_host(None, k)
        top = c.top_k(100)[0]
        ls = c.matfun_scale()
    base = [final, "--graph", "rmat", "--scale", "14", "-k", str(k), "--t", repr(t)]
    out1 = str(tmp_path / "one.txt")
    r = subprocess.run(base + ["--scaled", "--top", "100", "--write", out1], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0 and "result finite: yes" in r.stdout, r.stdout[-2000:] + r.stderr[-2000:]
    assert "log scale: " in r.stdout
    line = next(l for l in r.stdout.splitlines() if l.startswith("log scale: "))
    assert float(line.split()[2]) == pytest.approx(ls, rel=1e-15)
    assert "TOP 100 vertices by total communicability e^{tA} x" in r.stdout
    ranked = [int(l.split()[2]) for l in r.stdout.splitlines() if l.startswith("rank ")]
    assert ranked == list(top)
    r = subprocess.run(base, capture_output=True, text=True, timeout=300)
    assert r.returncode != 0
    assert subprocess.run(base[:-1] + ["1e3x"], capture_output=True, text=True, timeout=300).returncode == 2
    r = subprocess.run([final, "--graph", "rmat", "--scale", "14", "-k", str(k), "--katz", "0.01", "--top", "10"],
                       capture_output=True, text=True, timeout=300)
    assert r.returncode == 0 and "result finite: yes" in r.stdout and "Katz centrality" in r.stdout, r.stdout[-2000:]
    if lz.device_count() < 2:
        pytest.skip("the multi-GPU leg needs two GPUs")
    out2 = str(tmp_path / "two.txt")
    r = subprocess.run(base + ["--scaled", "--gpus", "2", "--write", out2], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and "result finite: yes" in r.stdout, r.stdout[-2000:] + r.stderr[-2000:]
    assert rel2(np.loadtxt(out2), np.loadtxt(out1)) < TOL
