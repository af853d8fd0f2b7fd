"""Per-step checks of the one-GPU Lanczos loop and of the coefficient solve.

Once Lanczos has converged, e^A·x hardly depends on the later steps: on rmat_s14_k50 (k = 50, plain, start = ones) a 1 %
error in alpha_49 moves e^A·x by 6e-18, in alpha_20 by 1e-15 and in beta_19 by 7e-12, all inside the 1e-9 that the parity
tests allow. So those tests cannot see a wrong coefficient or basis vector past the first few steps. This file checks every
step directly, with two kinds of reference:

* the step invariants (`step_invariants`) that floating-point Lanczos keeps at every step even after it has lost global
  orthogonality (Paige): the three-term relation A q_j = beta_{j-1} q_{j-1} + alpha_j q_j + beta_j q_{j+1}, alpha_j = q_j^T A q_j,
  unit norm and local orthogonality of neighbouring vectors. They hold for plain Lanczos at any k;
* with full reorthogonalisation, the same algorithm in extended precision (`lanczos_ld`): T and the basis of a CGS2 run are
  forward stable, so they must match it closely at every step.

Every tolerance is calibrated against the CPU oracle (oracle/lanczos_oracle.c, fp64, sequential sums) on the same graph, start
vector and k: the device may be at most FACTOR times worse than the oracle, plus a floor of a few eps (see `limits`).

The coefficient solve (k_tridiag_expv: QL eigen-solve + f(T) e_1) is checked against an extended-precision reference computed
from the device's own alpha and beta: Sturm bisection in long double for the eigenvalues, a 40-digit Taylor series for the
exponential and a 40-digit Thomas solve for the resolvent.

Tests marked gpu need a B200; the others check the checkers themselves and run anywhere.
"""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import scipy.sparse as sp
from scipy.linalg import eigh_tridiagonal

EPS = float(np.finfo(np.float64).eps)        # 2^-52
U32 = 2.0 ** -24                              # unit roundoff of fp32
LD = np.longdouble
FACTOR = 16                                   # device error <= FACTOR * oracle error + floor
GOLDEN = ["er_n257_k10_ragged", "er_n2000_k20", "rmat_s14_k50", "band_n4096_k40"]
GRAPHS = GOLDEN + ["crafted"]
PLAIN_K = 60                                  # plain runs far past the loss of global orthogonality
KEYS = ("resid", "alpha", "norm", "orth1", "orth2")


# ---- checkers (plain numpy) ----------------------------------------------------------------------------------------------
def adjacency(ro, ci, dtype=np.float64):
    n = len(ro) - 1
    return sp.csr_matrix((np.ones(len(ci), dtype), np.asarray(ci, np.int64), np.asarray(ro, np.int64)), shape=(n, n))


def norm_bound(ro):
    """||A||_2 <= sqrt(||A||_1 ||A||_inf) = max degree for a symmetric 0/1 matrix."""
    return max(1.0, float(np.diff(np.asarray(ro, np.int64)).max()))


def step_invariants(ro, ci, alpha, beta, rows):
    """Per-step invariants of a Lanczos run; rows[j] = q_j (k x n). Returns arrays indexed by step:

    resid[j]  = ||A q_j - beta_{j-1} q_{j-1} - alpha_j q_j - beta_j q_{j+1}|| / ||A||,  j <= k-2
    alpha[j]  = |alpha_j - q_j^T A q_j| / ||A||,                                         j <= k-1
    norm[j]   = | ||q_j|| - 1 |,                                                         j <= k-1
    orth1[j]  = |q_{j+1}^T q_j|,  orth2[j] = |q_{j+2}^T q_j|

    Only beta_0..beta_{k-2} and q_0..q_{k-1} exist, so column k-1 enters through alpha_{k-1} = q_{k-1}^T A q_{k-1} (and the
    relation at j = k-2): every number the API returns is pinned. Evaluated in long double; A is 0/1, so the sparse product adds
    no rounding of its own beyond the 64-bit-mantissa sums. ||A|| is bounded by the maximum degree."""
    A = adjacency(ro, ci, LD)
    nA = norm_bound(ro)
    Q = np.asarray(rows, LD)
    k = len(Q)
    a, b = np.asarray(alpha, LD), np.asarray(beta, LD)
    out = {key: [] for key in KEYS}
    for j in range(k):
        aq = A @ Q[j]
        out["alpha"].append(abs(a[j] - Q[j] @ aq) / nA)
        out["norm"].append(abs(np.sqrt(Q[j] @ Q[j]) - 1))
        if j + 1 < k:
            r = aq - a[j] * Q[j] - b[j] * Q[j + 1]
            if j:
                r -= b[j - 1] * Q[j - 1]
            out["resid"].append(np.sqrt(r @ r) / nA)
            out["orth1"].append(abs(Q[j + 1] @ Q[j]))
        if j + 2 < k:
            out["orth2"].append(abs(Q[j + 2] @ Q[j]))
    return {key: np.array(v, np.float64) for key, v in out.items()}


def limits(ref, floor=4 * EPS):
    """Tolerance per invariant from a reference run's invariants: FACTOR x its worst step, plus `floor`.

    FACTOR = 16 and floor = 4 eps: the device's tree reductions are no less accurate than the oracle's sequential sums, so a
    correct kernel sits at or below the oracle (measured on the CPU, oracle on the goldens: resid <= 5e-17, alpha <= 8e-15,
    norm <= 3e-14, orth1 <= 4e-14, orth2 <= 9e-14, plain and CGS2, k up to 60). The resulting limits stay below 1.5e-12, so an
    error of 1e-10 relative in any coefficient or basis entry fails (test_checker_rejects_late_step_errors)."""
    return {key: FACTOR * (float(v.max()) if v.size else 0.0) + floor for key, v in ref.items()}


def assert_invariants(inv, lim, what):
    for key in KEYS:
        v = inv[key]
        if v.size and not v.max() <= lim[key]:
            j = int(np.argmax(v))
            raise AssertionError(f"{what}: {key} = {v[j]:.3e} at step {j} > {lim[key]:.3e}")


def lanczos_ld(ro, ci, k, x):
    """Lanczos with full reorthogonalisation in long double: classical Gram-Schmidt twice every step, in the operation order of
    oracle/lanczos_oracle.c's CGS2 (three-term update first, then two projections against q_0..q_j). -> alpha, beta, Q (k x n)."""
    A = adjacency(ro, ci, LD)
    n = len(ro) - 1
    Q = np.zeros((k, n), LD)
    a, b = np.zeros(k, LD), np.zeros(max(k - 1, 0), LD)
    x = np.asarray(x, LD)
    Q[0] = x / np.sqrt(x @ x)
    for j in range(k):
        v = A @ Q[j]
        a[j] = v @ Q[j]
        v -= a[j] * Q[j]
        if j:
            v -= b[j - 1] * Q[j - 1]
        for _ in range(2):
            v -= (Q[:j + 1] @ v) @ Q[:j + 1]
        if j + 1 < k:
            b[j] = np.sqrt(v @ v)
            Q[j + 1] = v / b[j]
    return a, b, Q


def ld_distance(ro, alpha, beta, rows, ref):
    """(max |alpha - alpha_ld| / ||A||, max |beta - beta_ld| / ||A||, max_j ||q_j - q_j,ld||)."""
    a, b, Q = ref
    nA = norm_bound(ro)
    return (float(np.abs(np.asarray(alpha, LD) - a).max()) / nA,
            float(np.abs(np.asarray(beta, LD) - b).max()) / nA if len(b) else 0.0,
            float(np.sqrt(((np.asarray(rows, LD) - Q) ** 2).sum(axis=1)).max()))


def expv_from(alpha, beta, rows, x_norm):
    """e^A x = ||x|| Q e^T e_1 from a decomposition (fp64, scipy's tridiagonal eigensolver)."""
    w, Z = eigh_tridiagonal(alpha, beta)
    return x_norm * ((Z @ (np.exp(w) * Z[0])) @ rows)


# ---- inputs --------------------------------------------------------------------------------------------------------------
def crafted_csr(lz):
    """ER graph on 3001 vertices (not a multiple of 32) plus one hub joined to 1500 vertices (a warp-per-row item and a
    dense column) and five isolated vertices (empty rows, eigenvalue 0 with multiplicity)."""
    rng = np.random.default_rng(2024)
    n = 3001
    u, v = rng.integers(0, n - 6, 12000), rng.integers(0, n - 6, 12000)
    nbrs = rng.choice(np.arange(1, n - 6), 1500, replace=False)
    u = np.concatenate([u, np.zeros(1500, np.int64)])
    v = np.concatenate([v, nbrs])
    _, ro, ci = lz.csr_from_edges(n, u, v)
    return ro, ci


_GRAPHS = {}


def load_graph(name, lz, golden):
    """-> (row_offset, col_idx, k, x_random). The crafted graph uses k = 30."""
    if name not in _GRAPHS:
        if name == "crafted":
            ro, ci = crafted_csr(lz)
            _GRAPHS[name] = (ro, ci, 30, np.random.default_rng(5).standard_normal(len(ro) - 1))
        else:
            g = golden(name)
            _GRAPHS[name] = (g["row_offset"], g["col_idx"], int(g["k"]), g["x_random"])
    return _GRAPHS[name]


def runs_for(name, lz, golden):
    """The runs checked on each graph: plain at the golden k from ones (the reference's start), plain to PLAIN_K from a random
    start (global orthogonality long lost) and full reorthogonalisation at the golden k from the random start."""
    ro, ci, k, xr = load_graph(name, lz, golden)
    n = len(ro) - 1
    return [("plain", k, np.ones(n)), ("plain", PLAIN_K, xr), ("full", k, xr)]


_REF = {}


def oracle_reference(orc, name, lz, golden, mode, k, x, fp32=False):
    """Invariants of the CPU oracle's run (and, for full reorthogonalisation, its distance from lanczos_ld) on the same graph,
    start vector and k; fp32=True evaluates the oracle's rows rounded to fp32. Cached."""
    key = (name, mode, k, float(x[0]), fp32)
    if key not in _REF:
        ro, ci, _, _ = load_graph(name, lz, golden)
        a, b, Q = orc.lanczos(ro, ci, k, x, orc.FULL if mode == "full" else orc.PLAIN)
        rows = Q.T.astype(np.float32).astype(np.float64) if fp32 else Q.T
        r = {"inv": step_invariants(ro, ci, a, b, rows)}
        if mode == "full" and not fp32:
            ld = lanczos_ld(ro, ci, k, x)
            r["ld"] = ld
            r["ld_dist"] = ld_distance(ro, a, b, Q.T, ld)
        _REF[key] = r
    return _REF[key]


def read_run(c, k):
    a, b = c.get_tridiag()
    return a, b, np.stack([c.get_basis(j) for j in range(k)])


def check_run(orc, name, lz, golden, mode, k, x, alpha, beta, rows, what, fp32=False):
    """Step invariants against the oracle-calibrated limits; for fp64 CGS2 runs also the distance from lanczos_ld."""
    ro, ci, _, _ = load_graph(name, lz, golden)
    ref = oracle_reference(orc, name, lz, golden, mode, k, x, fp32)
    lim = limits(ref["inv"], floor=4 * U32 if fp32 else 4 * EPS)
    assert_invariants(step_invariants(ro, ci, alpha, beta, rows), lim, what)
    if mode == "full" and not fp32:
        d = ld_distance(ro, alpha, beta, rows, ref["ld"])
        for i, label in enumerate(("alpha", "beta", "basis row")):
            tol = FACTOR * ref["ld_dist"][i] + 4 * EPS
            assert d[i] <= tol, f"{what}: {label} differs from the extended-precision run by {d[i]:.3e} > {tol:.3e}"


# ---- CPU: the checkers themselves ----------------------------------------------------------------------------------------
def test_extended_reference_matches_oracle_cgs2(orc, golden):
    """lanczos_ld against the oracle's fp64 CGS2 on er_n2000_k20's graph with its random start. Measured on the CPU: alpha and
    beta differ by <= 5.0e-16 ||A|| (||A|| bounded by the max degree, 24) at k = 20 and at k = 200; basis entries by 2.2e-16
    (k = 20) and 3.2e-15 (k = 200), basis rows in 2-norm by 1.8e-15 and 2.6e-14. Asserted with a factor 2. lanczos_ld's own
    invariants at k = 200 reach 2.2e-17 (the three-term residual carries the long-double Gram-Schmidt corrections), asserted
    below 1e-16: ten times below the fp64 oracle's 1.1e-15."""
    g = golden("er_n2000_k20")
    ro, ci, x = g["row_offset"], g["col_idx"], g["x_random"]
    for k, entry in ((20, 4.4e-16), (200, 6.4e-15)):
        a, b, Q = orc.lanczos(ro, ci, k, x, orc.FULL)
        ref = lanczos_ld(ro, ci, k, x)
        da, db, drow = ld_distance(ro, a, b, Q.T, ref)
        assert da < 1e-15 and db < 1e-15, (k, da, db)
        assert float(np.abs(Q.T - ref[2]).max()) < entry, k
        assert drow < 100 * entry, (k, drow)
    inv = step_invariants(ro, ci, *[np.asarray(v, np.float64) for v in ref])
    assert max(float(v.max()) for v in inv.values()) < 1e-16, {key: float(v.max()) for key, v in inv.items()}


def test_checker_rejects_late_step_errors(orc, golden):
    """The blind spot and its closure, on the oracle's plain run on rmat_s14_k50 (k = 50, start = ones). Each perturbation of
    the last step by 1e-10 moves e^A x by less than 1e-12 relative, so no end-to-end test sees it; each is rejected by
    step_invariants with the limits calibrated on the unperturbed run, and so is a basis row left unnormalised."""
    g = golden("rmat_s14_k50")
    ro, ci, k, n = g["row_offset"], g["col_idx"], int(g["k"]), int(g["n"])
    a, b, Q = orc.lanczos(ro, ci, k, np.ones(n))
    rows = np.ascontiguousarray(Q.T)
    base = step_invariants(ro, ci, a, b, rows)
    lim = limits(base)
    assert_invariants(base, lim, "unperturbed")
    assert max(lim.values()) < 1.5e-12, lim
    y0 = expv_from(a, b, rows, np.sqrt(n))

    def perturbed(what):
        a2, b2, r2 = a.copy(), b.copy(), rows.copy()
        if what == "alpha":
            a2[k - 1] *= 1 + 1e-10
        elif what == "beta":
            b2[k - 2] *= 1 + 1e-10
        elif what == "entry":
            r2[k - 1, int(np.argmax(np.abs(r2[k - 1])))] += 1e-10
        else:   # u_{k-1} = beta_{k-2} q_{k-1}: the unnormalised vector the lagged loop stores
            r2[k - 1] *= b[k - 2]
        return a2, b2, r2

    for what in ("alpha", "beta", "entry", "unnormalised"):
        a2, b2, r2 = perturbed(what)
        if what != "unnormalised":
            y = expv_from(a2, b2, r2, np.sqrt(n))
            assert np.linalg.norm(y - y0) / np.linalg.norm(y0) < 1e-12, what
        with pytest.raises(AssertionError):
            assert_invariants(step_invariants(ro, ci, a2, b2, r2), lim, what)


# ---- GPU: every one-GPU loop path ----------------------------------------------------------------------------------------
# name -> (environment, SpMV variant). Context-creation knobs (LZ_LAGGED_NORM, LZ_SELL_GROUP) and ingest knobs (LZ_SELL_NARROW,
# LZ_SPMV_COLBLOCKS, LZ_ORDER) are set before the context and the upload; LZ_CUDA_GRAPH is read at every lz_lanczos_run.
CONFIGS = {
    "graph_replay": ({"LZ_CUDA_GRAPH": "1"}, "auto"),
    "launch_by_launch": ({"LZ_CUDA_GRAPH": "0"}, "auto"),
    "unlagged": ({"LZ_LAGGED_NORM": "0"}, "auto"),
    "csr_vector": ({}, "vector"),
    "csr_warp": ({}, "warp"),
    "quad_narrow_cols3_degree": ({"LZ_SELL_GROUP": "4", "LZ_SELL_NARROW": "1", "LZ_SPMV_COLBLOCKS": "3", "LZ_ORDER": "d"}, "auto"),
    "quad_narrow_cols3_natural": ({"LZ_SELL_GROUP": "4", "LZ_SELL_NARROW": "1", "LZ_SPMV_COLBLOCKS": "3", "LZ_ORDER": "n"}, "auto"),
}


def make_context(lz, monkeypatch, config):
    env, variant = CONFIGS[config]
    for key, val in env.items():
        monkeypatch.setenv(key, val)
    c = lz.Context(0)
    c.set_spmv_variant({"auto": lz.SPMV_AUTO, "vector": lz.SPMV_VECTOR, "warp": lz.SPMV_WARP}[variant])
    return c


@pytest.mark.gpu
@pytest.mark.parametrize("name", GRAPHS)
@pytest.mark.parametrize("config", list(CONFIGS))
def test_every_step_of_the_loop(lz, orc, golden, monkeypatch, config, name):
    """Every step of plain and reorthogonalised runs on every one-GPU loop variant: the step invariants on every column, and for
    CGS2 runs alpha, beta and every basis row against the extended-precision run (limits: see `limits` and `check_run`)."""
    ro, ci, _, _ = load_graph(name, lz, golden)
    with make_context(lz, monkeypatch, config) as c:
        c.csr_upload(ro, ci)
        for mode, k, x in runs_for(name, lz, golden):
            c.set_start_vector(x)
            c.lanczos_run(k, lz.REORTH_FULL if mode == "full" else lz.REORTH_NONE)
            a, b, rows = read_run(c, k)
            check_run(orc, name, lz, golden, mode, k, x, a, b, rows, f"{config}/{name}/{mode}/k={k}")


@pytest.mark.gpu
@pytest.mark.parametrize("name", GRAPHS)
def test_every_step_fp32_basis(lz, orc, golden, name):
    """LZ_BASIS_F32 stores the basis rows as floats; the recurrence of a plain run keeps fp64 copies of the last vectors, so its
    alpha and beta are bit-equal to the fp64 run's and every stored row is the fp32 rounding of the fp64 run's row. Read back, an
    entry may differ from the fp64 entry by 2^-24 relative (the rounding) plus 2^-51 (the read-out's division by ||u_j|| after a
    lagged run), plus 2^-140 absolute for subnormal floats. Reorthogonalised runs project against the fp32 rows, so they are held
    to the invariants at fp32 scale: the oracle's rows rounded to fp32, times FACTOR, plus 4 * 2^-24."""
    ro, ci, _, _ = load_graph(name, lz, golden)
    with lz.Context(0) as c:
        c.csr_upload(ro, ci)
        ref = []
        for mode, k, x in runs_for(name, lz, golden):
            c.set_start_vector(x)
            c.lanczos_run(k, lz.REORTH_FULL if mode == "full" else lz.REORTH_NONE)
            ref.append(read_run(c, k))
        c.set_basis_precision(lz.BASIS_F32)
        for (mode, k, x), (a64, b64, q64) in zip(runs_for(name, lz, golden), ref):
            c.set_start_vector(x)
            c.lanczos_run(k, lz.REORTH_FULL if mode == "full" else lz.REORTH_NONE)
            a, b, rows = read_run(c, k)
            what = f"fp32/{name}/{mode}/k={k}"
            if mode == "plain":
                assert np.array_equal(a, a64) and np.array_equal(b, b64), what
                dev = np.abs(rows - q64) - (U32 + 2.0 ** -51) * np.abs(q64) - 2.0 ** -140
                assert dev.max() <= 0, f"{what}: row {int(np.argmax(dev.max(axis=1)))} is not the fp32 rounding of the fp64 row"
            check_run(orc, name, lz, golden, mode, k, x, a, b, rows, what, fp32=True)


def _reorth_always_twice_dump(path):
    """Subprocess body of test_every_step_second_gram_schmidt_pass: LZ_REORTH_ALWAYS_TWICE is read once per process."""
    sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    import __graft_entry__ as g
    lz = g.load_package()
    gl = {name: np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", name + ".npz")) for name in GOLDEN}
    out, passes = {}, {}
    with lz.Context(0) as c:
        for name in GRAPHS:
            ro, ci, k, x = load_graph(name, lz, gl.__getitem__)
            c.csr_upload(ro, ci)
            c.set_start_vector(x)
            c.lanczos_run(k, lz.REORTH_FULL)
            passes[name] = int(c.timings().reorth_second_passes)
            a, b, rows = read_run(c, k)
            out[name + "/alpha"], out[name + "/beta"], out[name + "/rows"] = a, b, rows
    np.savez(path, **out)
    print(json.dumps(passes))


@pytest.mark.gpu
def test_every_step_second_gram_schmidt_pass(lz, orc, golden, tmp_path):
    """LZ_REORTH_ALWAYS_TWICE=1 forces the second Gram-Schmidt pass on every step (normally taken only when the first pass
    removed more than half of the vector). Same checks as the CGS2 runs of test_every_step_of_the_loop, in a subprocess."""
    path = str(tmp_path / "runs.npz")
    env = dict(os.environ, LZ_REORTH_ALWAYS_TWICE="1")
    r = subprocess.run([sys.executable, os.path.abspath(__file__), path], capture_output=True, text=True, env=env, timeout=600)
    assert r.returncode == 0, r.stderr[-3000:]
    passes = json.loads(r.stdout.strip().splitlines()[-1])
    d = np.load(path)
    for name in GRAPHS:
        _, _, k, x = load_graph(name, lz, golden)
        assert passes[name] == k - 1, (name, passes[name])
        check_run(orc, name, lz, golden, "full", k, x, d[name + "/alpha"], d[name + "/beta"], d[name + "/rows"],
                  f"always-twice/{name}")


# ---- GPU: CUDA-graph replay against launch by launch ---------------------------------------------------------------------
def _snapshot(c, k):
    a, b, rows = read_run(c, k)
    c.tridiag_expv()
    c.multout()
    return a, b, rows, c.get_ans()


@pytest.mark.gpu
@pytest.mark.parametrize("reorth", ["plain", "full"])
def test_graph_replay_bit_identical_to_launches(lz, orc, golden, monkeypatch, reorth):
    """The captured step loop replays the same kernels with the same grids as the launch-by-launch loop, and every reduction is
    deterministic, so alpha, beta, every basis row and e^A x are bit-identical. One long-lived context replays (LZ_CUDA_GRAPH=1,
    each state run twice: capture, then a cache hit) through a sequence of events that must each invalidate or keep the captured
    graph correctly: k 30 -> 20 -> 30, a new start vector, a switch of the basis precision (and back), and a re-upload of a
    different graph with the same n and nnz (a relabelled copy). Each state is compared with a fresh context run launch by
    launch. The replayed runs also pass the step invariants."""
    g = golden("rmat_s14_k50")
    ro, ci, n = g["row_offset"], g["col_idx"], int(g["n"])
    perm = np.random.default_rng(11).permutation(n)          # vertex i of the copy is vertex perm[i] of the original
    inv_perm = np.argsort(perm)
    deg = np.diff(ro.astype(np.int64))[perm]
    ro2 = np.concatenate([[0], np.cumsum(deg)]).astype(np.uint32)
    ci2 = np.concatenate([np.sort(inv_perm[ci[ro[p]:ro[p + 1]]]) for p in perm]).astype(np.uint32)
    graphs = {"original": (ro, ci), "relabelled": (ro2, ci2)}
    x1, x2 = np.ones(n), g["x_random"]
    mode = lz.REORTH_FULL if reorth == "full" else lz.REORTH_NONE
    states = [("original", "f64", x1, 30), ("original", "f64", x1, 20), ("original", "f64", x1, 30), ("original", "f64", x2, 30),
              ("original", "f32", x2, 30), ("original", "f64", x2, 30), ("relabelled", "f64", x2, 30)]

    def fresh(graph, prec, x, k):
        monkeypatch.setenv("LZ_CUDA_GRAPH", "0")
        with lz.Context(0) as f:
            if prec == "f32":
                f.set_basis_precision(lz.BASIS_F32)
            f.csr_upload(*graphs[graph])
            f.set_start_vector(x)
            f.lanczos_run(k, mode)
            return _snapshot(f, k)

    with lz.Context(0) as c:
        cur = (None, "f64")
        for graph, prec, x, k in states:
            if prec != cur[1]:
                c.set_basis_precision(lz.BASIS_F32 if prec == "f32" else lz.BASIS_F64)
            if graph != cur[0]:
                c.csr_upload(*graphs[graph])
            cur = (graph, prec)
            want = fresh(graph, prec, x, k)
            monkeypatch.setenv("LZ_CUDA_GRAPH", "1")
            for rep in range(2):
                c.set_start_vector(x)
                c.lanczos_run(k, mode)
                got = _snapshot(c, k)
                what = f"{reorth} {graph} {prec} k={k} x={'ones' if x is x1 else 'random'} replay {rep}"
                for label, u, v in zip(("alpha", "beta", "basis", "e^A x"), got, want):
                    assert np.array_equal(u, v), f"{what}: {label} differs from launch by launch"
            if graph == "original" and prec == "f64":
                gro, gci = graphs[graph]
                inv = step_invariants(gro, gci, got[0], got[1], got[2])
                assert max(float(inv[key].max()) for key in ("resid", "alpha")) < 1e-13, what


# ---- GPU: C3 at production size ------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_every_step_c3(lz):
    """R-MAT 2^24, k = 50, plain, start = ones: the only one-GPU configuration that runs launch by launch (n > 4M rows) with two
    column blocks by default. Step invariants over all 50 columns, three (four, for orth2) basis rows held at a time.

    Evaluated in fp64 with scipy (long double would take too long at 2.7e8 non-zeros), so the limits carry the test's own
    rounding: A q_j is a sequential sum of deg_i terms per row, off by at most gamma_{deg_i} (A |q_j|)_i (A |q_j| comes out of
    the same pass over A); dot products are numpy pairwise sums, off by at most 40 eps sum |x_i y_i|. On top of that the device
    may be off by 16 eps (relative to ||A||) in the residual and alpha and by 64 eps in the norm. Local orthogonality of plain
    Lanczos is only as good as eps ||A|| / beta (Paige), so orth1 and orth2 may be 64 eps theta_max / beta_j with theta_max the
    largest Ritz value (= ||A|| to many digits here). The oracle on the goldens reaches 0.2 eps, 35 eps and 130 eps (resid,
    alpha, norm) and 12 eps theta_max / beta_j (orth1, orth2) with sequential sums; the device's tree reductions are more
    accurate than that."""
    k = 50
    with lz.Context(0) as c:
        c.graph_generate(lz.GraphSpec.rmat(24, 8, 1))
        ro, ci = c.csr_download()
        n = len(ro) - 1
        c.set_start_vector(None)
        c.lanczos_run(k)
        alpha, beta = c.get_tridiag()
        A = sp.csr_matrix((np.ones(len(ci)), ci.astype(np.int32), ro.astype(np.int32)), shape=(n, n))
        deg = np.diff(ro.astype(np.int64)).astype(np.float64)
        gam = deg * EPS / 2 / (1 - deg * EPS / 2)
        nA = norm_bound(ro)
        theta_max = float(eigh_tridiagonal(alpha, beta, eigvals_only=True)[-1])
        win = {}

        def row(j):
            if j not in win:
                win[j] = c.get_basis(j)
            return win[j]

        def dot_err(x, y):
            return 40 * EPS * float(np.sum(np.abs(x * y)))

        worst = {key: 0.0 for key in KEYS}
        for j in range(k):
            for old in [i for i in win if i < j - 1]:
                del win[old]
            q = row(j)
            both = A @ np.stack([q, np.abs(q)], axis=1)
            aq, e = both[:, 0], gam * both[:, 1]
            qaq = float(np.sum(q * aq))
            tol_a = (float(np.sum(np.abs(q) * e)) + dot_err(q, aq)) / nA + 16 * EPS
            assert abs(alpha[j] - qaq) / nA <= tol_a, ("alpha", j, abs(alpha[j] - qaq) / nA, tol_a)
            qq = float(np.sum(q * q))
            assert abs(np.sqrt(qq) - 1) <= dot_err(q, q) + 64 * EPS, ("norm", j, abs(np.sqrt(qq) - 1))
            worst["alpha"] = max(worst["alpha"], abs(alpha[j] - qaq) / nA)
            worst["norm"] = max(worst["norm"], abs(np.sqrt(qq) - 1))
            if j + 1 < k:
                qn = row(j + 1)
                r = aq - alpha[j] * q - beta[j] * qn
                if j:
                    r -= beta[j - 1] * row(j - 1)
                # elementwise: 4 roundings of terms each <= |A q| + |alpha| |q| + 2 beta |q|, on top of the SpMV's own bound
                rn = float(np.sqrt(np.sum(r * r))) / nA
                tol_r = (float(np.linalg.norm(e)) + 4 * EPS * (nA + abs(alpha[j]) + 2 * max(beta[j], beta[j - 1] if j else 0))) / nA
                tol_r = tol_r * (1 + 1e-6) + 16 * EPS
                assert rn <= tol_r, ("resid", j, rn, tol_r)
                o1 = abs(float(np.sum(qn * q)))
                assert o1 <= dot_err(qn, q) + 64 * EPS * theta_max / beta[j], ("orth1", j, o1)
                worst["resid"], worst["orth1"] = max(worst["resid"], rn), max(worst["orth1"], o1)
            if j + 2 < k:
                o2 = abs(float(np.sum(row(j + 2) * q)))
                assert o2 <= dot_err(row(j + 2), q) + 64 * EPS * theta_max / min(beta[j], beta[j + 1]), ("orth2", j, o2)
                worst["orth2"] = max(worst["orth2"], o2)
        print("c3 worst", {key: f"{v:.2e}" for key, v in worst.items()})


# ---- GPU: the coefficient solve against an extended-precision reference --------------------------------------------------
def sturm_eigenvalues(alpha, beta):
    """All eigenvalues of the symmetric tridiagonal (alpha, beta), ascending, by bisection on the Sturm count in long double,
    vectorised over the k eigenvalues; converges to the long-double resolution of the Gershgorin interval."""
    a, b = np.asarray(alpha, LD), np.asarray(beta, LD)
    k = len(a)
    rad = np.zeros(k, LD)
    rad[:-1] += np.abs(b)
    rad[1:] += np.abs(b)
    lo = np.full(k, (a - rad).min() - 1, LD)
    hi = np.full(k, (a + rad).max() + 1, LD)
    idx = np.arange(k)
    b2 = b * b
    tiny = LD(np.finfo(LD).tiny)
    for _ in range(200):
        mid = (lo + hi) / 2
        cnt = np.zeros(k, np.int64)
        d = a[0] - mid
        for i in range(k):
            if i:
                d = a[i] - mid - b2[i - 1] / d
            d = np.where(d == 0, -tiny, d)
            cnt += d < 0
        below = cnt > idx            # more than idx eigenvalues lie below mid: eigenvalue idx is below mid
        hi = np.where(below, mid, hi)
        lo = np.where(below, lo, mid)
        if np.all(hi - lo <= 4 * np.finfo(LD).eps * np.maximum(np.abs(lo), np.abs(hi))):
            break
    return (lo + hi) / 2


def _mp_tridiag_matvec(a, b, v):
    k = len(a)
    out = [a[i] * v[i] for i in range(k)]
    for i in range(k - 1):
        out[i] += b[i] * v[i + 1]
        out[i + 1] += b[i] * v[i]
    return out


def mp_exp_e1(alpha, beta, t):
    """e^{tT} e_1 to 40 significant digits: e^{ts} * Taylor series of e^{t(T - sI)} e_1 on the vector, s the Gershgorin centre
    (so ||t(T - sI)|| <= t * radius and the series converges after ~e * t * radius terms). Working precision covers the
    cancellation of the series (up to e^{t radius}). Returns mpf values (no overflow)."""
    import mpmath as mp
    k = len(alpha)
    rad = np.zeros(k)
    rad[:-1] += np.abs(beta)
    rad[1:] += np.abs(beta)
    top, bot = float((np.asarray(alpha) + rad).max()), float((np.asarray(alpha) - rad).min())
    s, r = (top + bot) / 2, max((top - bot) / 2, 1e-300)
    with mp.workdps(45 + int(t * r / 2.3)):
        a = [mp.mpf(t) * (mp.mpf(float(x)) - mp.mpf(s)) for x in alpha]
        bb = [mp.mpf(t) * mp.mpf(float(x)) for x in beta]
        term = [mp.mpf(1)] + [mp.mpf(0)] * (k - 1)
        acc = list(term)
        m = 0
        while True:
            m += 1
            term = [x / m for x in _mp_tridiag_matvec(a, bb, term)]
            acc = [u + v for u, v in zip(acc, term)]
            if m > t * r and max(abs(x) for x in term) < mp.mpf(10) ** -45 * max(abs(x) for x in acc):
                break
        scale = mp.exp(mp.mpf(t) * mp.mpf(s))
        return [x * scale for x in acc]


def mp_resolvent_e1(alpha, beta, p):
    """(I - pT)^{-1} e_1 by a Thomas solve at 40 digits."""
    import mpmath as mp
    k = len(alpha)
    with mp.workdps(45):
        dg = [1 - mp.mpf(p) * mp.mpf(float(x)) for x in alpha]
        off = [-mp.mpf(p) * mp.mpf(float(x)) for x in beta]
        rhs = [mp.mpf(1)] + [mp.mpf(0)] * (k - 1)
        cp, dp = [mp.mpf(0)] * k, [mp.mpf(0)] * k
        for i in range(k):
            den = dg[i] - (off[i - 1] * cp[i - 1] if i else 0)
            cp[i] = off[i] / den if i + 1 < k else mp.mpf(0)
            dp[i] = (rhs[i] - (off[i - 1] * dp[i - 1] if i else 0)) / den
        xs = [mp.mpf(0)] * k
        for i in range(k - 1, -1, -1):
            xs[i] = dp[i] - (cp[i] * xs[i + 1] if i + 1 < k else 0)
        return xs


_TRIDIAG = {}


@pytest.mark.gpu
@pytest.mark.parametrize("k", [1, 2, 151, 152, 256, 257, 1024])
@pytest.mark.parametrize("reorth", ["plain", "full"])
def test_coefficient_solve_extended_precision(lz, reorth, k):
    """k_tridiag_expv on the device's own alpha, beta (er(3000, 9000, 21), start = ones) against an extended-precision
    reference: eigenvalues within 1e-13 ||T|| of Sturm bisection; the coefficient vector ||x|| f(T) e_1 for EXP (t = 1),
    EXP_SCALED (t = 1, compared as c e^ls) and RESOLVENT (p = 0.9 / theta_max) within 10x the error of the same quantity
    computed in fp64 from scipy's eigh_tridiagonal, plus 1e-15 ||c||. k <= 151 keeps the eigenvectors in shared memory and 152
    does not, 256 is the block size, 1024 the solver's limit. The plain run to k = 1024 carries clusters of ghost Ritz values,
    the hardest case for QL."""
    import mpmath as mp
    n, ro, ci = lz.generate_host(lz.GraphSpec.er(3000, 9000, 21))
    with lz.Context(0) as c:
        c.csr_upload(ro, ci)
        c.set_start_vector(None)
        c.lanczos_run(k, lz.REORTH_FULL if reorth == "full" else lz.REORTH_NONE)
        alpha, beta = c.get_tridiag()
        xn = np.sqrt(n)
        w_ref = sturm_eigenvalues(alpha, beta)
        tnorm = float(np.abs(w_ref).max())
        c.tridiag_expv()
        w, _, _ = c.get_eigen()
        err_w = float(np.abs(np.asarray(w, LD) - w_ref).max())
        assert err_w <= 1e-13 * tnorm, (err_w, tnorm)
        w64, Z64 = eigh_tridiagonal(alpha, beta) if k > 1 else (alpha.copy(), np.ones((1, 1)))
        theta_max = float(w_ref[-1])
        funs = [("exp", lz.MATFUN_EXP, 1.0), ("exp_scaled", lz.MATFUN_EXP_SCALED, 1.0), ("resolvent", lz.MATFUN_RESOLVENT, 0.9 / theta_max)]
        exp_ref = mp_exp_e1(alpha, beta, 1.0)
        for label, kind, p in funs:
            c.set_matfun(kind, p)
            c.tridiag_expv()
            _, _, coef = c.get_eigen()
            if kind == lz.MATFUN_RESOLVENT:
                ref = mp_resolvent_e1(alpha, beta, p)
                f64 = 1.0 / (1.0 - p * w64)
                scale = mp.mpf(1)
            else:
                ref = exp_ref
                f64 = np.exp(p * w64)
                scale = mp.exp(mp.mpf(c.matfun_scale()))
            ref_c = [xn * x for x in ref]                               # ||x|| f(T) e_1, unscaled
            c64 = xn * (Z64 @ (f64 * Z64[0]))
            refn = float(mp.sqrt(mp.fsum(x * x for x in ref_c)))
            dev = float(mp.sqrt(mp.fsum((mp.mpf(float(u)) * scale - x) ** 2 for u, x in zip(coef, ref_c))))
            e64 = float(mp.sqrt(mp.fsum((mp.mpf(float(u)) - x) ** 2 for u, x in zip(c64, ref_c))))
            assert dev <= 10 * e64 + 1e-15 * refn, (label, k, dev / refn, e64 / refn)


if __name__ == "__main__":
    _reorth_always_twice_dump(sys.argv[1])
