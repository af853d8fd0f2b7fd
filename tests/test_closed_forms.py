"""The one-GPU path against graphs whose spectra are known in closed form.

Every other check of the device takes its truth from another fp64 computation (the reference, the C oracle, a dense or sparse
eigensolver). Here the truth is exact: cycles, paths, circulants, complete and complete bipartite graphs, stars, hypercubes, tori,
grids and disjoint unions have eigenvalues and eigenvectors in closed form, evaluated with mpmath at 50 digits or in long double.
Each graph also comes randomly relabelled (A' = P A P^T: same spectrum, permuted eigenvectors), which destroys locality, so the
same exact answer exercises the degree order, several column blocks and scattered gathers.

With x = sum_i c_i v_i over s eigenvectors of distinct eigenvalues, f(A) x = sum_i c_i f(lambda_i) v_i exactly, and Lanczos is
exact at k = s; at k = s + 20 it runs 20 steps of rounding noise past the near-breakdown. The modes always include lambda_max and
lambda_min, so the noise cannot be amplified by a larger f(lambda) outside the modes.

Checks (the GPU ones are marked gpu; the others test the checkers and the references and run anywhere):
  (a) SpMV: |y^_i - y_i| <= gamma_{d_i} sum_j |x_j| per row with x spanning 2^+-40, and bit-exact on integer x, for every kernel.
  (b) f(A) x against the exact answer on every one-GPU loop path, within FACTOR x the fp64 oracle's error plus 4 eps times the
      condition number of f on the spectrum (`floor_f`; test_krylov_steps.py uses a flat 4 eps).
  (c) Ritz intervals and the spectral-radius bracket with zero slack, compared in mpmath with the exact spectrum.
  (d) eigenvector centrality within the sin-theta bound of the exact Perron vector.
  (e) Katz with alpha = 0.9 / hi: alpha lambda_max < 1 exactly, and the exact resolvent.
  (f) lz_top_k where the exact answer's gaps exceed the error bound.
  (g) lz_choose_k when x lies in an s-dimensional invariant subspace.
  (h) f(A)(2^p x) == 2^p f(A) x bit for bit.
"""
import functools
from dataclasses import dataclass, field

import mpmath as mp
import numpy as np
import pytest
import scipy.sparse as sp
import scipy.sparse.linalg as spl

mp.mp.dps = 50
LD = np.longdouble
EPS = float(np.finfo(np.float64).eps)        # 2^-52
U = EPS / 2                                   # unit roundoff of fp64
U_LD = float(np.finfo(LD).eps) / 2            # unit roundoff of the long double reference (2^-64 on x86-64)
FACTOR = 16                                   # device error <= FACTOR * oracle error + floor_f, as in test_krylov_steps.py


# ---- graphs -------------------------------------------------------------------------------------------------------------
@dataclass
class Graph:
    """Symmetric simple graph in CSR (columns ascending) with its exact spectrum.

    spectrum: the distinct eigenvalues as 50-digit mpmath numbers, ascending (None where too many to list).
    modes:    [(lambda, vector())] eigenvectors with distinct eigenvalues, lambda_max first and lambda_min second; vector() returns
              the unit eigenvector in long double. A repeated eigenvalue appears once (any vector of its eigenspace).
    perron:   unit Perron vector (long double) of a connected graph, and gap = lambda_max - next eigenvalue."""
    name: str
    n: int
    ro: np.ndarray
    ci: np.ndarray
    lmax: object
    lmin: object
    spectrum: list
    modes: list
    perron: object = None
    gap: object = None
    ones: object = None            # f -> exact f(A) 1 in long double (f maps an mpmath eigenvalue to an mpmath value)
    regular: bool = False
    extra: dict = field(default_factory=dict)


def mpld(v):
    """mpmath number -> long double (decimal string at 50 digits)."""
    return LD(mp.nstr(v, 40))


PI = mpld(mp.pi)


def unit(v):
    v = np.asarray(v, LD)
    return v / np.sqrt(v @ v)


def csr_from_edges(n, u, v):
    """Undirected edge list -> symmetric simple CSR, columns ascending."""
    u, v = np.asarray(u, np.int64), np.asarray(v, np.int64)
    keep = u != v
    r, c = np.concatenate([u[keep], v[keep]]), np.concatenate([v[keep], u[keep]])
    key = np.unique(r * n + c)
    r, c = key // n, key % n
    ro = np.zeros(n + 1, np.int64)
    np.cumsum(np.bincount(r, minlength=n), out=ro[1:])
    return ro.astype(np.uint32), c.astype(np.uint32)


def csr_from_neighbours(nb):
    """(n, d) neighbour table of a d-regular simple graph -> CSR."""
    nb = np.sort(np.asarray(nb, np.uint32), axis=1)
    n, d = nb.shape
    return (np.arange(n + 1, dtype=np.uint64) * d).astype(np.uint32), nb.reshape(-1)


def distinct(vals):
    vals = sorted(vals)
    out = [vals[0]]
    for v in vals[1:]:
        if v - out[-1] > mp.mpf(10) ** -40:
            out.append(v)
    return out


def circulant(n, offsets, name=None):
    """C_n(s_1..s_r): i ~ i +- s. Eigenvalues sum_s 2 cos(2 pi j s / n), eigenvectors cos(2 pi j i / n)."""
    i = np.arange(n)
    nb = np.concatenate([(i[:, None] + np.array(offsets)[None]) % n, (i[:, None] - np.array(offsets)[None]) % n], axis=1)
    ro, ci = csr_from_neighbours(nb)
    lam = {j: sum(2 * mp.cos(2 * mp.pi * j * s / n) for s in offsets) for j in range(n // 2 + 1)}
    spec = distinct(lam.values())
    jmin = min(lam, key=lambda j: lam[j])
    jmid = next(j for j in range(1, n // 2 + 1) if abs(lam[j] - lam[0]) > 1e-30 and abs(lam[j] - lam[jmin]) > 1e-30) \
        if len(spec) > 2 else None

    def vec(j):
        return lambda: unit(np.cos(2 * PI * LD(j) * np.arange(n, dtype=LD) / n))
    modes = [(lam[0], vec(0)), (lam[jmin], vec(jmin))] + ([(lam[jmid], vec(jmid))] if jmid is not None else [])
    second = spec[-2]
    return Graph(name or f"C{n}({','.join(map(str, offsets))})", n, ro, ci, spec[-1], spec[0], spec, modes,
                 perron=unit(np.ones(n, LD)), gap=spec[-1] - second, regular=True)


def cycle(n):
    return circulant(n, [1], f"cycle{n}")


def sines(a):
    """Unit eigenvectors of the path P_a as rows: S[j-1, i] ~ sin(pi j (i+1) / (a+1)), eigenvalue 2 cos(pi j / (a+1))."""
    j = np.arange(1, a + 1, dtype=LD)[:, None]
    i = np.arange(1, a + 1, dtype=LD)[None, :]
    return np.sin(PI * j * i / (a + 1)) * np.sqrt(LD(2) / (a + 1))


def path_eig(a):
    return [2 * mp.cos(mp.pi * j / (a + 1)) for j in range(1, a + 1)]


def grid(a, b):
    """P_a x P_b, vertex r * b + c. Eigenvalues mu_i + nu_j, eigenvectors outer products of path sines; degrees 2, 3 and 4.
    f(A) 1 from the sine transform of ones along each side."""
    r, c = np.divmod(np.arange(a * b), b)
    u = np.concatenate([np.flatnonzero(r + 1 < a), np.flatnonzero(c + 1 < b)])
    v = np.concatenate([np.flatnonzero(r + 1 < a) + b, np.flatnonzero(c + 1 < b) + 1])
    ro, ci = csr_from_edges(a * b, u, v)
    mu, nu = path_eig(a), path_eig(b)
    Sa, Sb = sines(a), sines(b)
    spec = distinct([x + y for x in mu for y in nu]) if a * b <= 4096 else None
    pairs = {(0, 0): mu[0] + nu[0], (a - 1, b - 1): mu[-1] + nu[-1]}
    for p in ((1, 0), (0, 1), (1, 1), (2, 0)):
        if p[0] < a and p[1] < b and all(abs(mu[p[0]] + nu[p[1]] - v) > 1e-30 for v in pairs.values()):
            pairs[p] = mu[p[0]] + nu[p[1]]
            break

    def vec(i, j):
        return lambda: np.outer(Sa[i], Sb[j]).reshape(-1)
    modes = [(lam, vec(*p)) for p, lam in pairs.items()]
    second = max(mu[0] + nu[1] if b > 1 else -mp.inf, mu[1] + nu[0] if a > 1 else -mp.inf)
    wa, wb = Sa @ np.ones(a, LD), Sb @ np.ones(b, LD)

    def ones(f):
        F = np.array([[mpld(f(x + y)) for y in nu] for x in mu], LD)
        return (Sa.T @ (wa[:, None] * F * wb[None, :]) @ Sb).reshape(-1)
    return Graph(f"grid{a}x{b}", a * b, ro, ci, mu[0] + nu[0], mu[-1] + nu[-1], spec, modes, perron=vec(0, 0)(),
                 gap=mu[0] + nu[0] - second, ones=ones, extra={"sines": (Sa, Sb, mu, nu)})


def torus(a, b):
    """C_a x C_b (a, b even), vertex r * b + c: eigenvalues 2 cos(2 pi i / a) + 2 cos(2 pi j / b), eigenvectors outer products."""
    r, c = np.divmod(np.arange(a * b, dtype=np.int64), b)
    nb = np.stack([((r + 1) % a) * b + c, ((r - 1) % a) * b + c, r * b + (c + 1) % b, r * b + (c - 1) % b], axis=1)
    ro, ci = csr_from_neighbours(nb)

    def vec(i, j):
        return lambda: unit(np.outer(np.cos(2 * PI * LD(i) * np.arange(a, dtype=LD) / a),
                                     np.cos(2 * PI * LD(j) * np.arange(b, dtype=LD) / b)).reshape(-1))
    lam = lambda i, j: 2 * mp.cos(2 * mp.pi * i / a) + 2 * mp.cos(2 * mp.pi * j / b)
    modes = [(lam(0, 0), vec(0, 0)), (lam(a // 2, b // 2), vec(a // 2, b // 2)), (lam(1, 0), vec(1, 0))]
    return Graph(f"torus{a}x{b}", a * b, ro, ci, mp.mpf(4), mp.mpf(-4), None, modes, perron=vec(0, 0)(), gap=4 - lam(1, 0)
                 if a <= b else 4 - lam(0, 1), regular=True)


def complete(n):
    """K_n: n - 1 (ones), -1 (multiplicity n - 1)."""
    i = np.arange(n)
    nb = (i[:, None] + np.arange(1, n)[None]) % n
    ro, ci = csr_from_neighbours(nb) if n > 1 else (np.zeros(2, np.uint32), np.zeros(0, np.uint32))
    e = np.zeros(n, LD)
    e[0], e[1] = 1, -1
    modes = [(mp.mpf(n - 1), lambda: unit(np.ones(n, LD))), (mp.mpf(-1), lambda: unit(e))]
    return Graph(f"K{n}", n, ro, ci, mp.mpf(n - 1), mp.mpf(-1), [mp.mpf(-1), mp.mpf(n - 1)], modes, perron=unit(np.ones(n, LD)),
                 gap=mp.mpf(n), regular=True)


def bipartite(a, b):
    """K_{a,b} (vertices 0..a-1 | a..a+b-1): +-sqrt(ab) with v = (1/sqrt(a) on one side, +-1/sqrt(b) on the other) / sqrt(2), and 0.
    Ones = ((sqrt a + sqrt b) v_+ + (sqrt a - sqrt b) v_-) / sqrt 2. The star is K_{1,b}."""
    n = a + b
    uu, vv = np.meshgrid(np.arange(a), np.arange(a, n), indexing="ij")
    ro, ci = csr_from_edges(n, uu.reshape(-1), vv.reshape(-1))
    s = mp.sqrt(a * b)

    def vpm(sign):
        v = np.empty(n, LD)
        v[:a] = 1 / np.sqrt(LD(a))
        v[a:] = sign / np.sqrt(LD(b))
        return v / np.sqrt(LD(2))
    modes = [(s, lambda: vpm(1)), (-s, lambda: vpm(-1))]
    if max(a, b) > 1:
        e = np.zeros(n, LD)
        e[[a, a + 1] if b > 1 else [0, 1]] = (1, -1)
        modes.append((mp.mpf(0), lambda: unit(e)))
    cp, cm = (np.sqrt(LD(a)) + np.sqrt(LD(b))) / np.sqrt(LD(2)), (np.sqrt(LD(a)) - np.sqrt(LD(b))) / np.sqrt(LD(2))

    def ones(f):
        return cp * mpld(f(s)) * vpm(1) + cm * mpld(f(-s)) * vpm(-1)
    spec = [-s, mp.mpf(0), s] if n > 2 else [-s, s]
    return Graph(f"K{a},{b}" if a > 1 else f"star{b}", n, ro, ci, s, -s, spec, modes, perron=vpm(1), gap=s if n > 2 else 2 * s,
                 ones=ones)


def star(b):
    return bipartite(1, b)


def hypercube(d):
    """Q_d: d - 2w (w = 0..d), Walsh vectors (-1)^popcount(i & S)."""
    n = 1 << d
    i = np.arange(n, dtype=np.int64)
    ro, ci = csr_from_neighbours(i[:, None] ^ (1 << np.arange(d))[None])

    def walsh(S):
        return lambda: np.where(np.bitwise_count(i & S) % 2 == 0, LD(1), LD(-1)) / np.sqrt(LD(n))
    modes = [(mp.mpf(d), walsh(0)), (mp.mpf(-d), walsh(n - 1))] + ([(mp.mpf(d - 2), walsh(1))] if d > 1 else [])
    return Graph(f"Q{d}", n, ro, ci, mp.mpf(d), mp.mpf(-d), [mp.mpf(d - 2 * w) for w in range(d, -1, -1)], modes,
                 perron=walsh(0)(), gap=mp.mpf(2), regular=True)


def union(parts, name):
    """Disjoint union (block diagonal). parts: list of Graph; the modes are those of the parts, padded with zeros, merged where
    their eigenvalues coincide (any combination of the copies is an eigenvector)."""
    offs = np.cumsum([0] + [p.n for p in parts])
    n = int(offs[-1])
    ro = np.concatenate([[0]] + [p.ro[1:].astype(np.int64) + int(np.sum([q.ro[-1] for q in parts[:k]], dtype=np.int64))
                                 for k, p in enumerate(parts)]).astype(np.uint32)
    ci = np.concatenate([p.ci.astype(np.int64) + offs[k] for k, p in enumerate(parts)]).astype(np.uint32)
    spec = distinct([v for p in parts for v in p.spectrum])
    groups = {}
    for k, p in enumerate(parts):
        for lam, fn in p.modes:
            key = mp.nstr(lam, 30)
            groups.setdefault(key, (lam, []))[1].append((k, fn))
    rng = np.random.default_rng(5)

    def combo(members):
        w = [LD(rng.uniform(0.5, 1.5)) for _ in members]       # drawn once: every call returns the same vector

        def f():
            v = np.zeros(n, LD)
            for (k, fn), wk in zip(members, w):
                v[offs[k]:offs[k + 1]] = fn() * wk
            return unit(v)
        return f
    modes = sorted(((lam, combo(m)) for lam, m in groups.values()), key=lambda t: -t[0])
    modes = [modes[0], modes[-1]] + modes[1:-1][:1]
    return Graph(name, n, ro, ci, spec[-1], spec[0], spec, modes)


def isolated(n):
    e = np.zeros(n, LD)
    e[0] = 1
    return Graph(f"isolated{n}", n, np.zeros(n + 1, np.uint32), np.zeros(0, np.uint32), mp.mpf(0), mp.mpf(0), [mp.mpf(0)],
                 [(mp.mpf(0), lambda: e.copy())])


def path(a):
    S = sines(a)
    lam = path_eig(a)
    ro, ci = csr_from_edges(a, np.arange(a - 1), np.arange(1, a))
    return Graph(f"path{a}", a, ro, ci, lam[0], lam[-1], lam[::-1], [(lam[0], lambda: S[0]), (lam[-1], lambda: S[-1]),
                                                                      (lam[1], lambda: S[1])], perron=S[0], gap=lam[0] - lam[1])


def relabel(g, seed=1):
    """A' = P A P^T with a random permutation: new id of vertex i is perm[i]; eigenvectors move with it."""
    n = g.n
    perm = np.random.default_rng(seed).permutation(n)
    deg = np.diff(g.ro.astype(np.int64))
    if g.regular and len(g.ci) == n * int(deg[0]):
        nb = perm[g.ci.astype(np.int64).reshape(n, int(deg[0]))]
        nbn = np.empty_like(nb)
        nbn[perm] = nb
        ro, ci = csr_from_neighbours(nbn)
    else:
        rows = np.repeat(np.arange(n), deg)
        ro, ci = csr_from_edges(n, perm[rows], perm[g.ci.astype(np.int64)])

    def move(fn):
        def f():
            v = np.empty(n, LD)
            v[perm] = fn()
            return v
        return f
    out = Graph(g.name + "_relabelled", n, ro, ci, g.lmax, g.lmin, g.spectrum, [(lam, move(fn)) for lam, fn in g.modes],
                perron=None if g.perron is None else move(lambda: g.perron)(), gap=g.gap, regular=g.regular)
    if g.ones is not None:
        out.ones = lambda f: move(lambda: g.ones(f))()
    return out


BUILDERS = {
    "cycle1001": lambda: cycle(1001),
    "circ500_w4": lambda: circulant(500, [1, 2]),
    "circ400_w8_r": lambda: relabel(circulant(400, [1, 2, 3, 4])),
    "circ1000_w130_r": lambda: relabel(circulant(1000, list(range(1, 66)))),
    "circ600_w64_r": lambda: relabel(circulant(600, list(range(1, 33)))),
    "circ600_w128_r": lambda: relabel(circulant(600, list(range(1, 65)))),
    "K131_r": lambda: relabel(complete(131)),
    "K129": lambda: complete(129),
    "star5000_r": lambda: relabel(star(5000)),
    "K30,50": lambda: bipartite(30, 50),
    "Q10_r": lambda: relabel(hypercube(10)),
    "grid30x50_r": lambda: relabel(grid(30, 50)),
    "grid30x50": lambda: grid(30, 50),
    "torus64x64_r": lambda: relabel(torus(64, 64)),
    "path300": lambda: path(300),
    "grid8x13_r": lambda: relabel(grid(8, 13)),
    "union": lambda: union([complete(20), complete(20), isolated(5), path(7)], "2xK20+5+P7"),
    "union_mixed_r": lambda: relabel(union([star(300), grid(10, 12), cycle(9), isolated(3)], "star300+grid10x12+C9+3")),
}


@functools.lru_cache(maxsize=None)
def G(name):
    return BUILDERS[name]()


def mode_vector(g, coeffs):
    """x = sum_i c_i v_i over the graph's modes (fp64) and the modes as (lambda, v) in long double."""
    vs = [(lam, fn()) for lam, fn in g.modes[:len(coeffs)]]
    x = sum(LD(c) * v for c, (_, v) in zip(coeffs, vs)).astype(np.float64)
    return x, vs


def exact_f(vs, x, fn):
    """f(A) x for x in the span of the unit, mutually orthogonal vs: sum_i (v_i^T x) f(lambda_i) v_i in long double (the
    coefficient of the fp64 x, not of the coefficients it was built from)."""
    xl = np.asarray(x, LD)
    return sum((v @ xl) * mpld(fn(lam)) * v for lam, v in vs)


# ---- checkers (plain numpy / mpmath) ----------------------------------------------------------------------------------------
def gamma(d, u=U):
    d = np.asarray(d, np.float64)
    return d * u / (1 - d * u)


def spmv_violations(ro, ci, x, y_dev):
    """Rows where |y^_i - (A x)_i| > gamma_{d_i} sum_j |x_j|; the long double reference carries its own gamma^{LD}_{d_i}."""
    n = len(ro) - 1
    A = sp.csr_matrix((np.ones(len(ci), LD), np.asarray(ci, np.int64), np.asarray(ro, np.int64)), shape=(n, n))
    xl = np.asarray(x, LD)
    ref, mag = A @ xl, A @ np.abs(xl)
    d = np.diff(np.asarray(ro, np.int64))
    bound = (gamma(d).astype(LD) + gamma(d, U_LD).astype(LD)) * mag * (1 + LD(2) ** -60)
    return np.flatnonzero(np.abs(np.asarray(y_dev, LD) - ref) > bound)


def contains_eigenvalue(rho, r, spectrum):
    """[rho - r, rho + r] computed exactly from the two doubles contains one of the exact eigenvalues (no slack)."""
    lo, hi = mp.mpf(rho) - mp.mpf(r), mp.mpf(rho) + mp.mpf(r)
    return any(lo <= lam <= hi for lam in spectrum)


def rel_err(y, ref):
    y, ref = np.asarray(y, LD), np.asarray(ref, LD)
    return float(np.sqrt(((y - ref) @ (y - ref)) / (ref @ ref)))


FUNCS = [("exp", -1.0), ("exp", 0.5), ("exp", 1.0), ("exp", 2.0), ("scaled", 1.0), ("scaled", -1.0),
         ("resolvent", -0.5), ("resolvent", 0.5), ("resolvent", 0.99)]


def fparam(kind, p, lmax):
    return p / float(lmax) if kind == "resolvent" else p


def mpf_of(kind, t, ls=0.0):
    """f as a function of an mpmath eigenvalue; EXP_SCALED leaves out e^ls (ls as the device returned it)."""
    if kind == "resolvent":
        return lambda lam: 1 / (1 - mp.mpf(t) * lam)
    return lambda lam: mp.exp(mp.mpf(t) * lam - mp.mpf(ls))


def floor_f(kind, t, g):
    """4 eps times the condition number of f on the spectrum: a perturbation of A by eps ||A|| (what any fp64 Ritz value carries)
    moves f(A) x by |t| eps ||A|| relative for e^{tA}, and by |alpha| eps ||A|| / min |1 - alpha lambda| for the resolvent. Where the
    oracle's Ritz values happen to be exact its error alone sits below that: a reorthogonalised run on C_1000(1..65) at k = 3
    reaches 4.7e-14 under EXP_SCALED t = -1, above 16x the oracle plus the flat 4 eps of test_krylov_steps.py (whose invariants
    are not multiplied by t). Elsewhere the oracle's own error is 1-120x this floor, so 16x the oracle dominates. At most
    4 eps (1 + 260), for EXP t = 2 on K_131."""
    lmax = float(g.lmax)
    if kind == "resolvent":
        cond = abs(t) * lmax / min(1 - t * lmax, 1 + t * lmax)
    else:
        cond = abs(t) * lmax
    return 4 * EPS * (1 + cond)


def oracle_f(a, b, Q, xnorm, kind, t):
    """||x|| Q f(T) e_1 in fp64 from a Lanczos run (as krylov_f in test_matfun.py), with EXP_SCALED's shift max t theta."""
    th, Z = np.linalg.eigh(np.diag(a) + np.diag(b, 1) + np.diag(b, -1))
    if kind == "resolvent":
        fv = 1 / (1 - t * th)
    else:
        fv = np.exp(t * th - (np.max(t * th) if kind == "scaled" else 0.0))
    return xnorm * (Q @ (Z @ (fv * Z[0])))


# ---- CPU self-tests -----------------------------------------------------------------------------------------------------
SMALL = ["cycle1001", "circ500_w4", "K129", "K30,50", "Q10_r", "grid30x50_r", "path300", "union", "union_mixed_r"]


@pytest.mark.parametrize("name", SMALL + ["star5000_r", "circ600_w128_r"])
def test_builders_spectra(name):
    """CSR is symmetric, simple, columns ascending; the listed spectrum is eigvalsh's; every mode is a unit eigenvector."""
    g = G(name)
    n = g.n
    A = sp.csr_matrix((np.ones(len(g.ci)), g.ci.astype(np.int64), g.ro.astype(np.int64)), shape=(n, n))
    assert (A != A.T).nnz == 0 and A.diagonal().sum() == 0 and A.max() == 1
    assert all(np.all(np.diff(g.ci[g.ro[i]:g.ro[i + 1]].astype(np.int64)) > 0) for i in range(n))
    lam = np.linalg.eigvalsh(A.toarray()) if n <= 2100 else None
    if lam is not None and g.spectrum is not None:
        spec = np.array([float(v) for v in g.spectrum])
        assert np.abs(lam[:, None] - spec[None]).min(axis=1).max() < 1e-9          # every eigenvalue is listed ...
        assert np.abs(spec[:, None] - lam[None]).min(axis=1).max() < 1e-9          # ... and every listed value occurs
    assert float(g.lmax) == pytest.approx(float(max(g.spectrum)), abs=1e-12)
    Al = sp.csr_matrix((np.ones(len(g.ci), LD), g.ci.astype(np.int64), g.ro.astype(np.int64)), shape=(n, n))
    tol = 1e-15 + 1e-17 * np.diff(g.ro.astype(np.int64)).max()          # long double row sums of up to max-degree terms
    for lam_m, fn in g.modes:
        v = fn()
        assert abs(v @ v - 1) < 1e-15
        assert np.abs(Al @ v - mpld(lam_m) * v).max() < tol, (name, lam_m)
    assert g.modes[0][0] == g.lmax and g.modes[1][0] == g.lmin
    if g.perron is not None:
        assert np.abs(Al @ g.perron - mpld(g.lmax) * g.perron).max() < tol and g.perron.min() > 0
        if lam is not None:
            assert float(g.gap) == pytest.approx(lam[-1] - lam[lam < lam[-1] - 1e-9].max(), abs=1e-9)


@pytest.mark.parametrize("name", ["grid30x50_r", "K30,50", "union", "circ500_w4"])
def test_references_against_scipy_and_mpmath(name):
    """The long double f(A) x against scipy's expm_multiply and a sparse solve, and a 30-digit dense mpmath computation on a
    small member of each family."""
    g = G(name)
    n = g.n
    A = sp.csr_matrix((np.ones(len(g.ci)), g.ci.astype(np.int64), g.ro.astype(np.int64)), shape=(n, n))
    x, vs = mode_vector(g, [1.0, 0.7, -0.4])
    for t in (-1.0, 0.5, 2.0):
        assert rel_err(spl.expm_multiply(t * A, x), exact_f(vs, x, mpf_of("exp", t))) < 1e-12
    al = 0.5 / float(g.lmax)
    ref = spl.spsolve((sp.identity(n) - al * A).tocsc(), x)
    assert rel_err(ref, exact_f(vs, x, mpf_of("resolvent", al))) < 1e-12
    if g.ones is not None:
        assert rel_err(spl.expm_multiply(A, np.ones(n)), g.ones(mpf_of("exp", 1.0))) < 1e-12
    small = {"grid30x50_r": grid(4, 5), "K30,50": bipartite(3, 4), "union": union([complete(3), complete(3), isolated(2), path(3)], "u"),
             "circ500_w4": circulant(9, [1, 2])}[name]
    with mp.workdps(30):
        M = mp.matrix(small.n, small.n)
        for i in range(small.n):
            for j in small.ci[small.ro[i]:small.ro[i + 1]]:
                M[i, int(j)] = 1
        xs, vss = mode_vector(small, [1.0, 0.7, -0.4])
        y = mp.expm(M) * mp.matrix([mp.mpf(float(v)) for v in xs])
        # the fp64 x leaves its modes' span by its rounding (~eps), which the mode expansion does not see
        assert rel_err(np.array([mpld(v) for v in y], LD), exact_f(vss, xs, mpf_of("exp", 1.0))) < 1e-15
        if small.ones is not None:
            y1 = mp.expm(M) * mp.matrix([1] * small.n)
            assert rel_err(np.array([mpld(v) for v in y1], LD), small.ones(mpf_of("exp", 1.0))) < 1e-18


@pytest.mark.parametrize("name", SMALL + ["star5000_r", "circ400_w8_r"])
def test_mode_vectors_are_fixed(name):
    """Every call builds the same x: the device and the oracle each build it, and the oracle's error calibrates the device's."""
    g = G(name)
    assert np.array_equal(mode_vector(g, COEFFS)[0], mode_vector(g, COEFFS)[0])


def test_interval_checker_rejects_one_ulp():
    """An interval that misses an exact eigenvalue by one ulp is rejected; touching it is accepted (Q_10: eigenvalue 8); no
    degenerate interval around a double holds an irrational eigenvalue."""
    spec = G("Q10_r").spectrum
    rho = 8.0 + 2.0 ** -40
    r = rho - 8.0
    assert contains_eigenvalue(rho, r, spec)
    assert not contains_eigenvalue(rho, np.nextafter(r, 0.0), spec)
    irr = cycle(7).spectrum[-2]                                   # 2 cos(2 pi / 7): no double equals it
    assert not contains_eigenvalue(float(irr), 0.0, [irr])
    assert contains_eigenvalue(float(irr), 2.0 ** -52, [irr])


def test_spmv_checker_rejects_dropped_entry():
    """fp64 row sums pass the per-row bound; dropping one entry of magnitude 2^-40 from a row is caught."""
    g = G("grid30x50_r")
    rng = np.random.default_rng(2)
    x = np.ldexp(rng.uniform(1, 2, g.n) * rng.choice([-1, 1], g.n), rng.integers(-40, 41, g.n))
    A = sp.csr_matrix((np.ones(len(g.ci)), g.ci.astype(np.int64), g.ro.astype(np.int64)), shape=(g.n, g.n))
    y = A @ x
    assert len(spmv_violations(g.ro, g.ci, x, y)) == 0
    i = 0
    x2 = x.copy()                                                   # every entry of row i is 2^-40
    nb = g.ci[g.ro[i]:g.ro[i + 1]]
    x2[nb] = np.ldexp(1.0, -40)
    y2 = A @ x2
    y2[i] -= x2[nb[0]]
    assert list(spmv_violations(g.ro, g.ci, x2, y2)) == [i]


# ---- GPU ------------------------------------------------------------------------------------------------------------------
SPMV_CONFIGS = {
    "auto": ({}, "auto"),
    "vector": ({}, "vector"),
    "warp": ({}, "warp"),
    "group4_narrow0": ({"LZ_SELL_GROUP": "4", "LZ_SELL_NARROW": "0"}, "auto"),
    "group4_narrow1": ({"LZ_SELL_GROUP": "4", "LZ_SELL_NARROW": "1"}, "auto"),
    "cols1": ({"LZ_SPMV_COLBLOCKS": "1"}, "auto"),
    "cols3": ({"LZ_SPMV_COLBLOCKS": "3"}, "auto"),
    "cols7": ({"LZ_SPMV_COLBLOCKS": "7"}, "auto"),
    "order_d": ({"LZ_ORDER": "d"}, "auto"),
    "order_n": ({"LZ_ORDER": "n"}, "auto"),
}
SPMV_GRAPHS = ["grid30x50_r", "K129", "K130_r", "circ400_w8_r", "circ1000_w130_r", "circ600_w128_r", "star_2^20_r", "Q16_r",
               "union_mixed_r", "torus64x64_r"]
BUILDERS["star_2^20_r"] = lambda: relabel(star(1 << 20))
BUILDERS["Q16_r"] = lambda: relabel(hypercube(16))
BUILDERS["K130_r"] = lambda: relabel(complete(130))
BUILDERS["torus512_r"] = lambda: relabel(torus(512, 512), seed=4)   # calibrates the 2^24-vertex torus


def make_context(lz, monkeypatch, env, variant="auto"):
    for key, val in env.items():
        monkeypatch.setenv(key, val)
    c = lz.Context(0)
    c.set_spmv_variant({"auto": lz.SPMV_AUTO, "vector": lz.SPMV_VECTOR, "warp": lz.SPMV_WARP}[variant])
    return c


@pytest.mark.gpu
@pytest.mark.parametrize("config", list(SPMV_CONFIGS))
def test_spmv_per_row_bound(lz, monkeypatch, config):
    """Every row within gamma_{d_i} sum_j |x_j| (rigorous for any order of the d_i additions) on x spanning 2^-40..2^40, and
    bit-exact on integer x (every partial sum is an integer below 2^53)."""
    env, variant = SPMV_CONFIGS[config]
    rng = np.random.default_rng(7)
    with make_context(lz, monkeypatch, env, variant) as c:
        for name in SPMV_GRAPHS:
            if env.get("LZ_ORDER") == "n" and name.startswith("star"):
                continue          # the forced natural order pads every 32-row slice to the hub's 2^20 entries: refused by design
            g = G(name)
            c.csr_upload(g.ro, g.ci)
            x = np.ldexp(rng.uniform(1, 2, g.n) * rng.choice([-1, 1], g.n), rng.integers(-40, 41, g.n))
            bad = spmv_violations(g.ro, g.ci, x, c.spmv_host(x))
            assert len(bad) == 0, (config, name, bad[:10])
            xi = rng.integers(-1000, 1001, g.n).astype(np.float64)
            A = sp.csr_matrix((np.ones(len(g.ci), np.int64), g.ci.astype(np.int64), g.ro.astype(np.int64)), shape=(g.n, g.n))
            assert np.array_equal(c.spmv_host(xi), (A @ xi.astype(np.int64)).astype(np.float64)), (config, name)


# f(A) x on every loop path. name -> (environment, basis, reorth)
PATHS = {
    "graph_replay": ({"LZ_CUDA_GRAPH": "1"}, "f64", False),
    "launch_by_launch": ({"LZ_CUDA_GRAPH": "0"}, "f64", False),
    "unlagged": ({"LZ_LAGGED_NORM": "0"}, "f64", False),
    "reorth": ({}, "f64", True),
    "fp32_basis": ({}, "f32", False),
}
FAMILIES = ["cycle1001", "circ500_w4", "circ400_w8_r", "circ1000_w130_r", "K131_r", "star5000_r", "K30,50", "Q10_r", "grid30x50_r",
            "torus64x64_r", "path300", "union", "union_mixed_r"]
COEFFS = [1.0, -0.6, 0.35]


@functools.lru_cache(maxsize=None)
def oracle_run(orc, name, k, reorth, f32):
    """The fp64 oracle's Lanczos from the graph's mode vector -> alpha, beta, Q (rounded to fp32 when f32) and the x it used."""
    g = G(name)
    x, vs = mode_vector(g, COEFFS)
    a, b, Q = orc.lanczos(g.ro, g.ci, k, x, orc.FULL if reorth else orc.PLAIN)
    if f32:
        Q = Q.astype(np.float32).astype(np.float64)
    return a, b, Q, x


def oracle_sane(e, kind, t, g, f32):
    """The oracle's own error must be rounding-sized, else the reference (x, modes or exact answer) is broken and 16x it proves
    nothing: fp64 within 1000x floor_f (measured: 1-120x, the most on the 5000-entry hub row of star5000), fp32 basis within 1e-6
    (measured: <= 4e-8)."""
    assert e < (1e-6 if f32 else 1e3 * floor_f(kind, t, g)), (g.name, kind, t, e)


def modes_s(g):
    return min(len(g.modes), len(COEFFS))


@pytest.mark.gpu
@pytest.mark.parametrize("name", FAMILIES)
@pytest.mark.parametrize("path", list(PATHS))
def test_matfun_exact(lz, orc, monkeypatch, path, name):
    """f(A) x for every function (EXP t = -1, 0.5, 1, 2; EXP_SCALED t = +-1; RESOLVENT alpha = -0.5, 0.5, 0.99 / lambda_max) at
    k = s (exact Krylov) and k = s + 20 (past the near-breakdown; with full reorthogonalisation at most the number of distinct
    eigenvalues, beyond which beta = 0 exactly, the documented breakdown). Limit: FACTOR x the fp64 oracle's error against the same
    exact answer (same graph, x, k, function; its basis rounded to fp32 for the fp32-basis path) plus the floor `floor_f`. Also
    lz_choose_k (g)."""
    env, basis, reorth = PATHS[path]
    g = G(name)
    s = modes_s(g)
    x, vs = mode_vector(g, COEFFS)
    xnorm = float(np.sqrt(np.asarray(x, LD) @ np.asarray(x, LD)))
    with make_context(lz, monkeypatch, env) as c:
        if basis == "f32":
            c.set_basis_precision(lz.BASIS_F32)
        c.csr_upload(g.ro, g.ci)
        c.set_start_vector(x)
        kmax = min(s + 20, len(g.spectrum)) if reorth and g.spectrum is not None else s + 20
        for k in sorted({s, kmax}):
            c.lanczos_run(k, lz.REORTH_FULL if reorth else lz.REORTH_NONE)
            a, b, Q, x_orc = oracle_run(orc, name, k, reorth, basis == "f32")
            assert np.array_equal(x_orc, x)
            for kind, p in FUNCS:
                t = fparam(kind, p, g.lmax)
                c.set_matfun({"exp": lz.MATFUN_EXP, "scaled": lz.MATFUN_EXP_SCALED, "resolvent": lz.MATFUN_RESOLVENT}[kind], t)
                c.tridiag_expv()
                c.multout()
                y = c.get_ans()
                ls = c.matfun_scale()
                ref = exact_f(vs, x, mpf_of(kind, t, ls))
                y_orc = oracle_f(a, b, Q, xnorm, kind, t)
                if kind == "scaled":
                    ls_orc = float(np.max(t * np.linalg.eigvalsh(np.diag(a) + np.diag(b, 1) + np.diag(b, -1))))
                    y_orc = y_orc * np.exp(ls_orc - ls)
                oracle_sane(rel_err(y_orc, ref), kind, t, g, basis == "f32")
                lim = FACTOR * rel_err(y_orc, ref) + floor_f(kind, t, g)
                err = rel_err(y, ref)
                assert err <= lim, (path, name, k, kind, t, err, lim)
            if k == kmax and k > s:
                c.set_matfun(lz.MATFUN_EXP, 1.0)
                c.tridiag_expv()
                assert c.choose_k(1e-12)[0] <= s + 1, (path, name, c.choose_k(1e-12))


@pytest.mark.gpu
@pytest.mark.parametrize("path", ["graph_replay", "reorth", "fp32_basis"])
def test_matfun_ones(lz, orc, monkeypatch, path):
    """x = ones on the non-regular families, exact answers from the product sine transform (grids) and the two-mode closed form
    (stars, complete bipartite); Krylov is not exact here (k = 40 on the grid), so the oracle's error includes truncation."""
    env, basis, reorth = PATHS[path]
    with make_context(lz, monkeypatch, env) as c:
        if basis == "f32":
            c.set_basis_precision(lz.BASIS_F32)
        for name, k in (("grid30x50_r", 40), ("grid30x50", 40), ("star5000_r", 2), ("K30,50", 3)):
            g = G(name)
            c.csr_upload(g.ro, g.ci)
            c.set_start_vector(None)
            c.lanczos_run(k, lz.REORTH_FULL if reorth else lz.REORTH_NONE)
            a, b, Q = orc.lanczos(g.ro, g.ci, k, np.ones(g.n), orc.FULL if reorth else orc.PLAIN)
            if basis == "f32":
                Q = Q.astype(np.float32).astype(np.float64)
            for kind, p in (("exp", 1.0), ("exp", -1.0), ("resolvent", 0.9)):
                t = fparam(kind, p, g.lmax)
                c.set_matfun(lz.MATFUN_EXP if kind == "exp" else lz.MATFUN_RESOLVENT, t)
                c.tridiag_expv()
                c.multout()
                ref = g.ones(mpf_of(kind, t))
                lim = FACTOR * rel_err(oracle_f(a, b, Q, np.sqrt(g.n), kind, t), ref) + floor_f(kind, t, g)
                assert rel_err(c.get_ans(), ref) <= lim, (path, name, kind, rel_err(c.get_ans(), ref), lim)


def ritz_graphs():
    for n in (2, 3, 129, 130, 131, 2049, 4097):
        yield f"K{n}", lambda n=n: relabel(complete(n)) if n > 3 else complete(n)
    for d in (2, 3, 4, 10, 16, 22):
        yield f"Q{d}", lambda d=d: relabel(hypercube(d))
    for n in (3, 4, 5, 100, 1001, 65536):
        yield f"cycle{n}", lambda n=n: relabel(cycle(n))
    for b in (1, 2, 3, 100, 4096, 1 << 20, 1 << 22):
        yield f"star{b}", lambda b=b: relabel(star(b))


@pytest.mark.gpu
@pytest.mark.parametrize("reorth", [False, True])
def test_ritz_zero_slack(lz, reorth):
    """Every returned interval [rho_j - r_j, rho_j + r_j] holds an exact eigenvalue and lo <= lambda_max <= hi, compared in mpmath
    with no slack, for m = 1, 3, 5, 16 (every k_ritz_combine instance) on K_n, Q_d, C_n and stars, from a random start (converged
    to machine precision where the graph has few distinct eigenvalues) and from ones on the stars."""
    rng = np.random.default_rng(9)
    with lz.Context(0) as c:
        for name, build in ritz_graphs():
            g = build()
            c.csr_upload(g.ro, g.ci)
            starts = [rng.standard_normal(g.n)] + ([None] if name.startswith("star") else [])
            for x in starts:
                # under CGS2 beta = 0 exactly past the grade of x: the number of distinct eigenvalues, 2 for ones on a star
                k = min(g.n, 30, len(g.spectrum) if x is not None else 2) if reorth else min(g.n, 30)
                c.set_start_vector(x)
                c.lanczos_run(k, lz.REORTH_FULL if reorth else lz.REORTH_NONE)
                for m in (1, 3, 5, 16):
                    if m > k:
                        continue
                    th, rho, res = c.ritz(m)
                    for j in range(m):
                        assert contains_eigenvalue(rho[j], res[j], g.spectrum), (name, reorth, m, j, rho[j], res[j])
                    lo, hi = c.spectral_radius_bounds()
                    assert mp.mpf(lo) <= g.lmax <= mp.mpf(hi), (name, reorth, m, lo, hi)


@pytest.mark.gpu
def test_eigenvector_centrality_exact(lz):
    """||y_0 - v|| <= sqrt(2) r_0 / (gap - r_0) + 4 eps with v the exact Perron vector (sin-theta bound with the exact gap; r_0 is
    certified, so the bound is rigorous for the stored y_0; 4 eps covers the long double evaluation of v). Random positive start;
    graphs whose Perron pair converges within k = min(80, n) (relative gaps >= 0.02)."""
    rng = np.random.default_rng(12)
    with lz.Context(0) as c:
        for name in ("grid8x13_r", "star5000_r", "K131_r", "Q10_r", "circ1000_w130_r"):
            g = G(name)
            c.csr_upload(g.ro, g.ci)
            c.set_start_vector(rng.uniform(0.5, 1.5, g.n))
            c.lanczos_run(min(80, g.n))
            th, rho, res = c.ritz(1)
            y = np.asarray(c.get_ans(), LD)
            gap = float(g.gap)
            assert res[0] < gap / 2, (name, res[0], gap)
            bound = np.sqrt(2) * res[0] / (gap - res[0]) + 4 * EPS
            err = float(np.sqrt((y - g.perron) @ (y - g.perron)))
            assert err <= bound, (name, err, bound)


@pytest.mark.gpu
def test_katz_exact(lz, orc):
    """alpha = 0.9 / hi: alpha lambda_max < 1 holds exactly (mpmath), and the resolvent with x = ones matches the exact Katz vector
    within FACTOR x the oracle's error plus 4 eps."""
    with lz.Context(0) as c:
        for name, k in (("grid30x50_r", 60), ("star5000_r", 2), ("K30,50", 3)):
            g = G(name)
            c.csr_upload(g.ro, g.ci)
            c.set_start_vector(None)
            c.lanczos_run(k)
            c.ritz(1)
            lo, hi = c.spectral_radius_bounds()
            alpha = 0.9 / hi
            assert mp.mpf(alpha) * g.lmax < 1 and mp.mpf(lo) <= g.lmax <= mp.mpf(hi), (name, lo, hi)
            c.set_matfun(lz.MATFUN_RESOLVENT, alpha)
            c.tridiag_expv()
            c.multout()
            ref = g.ones(mpf_of("resolvent", alpha))
            a, b, Q = orc.lanczos(g.ro, g.ci, k, np.ones(g.n))
            lim = FACTOR * rel_err(oracle_f(a, b, Q, np.sqrt(g.n), "resolvent", alpha), ref) + floor_f("resolvent", alpha, g)
            assert rel_err(c.get_ans(), ref) <= lim, (name, rel_err(c.get_ans(), ref), lim)


@pytest.mark.gpu
def test_top_k_exact(lz, orc):
    """lz_top_k against the exact answer's ranking wherever that ranking is decided: the prefix of the top 100 up to the first
    gap (between consecutive exact values) within twice the error bound ||y - y_exact||_inf. The grid 30 x 50 with x on the sine
    modes (1,1), (2,1), (1,2), (2,2): the antisymmetric modes break both reflections, so the exact values have no ties."""
    with lz.Context(0) as c:
        for a, b in ((30, 50), (61, 40)):
            g = grid(a, b)
            Sa, Sb, mu, nu = g.extra["sines"]
            vs = [(mu[i] + nu[j], np.outer(Sa[i], Sb[j]).reshape(-1)) for i, j in ((0, 0), (1, 0), (0, 1), (1, 1))]
            x = sum(LD(w) * v for w, (_, v) in zip((1.0, 0.8, -0.7, 0.45), vs)).astype(np.float64)
            name = g.name
            c.csr_upload(g.ro, g.ci)
            c.set_start_vector(x)
            c.lanczos_run(14)
            c.tridiag_expv()
            c.multout()
            y = c.get_ans()
            ref = exact_f(vs, x, mpf_of("exp", 1.0))
            idx, val = c.top_k(100)
            assert np.array_equal(val, y[idx]) and np.array_equal(idx, orc.top_k(y))
            bound = float(np.abs(np.asarray(y, LD) - ref).max())
            order = np.argsort(-ref.astype(np.float64), kind="stable")
            sv = ref[order][:101]
            small = np.flatnonzero(sv[:-1] - sv[1:] <= 2 * bound)
            p = int(small[0]) if len(small) else 100
            assert p >= 10, (name, p)
            assert np.array_equal(idx[:p], order[:p]), name


@pytest.mark.gpu
def test_scale_invariance(lz, monkeypatch):
    """f(A)(2^p x) == 2^p f(A) x bit for bit, for p in [-1000, 1000] wherever 2^p x, every basis coefficient 2^p c_j and the
    answer stay normal: scaling by a power of two is exact, so one rounding of ||x|| differently would show. Also a zero or
    non-finite start vector is refused with LZ_ERR_ARG."""
    tiny, huge = np.finfo(np.float64).tiny, np.finfo(np.float64).max
    with lz.Context(0) as c:
        for name, reorth in (("grid30x50_r", False), ("union_mixed_r", True)):
            g = G(name)
            x, _ = mode_vector(g, COEFFS)
            x = x + 0.01 * np.random.default_rng(3).standard_normal(g.n)
            c.csr_upload(g.ro, g.ci)
            mode = lz.REORTH_FULL if reorth else lz.REORTH_NONE
            for kind, t in ((lz.MATFUN_EXP, 1.0), (lz.MATFUN_RESOLVENT, 0.5 / float(g.lmax))):
                c.set_matfun(kind, t)
                y0 = c.expv_host(x, 30, mode)
                _, _, coef = c.get_eigen()
                q = np.stack([c.get_basis(j) for j in range(30)])
                small = min(np.abs(coef[coef != 0]).min() * np.abs(q[q != 0]).min(), np.abs(y0[y0 != 0]).min(),
                            np.abs(x[x != 0]).min())
                large = max(np.abs(coef).max() * np.sqrt(g.n), np.abs(y0).max(), np.abs(x).max())
                tried = 0
                for p in list(range(-1000, 1001, 37)) + [-1000, 1000, -600, 600]:
                    if not (p + np.log2(small) >= np.log2(tiny) + 60 and p + np.log2(large) <= np.log2(huge) - 60):
                        continue
                    tried += 1
                    y = c.expv_host(np.ldexp(x, p), 30, mode)
                    assert np.array_equal(y, np.ldexp(y0, p)), (name, kind, p)
                assert tried >= 30
            for bad in (np.zeros(g.n), np.where(np.arange(g.n) == 3, np.nan, x), np.where(np.arange(g.n) == 5, np.inf, x)):
                with pytest.raises(lz.LzError) as e:
                    c.set_start_vector(bad)
                assert e.value.code == -1
            # entries far below 1e-154 (their squares underflow) and far above 1e154 (their squares overflow)
            c.set_matfun(lz.MATFUN_EXP, 1.0)
            y0 = c.expv_host(x, 30, mode)
            for p in (-1060, -1030, 1000, 1020):
                xs = np.ldexp(x, p)
                if p < 0:
                    ys = c.expv_host(xs, 30, mode)
                    # 2^-1030 x has subnormal entries (digits lost on input): close; 2^-1060 x: only finite
                    assert (rel_err(np.ldexp(ys, -p), y0) < 1e-10) if p > -1050 else np.isfinite(ys).all(), (name, p)
                else:
                    c.set_start_vector(xs)
                    c.lanczos_run(30, mode)
                    c.set_matfun(lz.MATFUN_EXP_SCALED, 1.0)
                    c.tridiag_expv()
                    c.multout()
                    ys = c.get_ans()
                    assert rel_err(np.ldexp(ys, -p) * np.exp(c.matfun_scale()), y0) < 1e-13, (name, p)
                    c.set_matfun(lz.MATFUN_EXP, 1.0)


@pytest.mark.gpu
def test_torus_2p24(lz, orc, monkeypatch):
    """C3 scale: torus 4096 x 4096 (2^24 vertices) relabelled, so the gathers span two column blocks. Every entry of f(A) x against
    the exact answer. The oracle is too slow here (its basis alone is 6 GB at k = 23), so the limits are calibrated on the same
    family one size down (torus 512 x 512, same modes, k, functions), on the default path and with full reorthogonalisation."""
    big = relabel(torus(4096, 4096), seed=4)
    cal = G("torus512_r")
    s = 3
    with lz.Context(0) as c:
        c.csr_upload(big.ro, big.ci)
        x, vs = mode_vector(big, COEFFS)
        c.set_start_vector(x)
        for reorth in (False, True):
            for k in (s, s + 20):
                c.lanczos_run(k, lz.REORTH_FULL if reorth else lz.REORTH_NONE)
                a, b, Q, xc_orc = oracle_run(orc, "torus512_r", k, reorth, False)
                xc, vsc = mode_vector(cal, COEFFS)
                assert np.array_equal(xc_orc, xc)
                xcn = float(np.sqrt(xc @ xc))
                for kind, p in (("exp", 1.0), ("exp", -1.0), ("resolvent", 0.99)):
                    t = fparam(kind, p, big.lmax)
                    c.set_matfun(lz.MATFUN_EXP if kind == "exp" else lz.MATFUN_RESOLVENT, t)
                    c.tridiag_expv()
                    c.multout()
                    ref = exact_f(vs, x, mpf_of(kind, t))
                    e_orc = rel_err(oracle_f(a, b, Q, xcn, kind, t), exact_f(vsc, xc, mpf_of(kind, t)))
                    oracle_sane(e_orc, kind, t, cal, False)
                    lim = FACTOR * e_orc + floor_f(kind, t, big)
                    err = rel_err(c.get_ans(), ref)
                    assert err <= lim, (reorth, k, kind, err, lim)
        c.set_start_vector(x)
        c.lanczos_run(s + 20)
        c.ritz(3)
        lo, hi = c.spectral_radius_bounds()
        assert mp.mpf(lo) <= big.lmax <= mp.mpf(hi)
