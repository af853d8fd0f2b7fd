"""Generates tests/golden/*.npz by running the UNMODIFIED reference (oracle/_ref/ref_final = parallel-final host path,
oracle/_ref/ref_serial = serial/ incl. its Arnoldi-assisted variant) on small seeded graphs from our deterministic
generators. Run in the build container (needs /root/reference compiled by `make -C oracle ref`):

    python tests/golden/make_golden.py

Each file stores the generator spec, alpha/beta/ans of the reference, and for the small cases the CSR itself, so the
tests can (1) pin the C restatement oracle/lanczos_oracle.c against the real reference without /root/reference, and
(2) compare the CUDA path with the reference's own output on the GPU box."""
import json
import os
import subprocess
import sys
import tempfile
import zipfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(HERE))
import __graft_entry__ as g  # noqa: E402
import oracle  # noqa: E402

lz = g.load_package()

CASES = {
    # name: (spec, k)          C1 = BASELINE.json configs[0]
    "c1_er_n10000_k20": (lz.GraphSpec.er(10000, 50000, 20261018), 20),
    "er_n2000_k20": (lz.GraphSpec.er(2000, 10000, 3), 20),
    "rmat_s12_k30": (lz.GraphSpec.rmat(12, 8, 1), 30),
    "rmat_s14_k50": (lz.GraphSpec.rmat(14, 8, 1), 50),
    "band_n4096_k40": (lz.GraphSpec.band(4096, 5), 40),
    "er_n257_k10_ragged": (lz.GraphSpec.er(257, 600, 11), 10),
}
# the Arnoldi-assisted answer is only stored where tests/test_oracle.py compares with it (keeps rmat_s14_k50 under 1 MB)
ARNOLDI_CASES = ("er_n2000_k20", "rmat_s12_k30", "band_n4096_k40")


def spec_dict(s):
    return {f: getattr(s, f) for f, _ in s._fields_}


def save_npz(path, **arrays):
    """np.savez with LZMA instead of deflate: np.load reads it like any .npz, and rmat_s14_k50 comes out 15% smaller."""
    with zipfile.ZipFile(path, "w", zipfile.ZIP_LZMA) as z:
        for name, a in arrays.items():
            with z.open(name + ".npy", "w") as f:
                np.lib.format.write_array(f, np.asanyarray(a), allow_pickle=False)


def main():
    assert oracle.have_ref(), "build the reference first: make -C oracle ref"
    for name, (spec, k) in CASES.items():
        n, ro, ci = lz.generate_host(spec)
        with tempfile.TemporaryDirectory() as td:
            mtx = os.path.join(td, "g.mtx")
            lz.write_text(mtx, ro, ci)
            # primary oracle: parallel-final host path through the reference's own text loader
            out = os.path.join(td, "f")
            subprocess.run([oracle.REF_FINAL, "--mtx", mtx, "-k", str(k), "--out", out], check=True, capture_output=True)
            ans = np.fromfile(out + ".ans.f64")
            alpha = np.fromfile(out + ".alpha.f64")
            beta = np.fromfile(out + ".beta.f64")
            # same through CSR injection must be bit-identical
            r2 = oracle.run_ref_final(ro, ci, k)
            assert np.array_equal(r2["ans"], ans) and np.array_equal(r2["alpha"], alpha)
            # secondary: serial/ (zero-new patched), plain and Arnoldi-assisted
            outs = os.path.join(td, "s")
            subprocess.run([oracle.REF_SERIAL, "--mtx", mtx, "-k", str(k), "--out", outs], check=True, capture_output=True)
            ans_serial = np.fromfile(outs + ".ans.f64")
            outa = os.path.join(td, "a")
            subprocess.run([oracle.REF_SERIAL, "--mtx", mtx, "-k", str(k), "--arnoldi", "--out", outa], check=True, capture_output=True)
            ans_arn = np.fromfile(outa + ".ans.f64")
            alpha_arn = np.fromfile(outa + ".alpha.f64")
        # a random (non-constant) start vector through CSR injection
        rng = np.random.default_rng(1234)
        xr = rng.random(n)
        r3 = oracle.run_ref_final(ro, ci, k, x=xr)
        # SpMV golden: the reference's spMV is exercised inside Lanczos; pin it directly with alpha_0 = q0.A.q0 and with
        # A*1 = degree vector (exact in fp64).
        arnoldi = dict(ans_arnoldi=ans_arn, alpha_arnoldi=alpha_arn) if name in ARNOLDI_CASES else {}
        save_npz(
            os.path.join(HERE, name + ".npz"),
            spec=json.dumps(spec_dict(spec)), k=k, n=n, row_offset=ro, col_idx=ci,
            ans=ans, alpha=alpha, beta=beta, ans_serial=ans_serial, **arnoldi,
            x_random=xr, ans_random=r3["ans"], alpha_random=r3["alpha"], beta_random=r3["beta"])
        rel_ser = np.linalg.norm(ans - ans_serial) / np.linalg.norm(ans)
        rel_arn = np.linalg.norm(ans - ans_arn) / np.linalg.norm(ans)
        print(f"{name}: n={n} nnz={ro[-1]} k={k} |ans|={np.linalg.norm(ans):.6e} final-vs-serial={rel_ser:.2e} "
              f"final-vs-arnoldi={rel_arn:.2e} top100 gap={oracle.top_gap(ans):.2e}")


def main_float():
    """Single-precision goldens: the reference's own float instantiation (lanczosDecomp<float> -> eigenDecomp<float> ->
    multOut<float>, cu_lanczos.cu:144 / README.md:21) on two of the graphs above, stored as float32 next to the distance
    between the reference's float and double answers — the bar our fp32-basis mode is held to (SURVEY 8f-4)."""
    out = {}
    for name in ("rmat_s14_k50", "c1_er_n10000_k20", "band_n4096_k40"):
        spec, k = CASES[name]
        n, ro, ci = lz.generate_host(spec)
        r64 = oracle.run_ref_final(ro, ci, k)
        r32 = oracle.run_ref_final(ro, ci, k, single=True)
        d = float(np.linalg.norm(r32["ans"] - r64["ans"]) / np.linalg.norm(r64["ans"]))
        out[name + "__ans_f32"] = r32["ans"].astype(np.float32)
        out[name + "__ref_f32_vs_f64"] = np.float64(d)
        print(f"{name}: reference float vs double relative 2-norm {d:.3e}")
    np.savez_compressed(os.path.join(HERE, "reference_float.npz"), **out)


if __name__ == "__main__":
    if len(sys.argv) > 1 and sys.argv[1] == "--float":
        main_float()
    else:
        main()
