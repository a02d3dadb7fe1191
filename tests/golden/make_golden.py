"""Generate the golden fixtures of tests/golden/ from the UNMODIFIED reference.

Needs the reference binaries under oracle/_ref (`make -C oracle ref REF=<SuperLU_DIST source tree>`):

    python tests/golden/make_golden.py

Each fixture is the input of pdgstrf3d (dLUstruct_t + dtrf3Dpartition_t as the reference built them)
and the factors the reference's own pdgstrf3d (CPU path, 1x1x1, OMP_NUM_THREADS=1, scipy OpenBLAS)
produced, captured by the hook oracle/ref_build/pdgstrf3d_hook.c (SLU_B200_HOOK=dump).
"""
import gzip
import os
import shutil
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from superlu_dist_b200 import dumpio, hostlib, matgen  # noqa: E402

REF = os.path.join(ROOT, "oracle", "_ref")
OUT = os.path.dirname(os.path.abspath(__file__))


def run(cmd, dump):
    env = dict(os.environ, SLU_B200_HOOK="dump", SLU_B200_DUMP=dump, OMP_NUM_THREADS="1")
    subprocess.run(cmd, env=env, check=True, stdout=subprocess.DEVNULL)
    return dumpio.read_records(dump + ".pre"), dumpio.read_records(dump + ".post")


def main():
    with tempfile.TemporaryDirectory() as tmp:
        # the reference's EXAMPLE matrices are stored here gzipped; the drivers read them unpacked
        for f in ("g4.rua", "g20.rua", "cg20.cua"):
            with gzip.open(os.path.join(OUT, f + ".gz"), "rb") as src, open(os.path.join(tmp, f), "wb") as dst:
                shutil.copyfileobj(src, dst)
        # config #1 of BASELINE.json: EXAMPLE/pddrive3d on g20.rua, 1x1x1 (default options:
        # equilibration, MC64 row permutation, MMD(A'+A) column ordering)
        for name in ("g4", "g20"):
            pre, post = run([os.path.join(REF, "pddrive3d"), "-r", "1", "-c", "1", "-d", "1",
                             os.path.join(tmp, name + ".rua")], os.path.join(tmp, name))
            dumpio.save_npz(os.path.join(OUT, name + "_pddrive3d.npz"), pre, post)
        # config #5 of BASELINE.json (doublecomplex mirror): pzdrive3d on cg20.cua, and the same file with every
        # value scaled by 1000 ("cg20.cua scaled x1000", reading B of SURVEY 8d: exercises anorm/thresh scaling)
        pre, post = run([os.path.join(REF, "pzdrive3d"), "-r", "1", "-c", "1", "-d", "1", os.path.join(tmp, "cg20.cua")],
                        os.path.join(tmp, "cg20"))
        dumpio.save_npz(os.path.join(OUT, "cg20_pzdrive3d.npz"), pre, post)
        # same matrix, tiny-pivot replacement on, no row permutation, smaller supernodes
        mat = os.path.join(tmp, "p.bin")
        for tag, N, leaf, extra in (("poisson8_nd", 8, 8, ["--maxsup", "16", "--relax", "4"]),
                                    ("poisson9_nd_tiny", 9, 16, ["--maxsup", "24", "--relax", "6", "--tiny", "1"])):
            rp, ci, v = hostlib.poisson3d(N)
            matgen.write_matrix_bin(mat, rp, ci, v)
            perm = hostlib.nd_order(N, leaf=leaf)
            pf = os.path.join(tmp, "perm.bin")
            matgen.write_perm_bin(pf, perm)
            pre, post = run([os.path.join(REF, "ref_driver"), mat, "--permc", pf] + extra, os.path.join(tmp, tag))
            dumpio.save_npz(os.path.join(OUT, tag + ".npz"), pre, post)
        # unsymmetric values / unsymmetric-looking skyline: fem-like 2 dof, MMD ordering from the reference
        rp, ci, v = hostlib.fem3d(5, 5, 5, dof=2, seed=20260924)
        matgen.write_matrix_bin(mat, rp, ci, v)
        pre, post = run([os.path.join(REF, "ref_driver"), mat, "--colperm", "mmd", "--maxsup", "20", "--relax", "5"],
                        os.path.join(tmp, "fem"))
        dumpio.save_npz(os.path.join(OUT, "fem5_mmd.npz"), pre, post)
        # unsymmetric PATTERN (skyline U with short segments): banded random matrix, dominant diagonal
        import numpy as np
        import scipy.sparse as sp
        rng = np.random.default_rng(20260924)
        n = 360
        M = sp.random(n, n, density=0.012, random_state=rng, format="lil")
        for i in range(n - 1):
            M[i + 1, i] = rng.uniform(-1, 0)          # sub-diagonal chain -> long etree paths
        M = sp.csr_matrix(M)
        M = (M + sp.diags(np.asarray(abs(M).sum(axis=1)).ravel() + 1.0)).tocsr()
        M.sort_indices()
        matgen.write_matrix_bin(mat, M.indptr, M.indices, M.data)
        pre, post = run([os.path.join(REF, "ref_driver"), mat, "--colperm", "mmd", "--maxsup", "32", "--relax", "8"],
                        os.path.join(tmp, "unsym"))
        dumpio.save_npz(os.path.join(OUT, "unsym360_mmd.npz"), pre, post)
    for f in sorted(os.listdir(OUT)):
        if f.endswith(".npz"):
            print(f, os.path.getsize(os.path.join(OUT, f)))


if __name__ == "__main__":
    main()
