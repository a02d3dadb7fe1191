"""The doublecomplex solve and device-side distribution on the HBM-resident factors (slu_b200_z_solve, the job of
pzgstrs3d, SRC/complex16/pzgstrs3d.c:6694; slu_b200_z_fill_csr, the job of pzdistribute3d,
SRC/complex16/pzdistribute3d.c:24): forward error on generated matrices, the widest complex supernodes, the reference's
own cg20 matrix, the CSR scatter against the host-distributed panels, and the Z-distributed solve on 1 x 1 x Pz."""
import os
import subprocess
import sys

import numpy as np
import pytest
import scipy.sparse as sp

from oracle import oracle
from superlu_dist_b200 import capi
from util import complex_problem, load_fixture, poisson_problem, rel_err

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))


def complex_csr(seed=0, **kw):
    """The CSR of the matrix complex_problem(seed, **kw) distributes: poisson_problem's matrix plus 1j * vi, vi drawn by
    the same seeded recipe.  -> (rowptr, colind, complex values)"""
    _, (rp, ci, v) = poisson_problem(**kw)
    rng = np.random.default_rng(seed)
    rows = np.repeat(np.arange(len(rp) - 1), np.diff(rp))
    vi = np.where(rows == ci, 0.25, 0.5 * rng.uniform(-1.0, 1.0, len(v)))
    return rp, ci, v + 1j * vi


def permuted_matvec(perm, rp, ci, val, x):
    """(P A P^T) x for perm[old] = new: the right-hand side in the ordering of the factored matrix.  x: (n,) or (k, n)."""
    n = len(rp) - 1
    rows = np.repeat(np.arange(n), np.diff(rp))
    a = sp.csr_matrix((val, (perm[rows], perm[ci])), shape=(n, n))
    return (a @ np.asarray(x).T).T


def crandn(rng, *shape):
    return rng.standard_normal(shape) + 1j * rng.standard_normal(shape)


def _check_solves(h, prob, rp, ci, val, seed):
    xtrue = crandn(np.random.default_rng(seed), 3, prob.n)
    b = permuted_matvec(prob.perm, rp, ci, val, xtrue)
    for _ in range(2):
        for rhs, ref in ((b, xtrue), (b[0], xtrue[0])):
            x = h.solve(rhs)
            assert x.dtype == np.complex128 and x.shape == ref.shape
            err = np.abs(x - ref).max()
            assert err <= 1e-10 * np.abs(ref).max(), err


@pytest.mark.parametrize("kw", [dict(N=10, leaf=8, relax=8, maxsup=32), dict(N=16, leaf=16, relax=32, maxsup=256),
                                dict(N=6, leaf=4, relax=8, maxsup=200, fem=3)])
def test_complex_solve_on_resident_factors(kw):
    prob = complex_problem(**kw)
    rp, ci, val = complex_csr(**kw)
    h = capi.Handle(prob, 0)
    with pytest.raises(RuntimeError):
        h.solve(np.ones(prob.n, np.complex128))   # not factored yet
    h.upload()
    assert h.factor() == 0
    _check_solves(h, prob, rp, ci, val, seed=1)
    st = h.stats()
    assert st.reserved[4] > 0 and st.reserved[5] > 0
    h.close()


def test_complex_solve_widest_supernodes():
    """Supernodes of MAX_NS_HELD = 256 columns, with U panels: the diagonal sweep and the U-update buffer at their
    limit in the doublecomplex build."""
    kw = dict(N=20, leaf=16, relax=32, maxsup=256)
    prob = complex_problem(**kw)
    ns = np.diff(prob.xsup)
    assert ns.max() == 256
    assert any(prob.uval_len[k] > 0 for k in np.nonzero(ns == 256)[0])
    rp, ci, val = complex_csr(**kw)
    h = capi.Handle(prob, 0)
    h.upload()
    assert h.factor() == 0
    _check_solves(h, prob, rp, ci, val, seed=2)
    h.close()


def test_complex_solve_reference_matrix():
    """cg20 as the reference's pzdrive3d factors it.  The matrix is not diagonally dominant: backward error."""
    prob, _, post = load_fixture("cg20_pzdrive3d")
    lay = prob.layers[0]
    a = prob.dense(lay, False)
    assert a.shape == (400, 400)
    xtrue = crandn(np.random.default_rng(3), prob.n)
    b = a @ xtrue
    h = capi.Handle(prob, 0)
    h.upload()
    assert h.factor() == int(post["info"][0]) == 0
    x = h.solve(b)
    h.close()
    berr = np.abs(a @ x - b).max() / (np.abs(a).sum(axis=1).max() * np.abs(x).max())
    assert berr <= 1e-13, berr


@pytest.mark.parametrize("kw", [dict(N=10, leaf=8, relax=8, maxsup=32), dict(N=6, leaf=4, relax=8, maxsup=200, fem=3)])
def test_complex_device_side_distribution(kw):
    """slu_b200_z_fill_csr puts exactly the values into HBM that the host distribution of complex_problem does
    (which also pins complex_csr to that recipe); the factors then match the oracle and solve."""
    prob = complex_problem(**kw)
    rp, ci, val = complex_csr(**kw)
    want = prob.layers[0].copy()
    prob.layers[0].lval[:] = -7.0 + 3.0j              # poison the host arrays: they must not be read
    prob.layers[0].uval[:] = -7.0 + 3.0j
    h = capi.Handle(prob, 0)
    h.fill_csr(rp, ci, val, prob.perm)
    h.download()
    assert np.array_equal(prob.layers[0].lval, want.lval) and np.array_equal(prob.layers[0].uval, want.uval)
    assert h.factor() == 0
    h.download()
    chk = complex_problem(**kw)
    oracle.factor(chk)
    assert rel_err(prob.layers[0].lval, chk.layers[0].lval) < 1e-10
    assert rel_err(prob.layers[0].uval, chk.layers[0].uval) < 1e-10
    _check_solves(h, prob, rp, ci, val, seed=4)
    h.close()


@pytest.mark.parametrize("world", [2, 4])
def test_complex_solve_1x1xPz(world):
    """The Z-distributed complex solve (all-reduces climb the Z tree and spread the owner's solution back): every rank
    passes the same b and receives the full x."""
    if capi.device_count() < world:
        pytest.skip(f"needs {world} GPUs")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={world}",
           "--master-addr", "127.0.0.1", "--master-port", str(29820 + world), os.path.join(HERE, "zsolve_worker.py"), "14"]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=900)
    assert out.returncode == 0, out.stdout[-2000:] + out.stderr[-3000:]
    assert out.stdout.count("complex solve err") == world
