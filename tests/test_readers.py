"""Matrix-file readers of libslu_b200_host (SURVEY 8f N4): Harwell-Boeing, Matrix Market, the reference's binary dump.
Checked against SciPy's independent readers/writers on generated matrices, and against the reference's own EXAMPLE
fixtures (g4.rua, g20.rua, big.rua, cg20.cua, stored gzipped and otherwise unchanged in tests/golden)."""
import gzip
import os

import numpy as np
import pytest
import scipy.io
import scipy.sparse as sp

from superlu_dist_b200 import hostlib, matgen

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def _rand(n, density, seed, sym=False, cx=False):
    rng = np.random.default_rng(seed)
    a = sp.random(n, n, density=density, random_state=rng, format="csr") + sp.eye(n) * n
    if cx:
        a = a + 1j * sp.random(n, n, density=density, random_state=rng, format="csr")
    if sym:
        a = a + a.T
    a = a.tocsr()
    a.sort_indices()
    return a


def _as_csr(nr, nc, ptr, ind, val):
    return sp.csr_matrix((val, ind, ptr), shape=(nr, nc))


@pytest.mark.parametrize("sym", [False, True])
def test_matrix_market_roundtrip(tmp_path, sym):
    a = _rand(37, 0.1, 1, sym=sym)
    path = str(tmp_path / "a.mtx")
    scipy.io.mmwrite(path, a, symmetry="symmetric" if sym else "general")
    b = _as_csr(*hostlib.read_matrix(path))
    assert abs(a - b).max() < 1e-14 * abs(a).max()


def test_matrix_market_complex_and_pattern(tmp_path):
    a = _rand(20, 0.2, 2, cx=True)
    path = str(tmp_path / "c.mtx")
    scipy.io.mmwrite(path, a)
    nr, nc, ptr, ind, val = hostlib.read_matrix(path)
    assert val.dtype == np.complex128
    assert abs(a - _as_csr(nr, nc, ptr, ind, val)).max() < 1e-14 * abs(a).max()
    with open(tmp_path / "p.mtx", "w") as f:      # pattern, 0-based indices (dreadMM.c:147-160 detects the base)
        f.write("%%MatrixMarket matrix coordinate pattern general\n% comment\n3 3 3\n0 0\n1 2\n2 1\n")
    nr, nc, ptr, ind, val = hostlib.read_matrix(str(tmp_path / "p.mtx"))
    assert _as_csr(nr, nc, ptr, ind, val).toarray().tolist() == [[1, 0, 0], [0, 0, 1], [0, 1, 0]]


def test_harwell_boeing_roundtrip(tmp_path):
    a = _rand(45, 0.08, 3)
    path = str(tmp_path / "a.rua")
    matgen.write_harwell_boeing(path, a.indptr.astype(np.int32), a.indices.astype(np.int32), a.data)
    b = _as_csr(*hostlib.read_matrix(path))
    assert abs(a - b).max() < 1e-13 * abs(a).max()
    # SciPy's own HB writer uses different Fortran formats: the fixed-width parser must follow the format line
    path2 = str(tmp_path / "b.rua")
    scipy.io.hb_write(path2, a.tocsc())
    assert abs(a - _as_csr(*hostlib.read_matrix(path2))).max() < 1e-13 * abs(a).max()


def test_reference_binary_roundtrip(tmp_path):
    a = _rand(30, 0.1, 4).tocsc()
    a.sort_indices()
    path = str(tmp_path / "m.bin")
    hostlib.write_binary(path, 30, a.indptr, a.indices, a.data)
    nr, nc, ptr, ind, val = hostlib.read_matrix(path, layout="csc")
    assert nr == nc == 30 and np.array_equal(ptr, a.indptr) and np.array_equal(ind, a.indices) and np.array_equal(val, a.data)


@pytest.mark.parametrize("base", [0, 1])
@pytest.mark.parametrize("header", [True, False])
def test_triplet_files(tmp_path, base, header):
    """"m n nnz" + "row col value" lines (dreadtriple.c, suffix .dat) and the header-less form (dreadtriple_noheader.c,
    suffix .datnh: n = largest index); 0- or 1-based, detected from the smallest index."""
    a = _rand(40, 0.08, 3).tocoo()
    lines = [f"{r + base} {c + base} {v:.17e}" for r, c, v in zip(a.row, a.col, a.data)]
    if header:
        lines.insert(0, f"{a.shape[0]} {a.shape[1]} {a.nnz}")
    path = tmp_path / ("t.dat" if header else "t.datnh")
    path.write_text("\n".join(lines) + "\n")
    nr, nc, ptr, ind, val = hostlib.read_matrix(str(path))
    assert (nr, nc) == a.shape
    assert abs(_as_csr(nr, nc, ptr, ind, val) - a.tocsr()).max() == 0.0


def test_triplet_complex_and_errors(tmp_path):
    a = _rand(12, 0.2, 4, cx=True).tocoo()
    (tmp_path / "z.dat").write_text(f"12 12 {a.nnz}\n" + "".join(f"{r + 1} {c + 1} {v.real:.17e} {v.imag:.17e}\n" for r, c, v in zip(a.row, a.col, a.data)))
    nr, nc, ptr, ind, val = hostlib.read_matrix(str(tmp_path / "z.dat"))
    assert val.dtype == np.complex128 and abs(_as_csr(nr, nc, ptr, ind, val) - a.tocsr()).max() == 0.0
    (tmp_path / "short.dat").write_text("3 3 4\n1 1 2.0\n2 2 2.0\n")
    with pytest.raises(ValueError, match="fewer entries"):
        hostlib.read_matrix(str(tmp_path / "short.dat"))
    (tmp_path / "oob.dat").write_text("3 3 2\n1 1 2.0\n5 2 2.0\n")
    with pytest.raises(ValueError, match="out of range"):
        hostlib.read_matrix(str(tmp_path / "oob.dat"))


def test_rutherford_boeing(tmp_path):
    """The RB header (dreadrb.c): four counts on line 2, three formats on line 4, no right-hand-side line; symmetric
    storage (rsa) expanded."""
    # lower triangle of [[4,-1,0],[-1,4,-2],[0,-2,5]]
    text = ("a small symmetric matrix                                                 KEY     \n"
            "             4             1             1             2\n"
            "rsa                        3             3             5             0\n"
            "(4I6)           (5I6)           (3E22.14)           \n"
            "     1     3     5     6\n"
            "     1     2     2     3     3\n"
            "  4.00000000000000E+00 -1.00000000000000E+00  4.00000000000000E+00\n"
            " -2.00000000000000E+00  5.00000000000000E+00\n")
    (tmp_path / "s.rb").write_text(text)
    nr, nc, ptr, ind, val = hostlib.read_matrix(str(tmp_path / "s.rb"))
    assert np.array_equal(_as_csr(nr, nc, ptr, ind, val).toarray(), np.array([[4.0, -1, 0], [-1, 4, -2], [0, -2, 5]]))


def test_errors(tmp_path):
    with pytest.raises(ValueError):
        hostlib.read_matrix(str(tmp_path / "missing.rua"))
    (tmp_path / "bad.mtx").write_text("not a banner\n")
    with pytest.raises(ValueError):
        hostlib.read_matrix(str(tmp_path / "bad.mtx"))


@pytest.mark.parametrize("name", ["g4.rua", "g20.rua", "big.rua", "cg20.cua"])
def test_reference_fixtures(tmp_path, name):
    with gzip.open(os.path.join(GOLDEN, name + ".gz"), "rb") as f:
        (tmp_path / name).write_bytes(f.read())
    nr, nc, ptr, ind, val = hostlib.read_matrix(str(tmp_path / name))
    a = _as_csr(nr, nc, ptr, ind, val)
    expect = {"g4.rua": (16, 64), "g20.rua": (400, 1920), "big.rua": (4960, 23884), "cg20.cua": (400, 1920)}[name]
    assert (nr, a.nnz) == expect
    assert np.isfinite(val.view(np.float64)).all() and (a.diagonal() != 0).all()
    pat = (a != 0).astype(np.int8)
    assert (pat - pat.T).nnz == 0                      # all four fixtures have a symmetric pattern
    if name.endswith(".rua"):                          # write it back with our HB writer and read again: identical
        import tempfile
        with tempfile.TemporaryDirectory() as tmp:
            path = os.path.join(tmp, "again.rua")
            matgen.write_harwell_boeing(path, ptr, ind, val)
            b = _as_csr(*hostlib.read_matrix(path))
            assert abs(a - b).max() <= 1e-12 * abs(a).max()     # the writer prints 16 significant digits
    else:
        assert val.dtype == np.complex128
