"""Kernel variants and the doublecomplex path (pzgstrf3d_b200, SURVEY 8a row a15): gating.

Round 1 wrote these pieces after its GPU minutes were spent and kept them xfail(strict=False); all seven XPASSED on
the driver's B200 (GPUTEST_r01.json), so they gate now.  Each group still runs in a child process
(tests/optin_worker.py): several of them select a kernel through an environment variable that the library reads once
per process."""
import os
import subprocess
import sys

import pytest

from test_dropin import ZDRV

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))


def _run(what):
    r = subprocess.run([sys.executable, os.path.join(HERE, "optin_worker.py"), what], capture_output=True, text=True,
                       timeout=420)
    assert r.returncode == 0, (r.stdout[-2000:], r.stderr[-4000:])


def test_optin_gemm_tile_v2():
    _run("gemm")


def test_optin_schur_variant_4_5():
    _run("factor")


def test_optin_complex_kernels():
    _run("zkernels")


def test_optin_pzgstrf3d():
    _run("zfactor")


def test_optin_diag_lu_v3():
    _run("diagv3")


def test_trsm_right_looking():
    _run("trsmrl")


def test_diag_lu_cluster():
    _run("diagcluster")


@pytest.mark.skipif(not os.path.exists(ZDRV), reason="oracle/_ref/pzdrive3d (the reference's own driver) not built")
def test_optin_pzdrive3d_dropin():
    _run("zdropin")


def test_optin_overlapped_upload():
    _run("h2d")
