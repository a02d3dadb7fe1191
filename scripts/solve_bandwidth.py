"""Bandwidth of the resident-factor solve (slu_b200_solve / slu_b200_z_solve) in both precisions.

One structure -- default: 7-point Poisson G^3, G = 64, geometric nested dissection, maxsup 256, about 3 GB of double
factors in HBM, far beyond the 126 MB L2 of a B200, so every solve streams L and U from HBM -- is distributed on the
device (slu_b200_fill_csr), factored in double and in doublecomplex, and solved with nrhs = 1 and 8.  One JSON line per
(precision, nrhs):
  seconds      host clock around the synchronising solve call (H2D of b and D2H of x included, as stats.reserved[4])
  bytes        (nnz_l + nnz_u) * sizeof(element) * nrhs: the factor entries one solve streams
  gb_s         bytes / seconds, and its fraction of the 7.7 TB/s HBM3e data-sheet figure of one B200
The card's name and power limit are read in the same run and printed on the first line.
    python scripts/solve_bandwidth.py [--grid 64] [--steps 10] [--warmup 3] [--device 0]"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import scipy.sparse as sp

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from superlu_dist_b200 import LUProblem, capi, hostlib  # noqa: E402

HBM_TBS = 7.7


def card(device):
    try:
        out = subprocess.run(["nvidia-smi", "-i", str(device), "--query-gpu=name,power.limit,clocks.max.sm",
                              "--format=csv,noheader"], capture_output=True, text=True, timeout=60)
        name, power, sm = [f.strip() for f in out.stdout.strip().split(",")]
        return {"card": name, "power_limit": power, "sm_max_clock": sm}
    except Exception as e:   # the measurement still stands; say that the card could not be read
        return {"card": None, "power_limit": None, "error": f"nvidia-smi: {e}"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--grid", type=int, default=64)
    ap.add_argument("--leaf", type=int, default=64)
    ap.add_argument("--relax", type=int, default=64)
    ap.add_argument("--maxsup", type=int, default=256)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--device", type=int, default=0)
    args = ap.parse_args()
    capi.require_gpu()

    G = args.grid
    rp, ci, v = hostlib.poisson3d(G)
    perm = hostlib.nd_order(G, leaf=args.leaf)
    n = len(rp) - 1
    sym = hostlib.Symbolic(n, rp, ci, perm, relax=args.relax, maxsup=args.maxsup, amalg=0.05)
    # doublecomplex values on the same pattern: i * (random off-diagonal perturbation), still diagonally dominant
    rows = np.repeat(np.arange(n), np.diff(rp))
    vi = np.where(rows == ci, 0.25, 0.5 * np.random.default_rng(0).uniform(-1.0, 1.0, len(v)))
    head = {"workload": f"poisson3d-7pt-{G}^3-geometricND-maxsup{args.maxsup}", "n": n, "nnz_a": len(v),
            "steps": args.steps, "warmup": args.warmup, "hbm_datasheet_tb_s": HBM_TBS}
    head.update(card(args.device))
    print(json.dumps(head), flush=True)

    for prec, dt, val in (("double", np.float64, v), ("doublecomplex", np.complex128, v + 1j * vi)):
        prob = LUProblem.from_symbolic(sym)
        prob.dtype = np.dtype(dt)
        prob.add_layer(0)                         # never read: the values are distributed on the device
        planned = capi.plan(prob)
        h = capi.Handle(prob, 0, device=args.device)
        h.fill_csr(rp, ci, val, perm)
        assert h.factor() == 0
        st = h.stats()
        elem = np.dtype(dt).itemsize
        a = sp.csr_matrix((np.asarray(val, dt), (perm[rows], perm[ci])), shape=(n, n))   # P A P^T, perm[old] = new
        for nrhs in (1, 8):
            rng = np.random.default_rng(nrhs)
            xtrue = rng.standard_normal((nrhs, n)).astype(dt)
            if dt == np.complex128:
                xtrue = xtrue + 1j * rng.standard_normal((nrhs, n))
            b = (a @ xtrue.T).T
            for _ in range(args.warmup):
                x = h.solve(b)
            secs, lib_secs = [], []
            for _ in range(args.steps):
                t0 = time.perf_counter()
                x = h.solve(b)
                secs.append(time.perf_counter() - t0)
                lib_secs.append(h.stats().reserved[4])
            err = float(np.abs(x - xtrue).max() / np.abs(xtrue).max())
            nbytes = (st.nnz_l + st.nnz_u) * elem * nrhs
            med = float(np.median(secs))
            print(json.dumps({"precision": prec, "nrhs": nrhs, "seconds_median": med, "seconds_min": float(min(secs)),
                              "seconds_max": float(max(secs)), "reserved4_median": float(np.median(lib_secs)),
                              "launches": int(h.stats().reserved[5]), "nnz_l": st.nnz_l, "nnz_u": st.nnz_u,
                              "lu_device_bytes": st.lu_device_bytes, "planned_lu_device_bytes": planned.lu_device_bytes,
                              "bytes": nbytes, "gb_s": nbytes / med / 1e9,
                              "fraction_of_hbm": nbytes / med / (HBM_TBS * 1e12), "fwd_err": err}), flush=True)
        h.close()
        del prob


if __name__ == "__main__":
    main()
