#!/usr/bin/env python
"""bench.py -- pdgstrf3d factorization GFlop/s (FP64) of the B200-native path, with its roofline,
end-to-end (host buffers) figure and the reference's CPU path timed beside it.

    python bench.py [--gpus N --steps K --warmup W] [--grid G] [--impl reference] [--dump-outputs DIR]

One "step" = one numeric factorization (pdgstrf3d) of the 3D 7-point Poisson matrix on a G^3 grid
(BASELINE.json configs[1] shape; geometric nested dissection as MY_PERMC, NOROWPERM, no
equilibration, superlu_maxsup=256), FP64.  Flops are counted exactly as the reference counts
stat->ops[FACT] (pdgstrf2.c:578,590; trfAux.c:2303; sec_structs.c:692-693).
  value : sum over ranks of those flops / max over ranks of the device time of slu_b200_factor()
          (CUDA events on the library's stream), L/U already resident in HBM.
  e2e   : the same through the drop-in call pdgstrf3d_b200() with HOST buffers: handle creation (structure
          analysis, HBM allocation, index upload), H2D of the pinned host L/U arrays, factorization, D2H back
          into them, destruction -- host clock around the ONE C-ABI call a pdgstrf3d caller makes.
          (`e2e_handle`: the same on a pre-built handle, the reference's dCreateLUgpuHandle /
          pdgstrf3d_LUv1 / dCopyLUGPU2Host split, superlu_upacked.h:17-28.)
N > 1 (torchrun): 1 x 1 x N process grid -- Z-forests + NCCL ancestor reduction; same matrix, so
"scaling" is "strong".  Every line carries residual_probe = ||(LU - A) x|| / ||A x|| of the factors the
e2e call returned (N > 1: every rank applies the supernodes it finally owns, partial vectors all-reduced).
"""
import argparse
import json
import math
import os
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

METRIC = "pdgstrf3d_factor_gflops_fp64"
UNIT = "GFlop/s"
DUMP_SAMPLE = 3_000_000     # --dump-outputs: values per factor arena, so that the two float64 samples stay under 64 MB



def json_line(obj):
    """One strict JSON line: non-finite floats become null (json.dumps would print NaN, which is not JSON)."""
    def clean(x):
        if isinstance(x, float):
            return x if math.isfinite(x) else None
        if isinstance(x, dict):
            return {k: clean(v) for k, v in x.items()}
        if isinstance(x, (list, tuple)):
            return [clean(v) for v in x]
        return x
    return json.dumps(clean(obj), allow_nan=False)

def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default=os.environ.get("SLU_BENCH_WORKLOAD", "fem3"), choices=["poisson", "fem3"],
                    help="fem3: audikw_1-shaped 27-pt, 3 dof/node, G^3 nodes (BASELINE configs[2], default G=68: n=943,296, "
                         "nnz=74.2M); poisson: 7-pt Laplacian G^3 (configs[1] shape; 200^3 does not fit one B200, default G=128)")
    ap.add_argument("--grid", type=int, default=int(os.environ.get("SLU_BENCH_GRID", "0")))
    ap.add_argument("--cpu-grid", type=int, default=int(os.environ.get("SLU_BENCH_CPU_GRID", "0")))
    ap.add_argument("--maxsup", type=int, default=256)
    ap.add_argument("--relax", type=int, default=64)
    ap.add_argument("--leaf", type=int, default=64)
    ap.add_argument("--ordering", choices=["geometric", "graph"], default="geometric",
                    help="geometric: dissection of the grid by coordinates (default, the configuration every committed number uses); "
                         "graph: nested dissection of the sparsity pattern alone (host library, no geometry)")
    ap.add_argument("--amalg", type=float, default=0.05)
    ap.add_argument("--e2e-steps", type=int, default=2)
    ap.add_argument("--schur-variant", type=int, default=int(os.environ.get("SLU_SCHUR_VARIANT", "0")))
    ap.add_argument("--tc-slices", type=int, default=int(os.environ.get("SLU_BENCH_TC_SLICES", "0")),
                    help="tcgen05 path for wide supernodes: int8 slices per operand (0: library default, -1: off, 5..8)")
    ap.add_argument("--tc-min-ns", type=int, default=0, help="narrowest supernode on the tcgen05 path (0: library default)")
    ap.add_argument("--no-lookahead", type=int, default=0)
    ap.add_argument("--no-coop", type=int, default=0)
    ap.add_argument("--overlap-d2h", type=int, default=1, help="e2e through slu_b200_factor_host (download overlapped)")
    ap.add_argument("--overlap-h2d", type=int, default=0,
                    help="opt-in: level-by-level arena, factor_host also overlaps the upload (options.reserved[3])")
    ap.add_argument("--ref-mode", default=os.environ.get("SLU_BENCH_REF_MODE", "full"), choices=["sample", "full"],
                    help="--impl reference: full (default) = ONE factorization of the full-size workload (the like-for-like "
                         "number: 96 s on the 16 host cores of a B200 box, 142 s with its setup); sample = K + W steps on --cpu-grid")
    ap.add_argument("--device-fill", type=int, default=0,
                    help="1: distribute A on the device (slu_b200_fill_csr) instead of uploading host panels, check through "
                         "slu_b200_solve (no host copy of L/U at all: the mode of the largest runs); e2e is not measured")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--profile-phases", type=int, default=1)
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the L and U factors of the last one to DIR/*.npy (float64; a fixed, "
                         f"seeded sample of each arena larger than {DUMP_SAMPLE:,} values), to compare two builds")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.grid <= 0:
        a.grid = 68 if a.workload == "fem3" else 128
    if a.cpu_grid <= 0:
        a.cpu_grid = 36 if a.workload == "fem3" else 48
    return a


def make_matrix(args, g):
    """CSR matrix + nested-dissection permutation of the workload at grid size g."""
    from superlu_dist_b200 import hostlib
    if args.workload == "fem3":
        rp, ci, v = hostlib.fem3d(g, g, g, dof=3)
        geo = lambda: hostlib.nd_order(g, dof=3, leaf=max(1, args.leaf // 3))
    else:
        rp, ci, v = hostlib.poisson3d(g)
        geo = lambda: hostlib.nd_order(g, leaf=args.leaf)
    # --ordering graph: nested dissection of the pattern alone (sluh_nd_order_graph), as for a matrix read from a file
    return rp, ci, v, (hostlib.nd_order_graph(rp, ci, leaf=args.leaf) if args.ordering == "graph" else geo())


def bench_config(args):
    """The `config` object, identical in the b200 arm and the reference arm (same matrix, same symbolic knobs)."""
    return {"workload": workload_name(args.grid, args.workload, args.ordering), "ordering": ("geometric" if args.ordering == "geometric" else "graph") + " nested dissection as MY_PERMC, NOROWPERM, no equilibration",
            "maxsup": args.maxsup, "relax": args.relax,
            "l2": "inputs (L/U arena, GBs) larger than L2; arena re-uploaded between timed steps"}


def workload_name(g, kind="poisson", ordering="geometric"):
    if kind == "fem3":
        return f"audikw_1-shaped-27pt-3dof-{g}^3-nodes-fp64-{ordering}ND-maxsup256"
    return f"poisson3d-7pt-{g}^3-fp64-{ordering}ND-maxsup256"


# ---------------------------------------------------------------------------------------------
# reference arm / cpu_baseline: the UNMODIFIED reference CPU path (oracle/_ref, built by
# oracle/Makefile from /root/reference) on a bounded sample of the workload
# ---------------------------------------------------------------------------------------------
def host_threads():
    n = len(os.sched_getaffinity(0))
    try:
        q, p = open("/sys/fs/cgroup/cpu.max").read().split()
        if q != "max":
            n = min(n, max(1, int(int(q) / int(p))))
    except Exception:
        pass
    return n


def run_reference_once(args, grid, threads, tmp, plan=False):
    """One run of oracle/_ref/ref_driver (the unmodified reference's pdgssvx3d on the one-rank MPI stub).
    plan=True: the pdgstrf3d hook also prints slu_b200_plan's flop count for the reference's own symbolic structure
    (no device needed) -- returned under key "plan"."""
    from superlu_dist_b200 import matgen
    from superlu_dist_b200._paths import CUDA_SO
    drv = os.path.join(ROOT, "oracle", "_ref", "ref_driver")
    if not os.path.exists(drv):
        return None, "oracle/_ref/ref_driver is missing (build it where /root/reference exists: make -C oracle ref)"
    mat, pf = os.path.join(tmp, f"p{grid}.bin"), os.path.join(tmp, f"perm{grid}.bin")
    if not os.path.exists(mat):
        rp, ci, v, perm = make_matrix(args, grid)
        matgen.write_matrix_bin(mat, rp, ci, v)
        matgen.write_perm_bin(pf, perm)
    env = dict(os.environ, OMP_NUM_THREADS=str(threads), OPENBLAS_NUM_THREADS="1", SLU_B200_HOOK="plan" if plan else "ref",
               SLU_B200_LIB=CUDA_SO)
    out = subprocess.run([drv, mat, "--permc", pf, "--maxsup", str(args.maxsup), "--relax", str(args.relax)],
                         env=env, capture_output=True, text=True)
    res, planned = None, None
    for line in out.stdout.splitlines():
        if line.startswith('{"hook"'):
            planned = json.loads(line)
        elif line.startswith("{"):
            res = json.loads(line)
    if res is None:
        return None, "ref_driver failed: " + (out.stderr or out.stdout)[-300:]
    res["plan"] = planned
    return res, None


def flops_check(args, grid, r):
    """The flop numerator, three ways, for the matrix the reference just factored (SURVEY 8d: stat->ops[FACT]):
    the reference's own count, slu_b200_plan on the reference's symbolic structure, and the count of OUR host symbolic
    (the one bench.py's `value` uses).  The reference accumulates in float32 (flops_t), hence ~1e-4 of noise."""
    from superlu_dist_b200 import hostlib
    rp, ci, v, perm = make_matrix(args, grid)
    sym = hostlib.Symbolic(len(rp) - 1, rp, ci, perm, relax=args.relax, maxsup=args.maxsup, amalg=args.amalg)
    out = {"matrix": workload_name(grid, args.workload, args.ordering), "reference_stat_ops_fact": r["factor_flops"],
           "b200_plan_on_reference_structure": r["plan"]["b200_plan_ops_fact"] if r.get("plan") else None,
           "reference_nsupers": r["plan"]["nsupers"] if r.get("plan") else None,
           "b200_own_symbolic": float(sym.ops_fact), "b200_own_nsupers": int(sym.nsupers)}
    out["own_over_reference"] = round(out["b200_own_symbolic"] / out["reference_stat_ops_fact"], 6)
    return out


def cpu_baseline(args, tmp):
    threads = host_threads()
    r, err = run_reference_once(args, args.cpu_grid, threads, tmp, plan=True)
    if r is None:
        return {"value": None, "unit": UNIT, "cores": threads, "kind": "reference", "sample": err}
    try:
        fc = flops_check(args, args.cpu_grid, r)
    except Exception as exc:
        fc = {"error": str(exc)}
    return {"value": round(r["factor_gflops"], 3), "unit": UNIT, "cores": threads, "kind": "reference",
            "sample": f"{workload_name(args.cpu_grid, args.workload, args.ordering)} (bounded sample of the workload: {r['factor_flops']:.3e} flops, "
                      f"factor {r['factor_s']:.2f} s; unmodified reference pdgstrf3d CPU path, 1x1x1, OpenMP {threads} threads, "
                      f"scipy-OpenBLAS 1 thread/call, one-rank MPI stub)",
            "flops_check": fc,
            "scaling_note": "the reference's intra-rank OpenMP covers only the GEMM+scatter loop; diagonal LU (-O0), the owner-branch "
                            "L-panel TRSM and the gather are serial: 1/2/4-thread runs fit a serial fraction of ~0.25 "
                            "(profiles/r02_notes.md), so 16 and 96 threads give the same ~150 GFlop/s"}


def main_reference(args):
    """The reference arm: the UNMODIFIED reference pdgstrf3d (CPU path, oracle/_ref) on the box's host cores, same
    metric / unit / config as the b200 arm.  --ref-mode full (default): ONE factorization of the full-size matrix
    (~2.5 minutes with its symbolic phase on a B200 box; steps_run says 1) -- the like-for-like number: CPU supernodal
    LU gets more efficient with size (356 GFlop/s at 68^3 against 147 on the 36^3 sample, profiles/r02_*).
    --ref-mode sample: every step factors the bounded sample (--cpu-grid), K + W steps."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    full = args.ref_mode == "full"
    grid = args.grid if full else args.cpu_grid
    nrun = 1 if full else args.warmup + args.steps
    with tempfile.TemporaryDirectory() as tmp:
        threads = host_threads()
        times, last = [], None
        for i in range(nrun):
            r, err = run_reference_once(args, grid, threads, tmp, plan=full)
            if r is None:
                print(json.dumps({"impl": "reference", "unavailable": err}))
                return
            if full or i >= args.warmup:
                times.append(r["factor_s"])
            last = r
        t = float(np.mean(times))
        val = last["factor_flops"] / t * 1e-9
        sample = (f"{workload_name(grid, args.workload, args.ordering)}: the full-size workload, ONE factorization (no warm-up)" if full else
                  f"{workload_name(grid, args.workload, args.ordering)}: bounded sample of {workload_name(args.grid, args.workload, args.ordering)} "
                  f"({last['factor_flops']:.3e} flops per step)")
        cb = {"value": round(val, 3), "unit": UNIT, "cores": threads, "kind": "reference", "sample": sample,
              "how": "unmodified reference pdgstrf3d CPU path, 1x1x1, OpenMP, scipy-OpenBLAS 1 thread/call, one-rank MPI stub"}
        print(json.dumps({"impl": "reference", "metric": METRIC, "value": round(val, 3), "unit": UNIT,
                          "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "steps_run": len(times),
                          "ms_per_step": round(t * 1e3, 3), "higher_is_better": True, "scaling": "strong",
                          "vs_baseline": None, "dtype": "f64", "data": "synthetic",
                          "config": bench_config(args),
                          "problem": {"n": last["n"], "factor_flops": last["factor_flops"], "grid": "1x1x1", "threads": threads,
                                      "total_s": last["total_s"]},
                          "cpu_baseline": cb, "flops_check": flops_check(args, grid, last) if full else None,
                          "e2e": {"value": round(val, 3), "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                          "gpu_launches": 0}))


# ---------------------------------------------------------------------------------------------
class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md)."""

    def __init__(self, index):
        self.rows, self.proc, self.index = [], None, index

    def start(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm = [float(r[0]) for r in self.rows if r and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(len(r) > 3 + i and r[3 + i].lower().startswith("active") for r in self.rows)]
        pw = [float(r[2]) for r in self.rows if len(r) > 2 and r[2].replace(".", "").isdigit()]
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "power_w_max": max(pw) if pw else None, "samples": len(sm)}


def per_update_roofline_ms(prob, peak_tflops, hbm_gbs):
    """SURVEY 8(d): lower bound of the Schur phase, sum over supernodes of max(2mnk / P64, bytes / BW) with
    bytes = 8(mk + kn) + 16mn + 4(m+n); also returns the flop share of the compute-bound updates."""
    ns = np.diff(prob.xsup).astype(np.float64)
    nsupr = prob.lidx[prob.lidx_off[:-1] + 1].astype(np.float64)
    m = nsupr - ns
    n = np.where(ns > 0, prob.uval_len / np.maximum(ns, 1), 0.0)
    fl = 2.0 * m * n * ns
    by = 8.0 * (m * ns + ns * n) + 16.0 * m * n + 4.0 * (m + n)
    t_c, t_m = fl / (peak_tflops * 1e12), by / (hbm_gbs * 1e9)
    bound = np.maximum(t_c, t_m)
    return float(bound.sum() * 1e3), float(fl[t_c >= t_m].sum() / max(fl.sum(), 1.0))


def dgemm_peak_tflops(torch, m=8192, n=8192, k=256, reps=10):
    """cuBLAS FP64 GEMM at a Schur-update shape: the roofline denominator for the DMMA kernel
    (MEASURED_PEAKS.json carries only bf16 and HBM figures; FP64 has its own pipe rate)."""
    a = torch.randn(m, k, dtype=torch.float64, device="cuda")
    b = torch.randn(k, n, dtype=torch.float64, device="cuda")
    c = torch.zeros(m, n, dtype=torch.float64, device="cuda")
    for _ in range(3):
        torch.addmm(c, a, b, alpha=-1.0, out=c)
    best = 1e30
    for _ in range(3):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record()
        for _ in range(reps):
            torch.addmm(c, a, b, alpha=-1.0, out=c)
        e1.record()
        torch.cuda.synchronize()
        best = min(best, e0.elapsed_time(e1) / reps)
    del a, b, c
    torch.cuda.empty_cache()
    return 2.0 * m * n * k / best * 1e-9


def dump_outputs(path, layer, suffix=""):
    """The factors a caller of the timed path receives (L and U arenas of one layer) as float64 .npy files.  Arenas
    larger than DUMP_SAMPLE are sampled at sorted positions drawn from a fixed seed, so that the same arguments select
    the same entries in every run and two builds can be compared entry for entry."""
    os.makedirs(path, exist_ok=True)
    rng = np.random.default_rng(0)
    for name, arena in (("L", layer.lval), ("U", layer.uval)):
        pos = np.sort(rng.choice(arena.size, DUMP_SAMPLE, replace=False)) if arena.size > DUMP_SAMPLE else slice(None)
        np.save(os.path.join(path, f"{name}{suffix}.npy"), np.asarray(arena[pos], np.float64))


def main():
    args = parse()
    if args.impl == "reference":
        return main_reference(args)
    # keep stdout clean for the ONE JSON line (NCCL / torchrun banners go to stderr)
    saved_stdout = os.dup(1)
    os.dup2(2, 1)

    import torch
    import torch.distributed as dist
    from superlu_dist_b200 import LUProblem, capi, hostlib

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        if world == 1 and args.gpus > 1:
            raise SystemExit("launch with torchrun for --gpus > 1")
    capi.require_gpu()
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()

    def allmax(x):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def allsum(x):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        return float(t.item())

    # ---- the workload, in the reference's data layout (host side; not timed) -------------------
    t0 = time.time()
    G = args.grid
    rp, ci, v, perm = make_matrix(args, G)
    sym = hostlib.Symbolic(len(rp) - 1, rp, ci, perm, relax=args.relax, maxsup=args.maxsup, amalg=args.amalg)
    prob = LUProblem.from_symbolic(sym, npdep=world)
    del sym
    if args.device_fill:
        lay = prob.add_layer(rank)       # untouched (lazily zero) arrays: only their addresses enter the view
    else:
        lay = prob.add_layer(rank, alloc=capi.pinned_alloc)
        prob.fill_layer(rank, rp, ci, v)
    t_setup = time.time() - t0
    h2d = int(8 * (lay.lval_off[-1] + lay.uval_off[-1]))

    def fresh_id():
        if world == 1:
            return None
        box = [capi.nccl_unique_id() if rank == 0 else None]
        dist.broadcast_object_list(box, src=0)
        return box[0]

    def allsum_vec(x):
        if world == 1:
            return x
        t = torch.from_numpy(np.ascontiguousarray(x)).cuda()
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        return t.cpu().numpy()

    # one NCCL id for the whole run: the library caches the communicators built from it (as the reference's MPI
    # communicators outlive pdgstrf3d), so neither the handles below nor the e2e calls re-create them
    nccl_id = fresh_id()
    common = dict(device=local, world_size=world, world_rank=rank, nccl_id=nccl_id, pinned=1,
                  schur_variant=args.schur_variant, no_lookahead=args.no_lookahead, no_coop=args.no_coop,
                  tc_slices=args.tc_slices, tc_min_ns=args.tc_min_ns)
    h = capi.Handle(prob, rank, overlap_h2d=args.overlap_h2d, **common)
    t_create_first = h.stats().t_analyze_s          # includes the one-time NCCL communicator creation at N > 1

    def one_step():
        if args.device_fill:
            h.fill_csr(rp, ci, v, prob.perm)   # reset HBM to the unfactored matrix (outside the timed region)
        else:
            h.upload()
        barrier()
        info = h.factor()               # device-timed inside the library (CUDA events on its stream)
        barrier()
        assert info == 0, info
        return h.stats().t_factor_s

    for _ in range(args.warmup):
        one_step()
    sampler = ClockSampler(local)
    sampler.start()
    step_s = [allmax(one_step()) for _ in range(args.steps)]
    clocks = sampler.stop()
    if args.dump_outputs:
        h.download()                     # the factors of the last timed step, into the host arrays (refilled below)
        dump_outputs(args.dump_outputs, lay, f"_rank{rank}" if world > 1 else "")
    st = h.stats()
    total_ops = allsum(st.ops_fact)
    t_step = float(np.mean(step_s))
    value = total_ops / t_step * 1e-9

    # ---- e2e on the pre-built handle (the reference's handle API split): H2D + factor + D2H ---------------
    def timed_host_calls(call, steps):
        out = []
        for i in range(steps + 1):
            prob.fill_layer(rank, rp, ci, v)         # restore the host arrays (not timed)
            barrier()
            t1 = time.perf_counter()
            info, extra = call()
            torch.cuda.synchronize()
            dt = time.perf_counter() - t1
            assert info == 0, info
            if i > 0:                                # first pass is the warm-up
                out.append((allmax(dt), extra))
        return out

    def handle_call():
        if args.overlap_d2h:
            return h.factor_host(), None
        h.upload()
        info = h.factor()
        h.download()
        return info, None

    solve_check = None
    if args.device_fill:
        # correctness without any host copy of the factors: solve A x = b on the resident factors for a known x
        import scipy.sparse as sp
        A = sp.csr_matrix((v, ci, rp), shape=(prob.n, prob.n))
        pm = np.asarray(prob.perm)
        xt_perm = np.where(np.arange(prob.n) % 2 == 0, 1.0, -1.0)       # the reference's xtrue pattern (dutil_dist.c:598)
        b_perm = np.empty(prob.n)
        b_perm[pm] = A @ xt_perm[pm]
        t1 = time.perf_counter()
        xs = h.solve(b_perm)
        t_solve = time.perf_counter() - t1
        r_old = A @ xs[pm] - b_perm[pm]
        solve_check = {"solve_error_inf": float(np.abs(xs - xt_perm).max()), "residual_Ax_b_over_b": float(np.linalg.norm(r_old) / np.linalg.norm(b_perm)),
                       "solve_s": round(allmax(t_solve), 4), "what": "slu_b200_solve on the HBM-resident factors, x = +-1"}
        assert solve_check["residual_Ax_b_over_b"] < 1e-10, solve_check
        args.e2e_steps = 0
    eh = timed_host_calls(handle_call, args.e2e_steps) if args.e2e_steps > 0 else []
    eh_mean = float(np.mean([t for t, _ in eh])) if eh else None
    e2e_handle = {"value": round(total_ops / eh_mean * 1e-9, 2) if eh_mean else None, "unit": UNIT,
                  "ms_per_step": round(eh_mean * 1e3, 2) if eh_mean else None, "steps": len(eh),
                  "call": "slu_b200_factor_host on a pre-built handle (create/destroy outside)"}
    h.close()                            # one L/U arena at a time: two would not fit HBM at the large sizes

    # ---- e2e through the drop-in call: pdgstrf3d_b200 = create + H2D + factor + D2H + destroy ---------------
    def dropin_call():
        info, s1 = capi.pdgstrf3d(prob, rank, pipeline=args.overlap_d2h, overlap_h2d=args.overlap_h2d, **common)
        return info, s1

    ed = timed_host_calls(dropin_call, args.e2e_steps) if args.e2e_steps > 0 else []
    e2e_mean = float(np.mean([t for t, _ in ed])) if ed else None      # --e2e-steps 0: not measured (null, never NaN)
    last = ed[-1][1] if ed else None
    e2e = {"value": round(total_ops / e2e_mean * 1e-9, 2) if e2e_mean else None, "unit": UNIT,
           "h2d_bytes_per_step": int(allsum(float(h2d))), "d2h_bytes_per_step": int(allsum(float(h2d))), "steps": len(ed),
           "ms_per_step": round(e2e_mean * 1e3, 2) if e2e_mean else None,
           "t_analyze_s": round(allmax(last.t_analyze_s), 4) if last else None,
           "t_factor_s": round(allmax(last.t_factor_s), 4) if last else None,
           "t_upload_s": round(allmax(last.t_upload_s), 4) if last else None,
           "t_create_first_call_s": round(allmax(t_create_first), 4),
           "call": "pdgstrf3d_b200 (create + H2D + factor + D2H + destroy; " +
                   ("H2D and D2H overlapped with the factorization)" if args.overlap_h2d and args.overlap_d2h else
                    "D2H overlapped with the factorization)" if args.overlap_d2h else "no overlap)")}

    # ---- the same job without ever moving factors over PCIe (rows N1 + N2): CSR in, solution out -------------------
    # create + slu_b200_fill_csr (12 B per nonzero H2D, scatter on the device) + factor + slu_b200_solve + destroy
    e2e_csr = None
    if args.e2e_steps > 0 and not args.device_fill:
        import scipy.sparse as sp
        A = sp.csr_matrix((v, ci, rp), shape=(prob.n, prob.n))
        pm = np.asarray(prob.perm)
        xt_perm = np.where(np.arange(prob.n) % 2 == 0, 1.0, -1.0)
        b_perm = np.empty(prob.n)
        b_perm[pm] = A @ xt_perm[pm]
        ts, err_x = [], None
        for i in range(args.e2e_steps + 1):
            barrier()
            t1 = time.perf_counter()
            hc = capi.Handle(prob, rank, **common)
            hc.fill_csr(rp, ci, v, prob.perm)
            info = hc.factor()
            xs = hc.solve(b_perm)
            hc.close()
            dt = time.perf_counter() - t1
            assert info == 0, info
            if i > 0:
                ts.append(allmax(dt))
            err_x = float(np.abs(xs - xt_perm).max())
        assert err_x < 1e-8, err_x
        tm = float(np.mean(ts))
        e2e_csr = {"value": round(total_ops / tm * 1e-9, 2), "unit": UNIT, "ms_per_step": round(tm * 1e3, 2), "steps": len(ts),
                   "h2d_bytes_per_step": int(12 * len(v) + 4 * (2 * prob.n + 1) + 8 * prob.n), "d2h_bytes_per_step": int(8 * prob.n),
                   "solve_error_inf": err_x,
                   "call": "slu_b200_create + slu_b200_fill_csr (device-side distribution) + slu_b200_factor + slu_b200_solve + "
                           "slu_b200_destroy: host CSR matrix in, solution out, the factors never cross PCIe"}

    # ---- correctness of what was timed: ||(LU - A) x|| / ||A x|| with +-1 probes, at every N ----------------
    # The host arrays hold the factors the last e2e call returned.  N > 1: each rank applies only the supernodes it
    # finally owns (the layer that factored them, SURVEY 8b) -- t = U x and y = L t are summed over the ranks.
    resid = None
    if ed or eh:
        if not ed:                       # --e2e-steps 0 is handled above; eh without ed cannot happen
            pass
        rng = np.random.default_rng(0)
        x = rng.choice([-1.0, 1.0], size=(2, prob.n))
        mine = prob.final_owner_masks()[rank]
        tvec = allsum_vec(prob.matvec([(lay, mine)], x, 2))
        yl = allsum_vec(prob.matvec([(lay, mine)], tvec, 3))
        prob.fill_layer(rank, rp, ci, v)
        ya = allsum_vec(prob.matvec([(lay, mine)], x, 0))
        resid = float(np.linalg.norm(yl - ya) / np.linalg.norm(ya))
        assert resid < 1e-10, f"residual probe {resid} exceeds 1e-10"

    # ---- roofline of the dominant kernel (fused Schur GEMM+scatter) and the phase split, measured live ------
    roof = None
    if args.profile_phases:
        hp = capi.Handle(prob, rank, verbose=2, **common)     # verbose 2: single stream, events around every phase
        if args.device_fill:
            hp.fill_csr(rp, ci, v, prob.perm)
        else:
            hp.upload()
        barrier()
        hp.factor()
        barrier()
        sp = hp.stats()
        hp.close()
        phase = {"diag_lu": round(allmax(sp.t_diag_ms), 3), "panel_trsm": round(allmax(sp.t_trsm_ms), 3),
                 "schur_setup": round(allmax(sp.t_schur_setup_ms), 3), "schur": round(allmax(sp.t_schur_ms), 3),
                 "ancestor_reduce": round(allmax(sp.t_reduce_ms), 3),
                 "profiled_step_ms": round(allmax(sp.t_factor_s) * 1e3, 3),
                 "note": "max over ranks of each phase, single-stream profiling run (no look-ahead overlap)"}
        t_schur = allmax(sp.t_schur_ms)
        ops_schur = allsum(sp.ops_schur)
        schur_bytes = allsum(sp.schur_bytes)
        peak = dgemm_peak_tflops(torch)
        ach = ops_schur / world / (t_schur * 1e-3) * 1e-12      # per GPU
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        hbm_peak = peaks.get("hbm_gbs", 6650.0)
        try:
            roof_ms, cshare = per_update_roofline_ms(prob, peak, hbm_peak)
        except Exception as exc:      # an accounting extra must never cost the bench line
            print(f"per-update roofline skipped: {exc}", file=sys.stderr)
            roof_ms, cshare = float("nan"), float("nan")
        traffic = None
        for name in ("r02_schur_traffic.json", "r01_schur_traffic.json"):
            try:   # dram__bytes_read.sum + dram__bytes_write.sum of ONE profiled launch (ncu --set full), committed
                traffic = json.load(open(os.path.join(ROOT, "profiles", name)))
                break
            except Exception:
                pass
        S_tc = int(sp.reserved[3])
        tc_share = allsum(sp.reserved[1]) / max(ops_schur, 1.0)
        bf16_peak = peaks.get("bf16_tflops_sustained") or peaks.get("bf16_tflops") or 1590.0
        tc_extra = None
        if S_tc > 0:
            # executed int8 work of the tcgen05 kernel: S(S+1)/2 int8 products per FP64 product; the int8 pipe runs at twice
            # the bf16 rate (B200_PROFILING.md: 4.5 vs 2.25 PFLOP/s nominal), so its measured peak = 2 x MEASURED_PEAKS bf16
            prod = S_tc * (S_tc + 1) // 2
            tc_extra = {"slices": S_tc, "schur_flop_share": round(tc_share, 4), "int8_products_per_fp64_product": prod,
                        "int8_tops_executed": round(ach * tc_share * prod, 1),
                        "int8_peak_tops": round(2 * bf16_peak, 1), "int8_frac": round(ach * tc_share * prod / (2 * bf16_peak), 4),
                        "int8_peak_source": "2 x bf16 sustained GEMM of MEASURED_PEAKS.json (int8 pipe = 2 x bf16 pipe)" if peaks else "fallback",
                        "slice_workspace_bytes_rank0": int(sp.reserved[2]),
                        "note": "frac above is FP64-equivalent TF/s over the cuBLAS FP64 GEMM rate: > 1 means faster than the FP64 pipe"}
        roof = {"bound": "tensor",
                "kernel": ("schur_kernel_tc (tcgen05.mma.kind::i8 on int8 slices, TMEM accumulators, bulk-copy staged tiles, fused scatter) + "
                           "schur_kernel (DMMA) for supernodes < 128 columns") if S_tc > 0 else "schur_kernel (DMMA m8n8k4 GEMM + fused scatter)",
                "achieved": round(ach, 3), "peak": round(peak, 3), "unit": "TFLOP/s", "frac": round(ach / peak, 4),
                "peak_source": "cuBLAS FP64 GEMM 8192x8192x256 measured live on this GPU (FP64 pipe; MEASURED_PEAKS.json has bf16/HBM only)",
                "traffic": traffic.get("dram_bytes_read", 0) + traffic.get("dram_bytes_write", 0) if traffic else None,
                "traffic_capture": ({k: traffic[k] for k in ("kernel", "tiles", "duration_ms", "algorithmic_bytes_scatter", "capture") if k in traffic}
                                    if traffic else None),
                "hbm_achieved_gbs": round(schur_bytes / world / (t_schur * 1e-3) * 1e-9, 1),
                "hbm_peak_gbs": hbm_peak, "hbm_peak_source": "MEASURED_PEAKS.json" if peaks else "fallback",
                "kernel_ms": round(t_schur, 3), "kernel_share_of_step": round(t_schur * 1e-3 / allmax(sp.t_factor_s), 4),
                "per_update_roofline_ms": round(roof_ms / world, 3),
                "frac_of_per_update_roofline": round(roof_ms / world / t_schur, 4),
                "compute_bound_flop_share": round(cshare, 4), "phase_ms": phase,
                "tcgen05": tc_extra}

    cb = None
    if world == 1 and not args.no_cpu_baseline:   # the CPU baseline is timed at N = 1 only
        with tempfile.TemporaryDirectory() as tmp:
            cb = cpu_baseline(args, tmp)

    sys.stdout.flush()
    try:                                 # NCCL prints its version banner through C stdio: flush it to stderr too
        import ctypes
        ctypes.CDLL(None).fflush(None)
    except Exception:
        pass
    os.dup2(saved_stdout, 1)
    if rank == 0:
        print(json_line({
            "metric": METRIC, "value": round(value, 2), "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": round(t_step * 1e3, 3), "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": bench_config(args),
            "problem": {"n": prob.n, "nsupers": prob.nsupers, "grid": f"1x1x{world}", "factor_flops": total_ops,
                        "lu_bytes_rank0": h2d, "amalg": args.amalg, "host_setup_s": round(t_setup, 1),
                        "note": "BASELINE configs[1] (Poisson 200^3, ~280 GB of L+U) does not fit one 180 GB B200; it runs "
                                "on 1x1x8 (profiles/r02_*); scaled single-GPU instances: --workload poisson --grid 128|160"},
            "clocks": clocks, "e2e": e2e, "e2e_handle": e2e_handle, "e2e_csr_to_solution": e2e_csr, "gpu_launches": int(st.gpu_launches), "nlevels": int(st.nlevels),
            "residual_probe": resid if resid is not None else (solve_check or {}).get("residual_Ax_b_over_b"),
            "solve_check": solve_check, "roofline": roof, "cpu_baseline": cb}))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
