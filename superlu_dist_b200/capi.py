"""ctypes binding of lib/libslu_b200.so (include/slu_b200.h) -- the product's C-ABI.

There is no CPU fallback: if the shared library is missing, or no CUDA device is visible when a
compute entry point is called, this module raises.
"""
import ctypes as C
import os
import re

import numpy as np

from ._paths import CUDA_SO, INCLUDE
from .problem import my_tree_idxs, my_zero_tr_idxs

_lib = None
i32 = C.c_int32


class Forest(C.Structure):
    _fields_ = [("nNodes", i32), ("nodeList", C.c_void_p), ("numLvl", i32), ("eTreeTopLims", C.c_void_p)]


class LUView(C.Structure):
    _fields_ = [("n", i32), ("nsupers", i32), ("xsup", C.c_void_p),
                ("nprow", i32), ("npcol", i32), ("npdep", i32), ("myrow", i32), ("mycol", i32), ("mydep", i32),
                ("Lrowind_bc_ptr", C.c_void_p), ("Lnzval_bc_ptr", C.c_void_p),
                ("Ufstnz_br_ptr", C.c_void_p), ("Unzval_br_ptr", C.c_void_p),
                ("maxLvl", i32), ("myTreeIdxs", C.c_void_p), ("myZeroTrIdxs", C.c_void_p),
                ("nforests", i32), ("forests", C.c_void_p)]


class Options(C.Structure):
    _fields_ = [("device", i32), ("replace_tiny_pivot", i32), ("thresh", C.c_double), ("verbose", i32),
                ("pinned_host", i32), ("world_size", i32), ("world_rank", i32),
                ("nccl_id", C.c_ubyte * 128), ("schur_variant", i32), ("reserved", i32 * 7)]


class Stats(C.Structure):
    _fields_ = [("ops_fact", C.c_double), ("ops_schur", C.c_double), ("schur_bytes", C.c_double),
                ("tiny_pivots", C.c_int64), ("gpu_launches", C.c_int64),
                ("t_analyze_s", C.c_double), ("t_upload_s", C.c_double), ("t_factor_s", C.c_double),
                ("t_download_s", C.c_double), ("t_diag_ms", C.c_double), ("t_trsm_ms", C.c_double),
                ("t_schur_setup_ms", C.c_double), ("t_schur_ms", C.c_double), ("t_reduce_ms", C.c_double),
                ("lu_device_bytes", C.c_int64), ("index_device_bytes", C.c_int64),
                ("nnz_l", C.c_int64), ("nnz_u", C.c_int64), ("nlevels", i32), ("my_supernodes", i32),
                ("reserved", C.c_double * 8)]

    def as_dict(self):
        return {k: getattr(self, k) for k, _ in self._fields_ if k != "reserved"}


def declared_symbols():
    """Every function declared in include/slu_b200.h."""
    text = open(os.path.join(INCLUDE, "slu_b200.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b((?:slu_b200_|pdgstrf3d_b200|pzgstrf3d_b200)\w*)\s*\(", text)))


def lib():
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(CUDA_SO):
        raise RuntimeError(f"{CUDA_SO} is missing: the CUDA extension was not built "
                           "(python -c 'import __graft_entry__ as g; g.build()'); there is no CPU fallback")
    L = C.CDLL(CUDA_SO)
    for s in declared_symbols():
        if not hasattr(L, s):
            raise RuntimeError(f"libslu_b200.so does not export {s}")
    sizes = (i32 * 4)()
    L.slu_b200_struct_sizes(sizes)
    mine = [C.sizeof(Forest), C.sizeof(LUView), C.sizeof(Options), C.sizeof(Stats)]
    if list(sizes) != mine:
        raise RuntimeError(f"ctypes struct mirrors are out of date: library {list(sizes)} vs python {mine}")
    L.slu_b200_last_error.restype = C.c_char_p
    L.slu_b200_host_alloc.restype = C.c_void_p
    L.slu_b200_host_alloc.argtypes = [C.c_size_t]
    L.slu_b200_host_free.argtypes = [C.c_void_p]
    L.slu_b200_create.argtypes = [C.POINTER(C.c_void_p), C.POINTER(LUView), C.POINTER(Options)]
    for f in ("slu_b200_upload", "slu_b200_download"):
        getattr(L, f).argtypes = [C.c_void_p]
    L.slu_b200_factor.argtypes = [C.c_void_p, C.POINTER(C.c_int)]
    L.slu_b200_factor_host.argtypes = [C.c_void_p, C.POINTER(C.c_int)]
    L.slu_b200_get_stats.argtypes = [C.c_void_p, C.POINTER(Stats)]
    L.slu_b200_solve.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int]
    L.slu_b200_fill_csr.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    L.slu_b200_destroy.argtypes = [C.c_void_p]
    L.slu_b200_destroy.restype = None
    L.pdgstrf3d_b200.argtypes = [C.POINTER(LUView), C.POINTER(Options), C.POINTER(Stats), C.POINTER(C.c_int)]
    L.slu_b200_plan.argtypes = [C.POINTER(LUView), C.POINTER(Options), C.POINTER(Stats)]
    L.slu_b200_z_plan.argtypes = [C.POINTER(LUView), C.POINTER(Options), C.POINTER(Stats)]
    # doublecomplex twins (same structs; value arrays hold (re, im) pairs)
    L.slu_b200_z_create.argtypes = [C.POINTER(C.c_void_p), C.POINTER(LUView), C.POINTER(Options)]
    for f in ("slu_b200_z_upload", "slu_b200_z_download"):
        getattr(L, f).argtypes = [C.c_void_p]
    L.slu_b200_z_factor.argtypes = [C.c_void_p, C.POINTER(C.c_int)]
    L.slu_b200_z_factor_host.argtypes = [C.c_void_p, C.POINTER(C.c_int)]
    L.slu_b200_z_get_stats.argtypes = [C.c_void_p, C.POINTER(Stats)]
    L.slu_b200_z_solve.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int]
    L.slu_b200_z_fill_csr.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    L.slu_b200_z_destroy.argtypes = [C.c_void_p]
    L.slu_b200_z_destroy.restype = None
    L.pzgstrf3d_b200.argtypes = [C.POINTER(LUView), C.POINTER(Options), C.POINTER(Stats), C.POINTER(C.c_int)]
    _lib = L
    return L


def _is_complex(x):
    return np.dtype(x).kind == "c"


def _fn(name, complex_):
    """The double or the doublecomplex entry point: slu_b200_<name> / slu_b200_z_<name>."""
    return getattr(lib(), ("slu_b200_z_" if complex_ else "slu_b200_") + name)


def _check(rc):
    if rc != 0:
        raise RuntimeError("libslu_b200: " + lib().slu_b200_last_error().decode())


def device_count():
    return lib().slu_b200_device_count()


def require_gpu():
    if device_count() < 1:
        raise RuntimeError("libslu_b200 needs a CUDA device; there is no CPU fallback")


def pinned_alloc(nbytes):
    """alloc(nbytes) -> (address, keepalive) for LUProblem.add_layer(alloc=...)."""
    L = lib()
    p = L.slu_b200_host_alloc(nbytes)
    if not p:
        raise MemoryError(f"cudaHostAlloc({nbytes}) failed")

    class _Keep:
        def __init__(self, p):
            self.p = p

        def __del__(self):
            try:
                L.slu_b200_host_free(self.p)
            except Exception:
                pass
    return p, _Keep(p)


def make_view(prob, z):
    """Fill a slu_b200_lu_view_t from an LUProblem layer; returns (view, keepalive)."""
    lay = prob.layers[z]
    li, lv, ui, uv = prob.pointer_tables(lay)
    trees = my_tree_idxs(prob.npdep, z)
    zeros = my_zero_tr_idxs(prob.npdep, z)
    nf = (1 << prob.max_lvl) - 1
    forests = (Forest * nf)()
    lims = []
    for f in range(nf):
        nodes = prob.forest_nodes[f]
        forests[f].nNodes = len(nodes)
        forests[f].nodeList = nodes.ctypes.data
        lim = np.array([0, len(nodes)], np.int32)
        lims.append(lim)
        forests[f].numLvl = 1
        forests[f].eTreeTopLims = lim.ctypes.data
    v = LUView()
    v.n, v.nsupers, v.xsup = prob.n, prob.nsupers, prob.xsup.ctypes.data
    v.nprow = v.npcol = 1
    v.npdep = prob.npdep
    v.myrow = v.mycol = 0
    v.mydep = z
    v.Lrowind_bc_ptr, v.Lnzval_bc_ptr = li.ctypes.data, lv.ctypes.data
    v.Ufstnz_br_ptr, v.Unzval_br_ptr = ui.ctypes.data, uv.ctypes.data
    v.maxLvl, v.myTreeIdxs, v.myZeroTrIdxs = prob.max_lvl, trees.ctypes.data, zeros.ctypes.data
    v.nforests, v.forests = nf, C.addressof(forests)
    return v, (li, lv, ui, uv, trees, zeros, forests, lims, lay)


def make_view_2d(prob, local, z):
    """View of the pieces process (local.myrow, local.mycol) of layer z holds (problem.Local2D)."""
    v, keep = make_view(prob, z)
    li, lv, ui, uv = local.pointer_tables()
    v.nprow, v.npcol, v.myrow, v.mycol = local.nprow, local.npcol, local.myrow, local.mycol
    v.Lrowind_bc_ptr, v.Lnzval_bc_ptr = li.ctypes.data, lv.ctypes.data
    v.Ufstnz_br_ptr, v.Unzval_br_ptr = ui.ctypes.data, uv.ctypes.data
    return v, (keep, li, lv, ui, uv, local)


def pdgstrf3d_2d(prob, local, z, **opt):
    """pdgstrf3d_b200 on a Pr x Pc x Pz grid: factor my pieces in place.  -> (info, Stats)"""
    require_gpu()
    view, keep = make_view_2d(prob, local, z)
    o = make_options(prob, **opt)
    st, info = Stats(), C.c_int(0)
    fn = lib().pzgstrf3d_b200 if _is_complex(prob.dtype) else lib().pdgstrf3d_b200   # complex16 twin: pzgstrf3d.c:120
    _check(fn(C.byref(view), C.byref(o), C.byref(st), C.byref(info)))
    del keep
    return info.value, st


def make_options(prob, device=-1, verbose=0, world_size=1, world_rank=0, nccl_id=None, pinned=0, schur_variant=0,
                 no_lookahead=0, no_coop=0, pipeline=0, overlap_h2d=0, tc_slices=0, tc_min_ns=0):
    o = Options()
    o.device = device
    o.replace_tiny_pivot = int(prob.replace_tiny_pivot)
    o.thresh = float(prob.thresh)
    o.verbose = verbose
    o.pinned_host = pinned
    o.schur_variant = schur_variant
    o.reserved[0] = no_lookahead   # 1: single-stream level loop (no overlap of panel work with the bulk update)
    o.reserved[2] = pipeline       # 1: pdgstrf3d_b200 overlaps H2D / factor / D2H (slu_b200_factor_host)
    o.reserved[1] = no_coop        # 1: reference-style ancestors (owner layer factors alone after a pairwise reduce)
    o.reserved[3] = overlap_h2d    # 1: level-by-level arena; factor_host also overlaps the upload (opt-in, DESIGN 9)
    o.reserved[4] = tc_slices      # tcgen05 path: int8 slices per operand (0 default, < 0 off, 5..8)
    o.reserved[5] = tc_min_ns      # narrowest supernode on the tcgen05 path (0: default)
    o.world_size, o.world_rank = world_size, world_rank
    if nccl_id is not None:
        C.memmove(o.nccl_id, bytes(nccl_id), 128)
    return o


def plan(prob, z=0, **opt):
    """slu_b200_plan / slu_b200_z_plan: the analysis of layer z without a device -> Stats (HBM bytes, flops ...)."""
    view, keep = make_view(prob, z)
    o = make_options(prob, **opt)
    st = Stats()
    _check(_fn("plan", _is_complex(prob.dtype))(C.byref(view), C.byref(o), C.byref(st)))
    del keep
    return st


def nccl_unique_id():
    buf = (C.c_ubyte * 128)()
    _check(lib().slu_b200_nccl_unique_id(buf))
    return bytes(buf)


class Handle:
    """slu_b200_handle_t: create (analysis + HBM allocation) / upload / factor / download."""

    def __init__(self, prob, z=0, **opt):
        require_gpu()
        self.prob = prob
        self.z_ = _is_complex(prob.dtype)     # doublecomplex problem -> slu_b200_z_* (pzgstrf3d)
        self.view, self._keep = make_view(prob, z)
        self.opt = make_options(prob, **opt)
        self.h = C.c_void_p()
        _check(_fn("create", self.z_)(C.byref(self.h), C.byref(self.view), C.byref(self.opt)))

    def upload(self):
        _check(_fn("upload", self.z_)(self.h))

    def factor(self):
        info = C.c_int(0)
        _check(_fn("factor", self.z_)(self.h, C.byref(info)))
        return info.value

    def factor_host(self):
        """upload + factor + download with the transfers overlapped (slu_b200_factor_host)."""
        info = C.c_int(0)
        _check(_fn("factor_host", self.z_)(self.h, C.byref(info)))
        return info.value

    def download(self):
        _check(_fn("download", self.z_)(self.h))

    def fill_csr(self, rowptr, colind, val, perm):
        """Device-side distribution (slu_b200_fill_csr / slu_b200_z_fill_csr): P A P^T scattered into the HBM panels by
        a kernel; replaces upload().  perm[old] = new; val is complex128 for a complex handle."""
        rp = np.ascontiguousarray(rowptr, np.int32)
        ci = np.ascontiguousarray(colind, np.int32)
        if self.z_:
            v = np.ascontiguousarray(val, np.complex128).view(np.float64)
        else:
            v = np.ascontiguousarray(val, np.float64)
        pm = np.ascontiguousarray(perm, np.int32)
        _check(_fn("fill_csr", self.z_)(self.h, len(rp) - 1, rp.ctypes.data_as(C.c_void_p), ci.ctypes.data_as(C.c_void_p),
                                        v.ctypes.data_as(C.c_void_p), pm.ctypes.data_as(C.c_void_p)))

    def solve(self, b):
        """L U x = b on the device-resident factors (slu_b200_solve / slu_b200_z_solve); b: (n,) or (nrhs, n), ordering
        of the factored matrix, complex128 for a complex handle.  Returns x with the same shape."""
        x = np.array(b, np.complex128 if self.z_ else np.float64, order="C", copy=True)
        nrhs = 1 if x.ndim == 1 else x.shape[0]
        _check(_fn("solve", self.z_)(self.h, x.ctypes.data_as(C.c_void_p), self.prob.n, nrhs))
        return x

    def stats(self):
        s = Stats()
        _check(_fn("get_stats", self.z_)(self.h, C.byref(s)))
        return s

    def close(self):
        if self.h:
            _fn("destroy", self.z_)(self.h)
            self.h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def pdgstrf3d(prob, z=0, **opt):
    """The one-call drop-in (pdgstrf3d_b200): factor layer z of `prob` in place.  -> (info, Stats)"""
    require_gpu()
    if _is_complex(prob.dtype):
        raise TypeError("pdgstrf3d is the double entry point; use pzgstrf3d for a complex128 problem")
    view, keep = make_view(prob, z)
    o = make_options(prob, **opt)
    st, info = Stats(), C.c_int(0)
    _check(lib().pdgstrf3d_b200(C.byref(view), C.byref(o), C.byref(st), C.byref(info)))
    del keep
    return info.value, st


def pzgstrf3d(prob, z=0, **opt):
    """pzgstrf3d_b200 (SRC/complex16/pzgstrf3d.c:120): factor layer z of a complex128 `prob` in place."""
    require_gpu()
    if not _is_complex(prob.dtype):
        raise TypeError("pzgstrf3d needs a complex128 problem")
    view, keep = make_view(prob, z)
    o = make_options(prob, **opt)
    st, info = Stats(), C.c_int(0)
    _check(lib().pzgstrf3d_b200(C.byref(view), C.byref(o), C.byref(st), C.byref(info)))
    del keep
    return info.value, st


# ---- kernel-level entry points -------------------------------------------------------------------
def k_diag_lu(a, replace_tiny=0, thresh=0.0, col0=0):
    require_gpu()
    z = _is_complex(np.asarray(a).dtype)
    a = np.array(a, np.complex128 if z else np.float64, order="F", copy=True)
    ns = a.shape[1]
    info, tiny = C.c_int(0), C.c_int(0)
    _check(_fn("k_diag_lu", z)(a.ctypes.data_as(C.c_void_p), ns, a.shape[0], replace_tiny, C.c_double(thresh),
                                    col0, C.byref(info), C.byref(tiny)))
    return a, info.value, tiny.value


def k_trsm(lu, x, ucase):
    require_gpu()
    z = _is_complex(np.asarray(lu).dtype) or _is_complex(np.asarray(x).dtype)
    dt = np.complex128 if z else np.float64
    lu = np.array(lu, dt, order="F", copy=True)
    x = np.array(x, dt, order="F", copy=True)
    ns = lu.shape[1]
    if ucase:
        _check(_fn("k_trsm_u", z)(lu.ctypes.data_as(C.c_void_p), lu.shape[0], ns, x.ctypes.data_as(C.c_void_p),
                                       x.shape[1], x.shape[0]))
    else:
        _check(_fn("k_trsm_l", z)(lu.ctypes.data_as(C.c_void_p), lu.shape[0], ns, x.ctypes.data_as(C.c_void_p),
                                       x.shape[0], x.shape[0]))
    return x


def k_gemm_sub(a, b, c, reps=0):
    require_gpu()
    z = any(_is_complex(np.asarray(t).dtype) for t in (a, b, c))
    dt = np.complex128 if z else np.float64
    a = np.array(a, dt, order="F", copy=True)
    b = np.array(b, dt, order="F", copy=True)
    c = np.array(c, dt, order="F", copy=True)
    m, k = a.shape
    n = b.shape[1]
    ms = C.c_float(0)
    _check(_fn("k_gemm_sub", z)(m, n, k, a.ctypes.data_as(C.c_void_p), a.shape[0], b.ctypes.data_as(C.c_void_p),
                                     b.shape[0], c.ctypes.data_as(C.c_void_p), c.shape[0], reps, C.byref(ms)))
    return c, ms.value
