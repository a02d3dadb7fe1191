/*
 * slu_b200.h -- C-ABI of libslu_b200.so: a B200-native (sm_100a) implementation of
 * SuperLU_DIST's 3D supernodal numeric factorization hot path `pdgstrf3d`.
 *
 * Boundary.  The reference reaches a non-C factorization backend through an opaque handle
 * (SRC/include/superlu_upacked.h:17-28, called from SRC/double/pdgssvx3d.c:1013-1021):
 *
 *     dCreateLUgpuHandle(...)   -> slu_b200_create() + slu_b200_upload()
 *     pdgstrf3d_LUv1(handle)    -> slu_b200_factor()
 *     dCopyLUGPU2Host(handle,.) -> slu_b200_download()
 *     dDestroyLUgpuHandle(.)    -> slu_b200_destroy()
 *
 * and the plain CPU/“HALO” path through `pdgstrf3d(options, m, n, anorm, trf3Dpartition, SCT,
 * LUstruct, grid3d, stat, info)` (SRC/double/pdgstrf3d.c:121-124) -> pdgstrf3d_b200().
 *
 * No reference struct crosses this boundary.  The caller passes a flat *view* (plain pointers
 * and sizes) of the structures the reference already holds; the data those pointers address
 * keep the reference's exact layout (SRC/include/superlu_defs.h:156-204):
 *
 *   L block column k  (local index k / npcol):
 *     Lrowind_bc_ptr[lk] = [ nblk, nrows ; (ib, nbrow, row ids ...) x nblk ]   BC_HEADER=2, LB_DESCRIPTOR=2
 *     Lnzval_bc_ptr[lk]  = column-major nrows x SuperSize(k); diagonal block first on its owner
 *   U block row k     (local index k / nprow):
 *     Ufstnz_br_ptr[lk]  = [ nblk, nnz, indexlen ; (jb, nnz_blk, fstnz[SuperSize(jb)]) x nblk ]  BR_HEADER=3, UB_DESCRIPTOR=2
 *     Unzval_br_ptr[lk]  = concatenated skyline column segments [fstnz, xsup[k+1])
 *
 * The INTEGRATION.md shim (oracle/ref_build/pdgstrf3d_hook.c) shows the ~60 lines a reference
 * maintainer adds to fill this view from dLUstruct_t / dtrf3Dpartition_t / gridinfo3d_t.
 *
 * Error convention (mirrors pdgstrf3d.c:388-392): functions return 0 on success, <0 on an
 * argument/runtime error (message via slu_b200_last_error()); *info = 0, or the 1-based global
 * column of the first exactly-zero pivot, min-reduced over all ranks of the 3D grid.
 */
#ifndef SLU_B200_H
#define SLU_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SLU_B200_ABI_VERSION 1

/* int_t of the reference's default build (SRC/include/superlu_defs.h:126-129). */
typedef int32_t slu_int;

/* One sForest_t (SRC/include/superlu_defs.h:940-962): an elimination sub-forest. */
typedef struct {
    slu_int nNodes;               /* number of supernodes in the forest (0: empty)          */
    const slu_int *nodeList;      /* supernode ids in an order valid for factorization      */
    slu_int numLvl;               /* topoInfo.numLvl (informational)                        */
    const slu_int *eTreeTopLims;  /* topoInfo.eTreeTopLims[numLvl+1] (informational)        */
} slu_b200_forest_t;

/* Flat view of Glu_persist_t + gridinfo3d_t + dLocalLU_t + dtrf3Dpartition_t. */
typedef struct {
    /* Glu_persist_t (superlu_defs.h:454-457) */
    slu_int n;                    /* matrix order                                            */
    slu_int nsupers;              /* number of supernodes                                    */
    const slu_int *xsup;          /* [nsupers+1] first column of each supernode              */
    /* gridinfo3d_t (superlu_defs.h:417-438) */
    slu_int nprow, npcol, npdep;  /* process grid Pr x Pc x Pz (Pz a power of two)                */
    slu_int myrow, mycol, mydep;  /* my coordinates                                          */
    /* dLocalLU_t (superlu_ddefs.h:97-307): arrays of per-local-block pointers (host memory) */
    slu_int **Lrowind_bc_ptr;     /* [ceil(nsupers/npcol)]                                   */
    double **Lnzval_bc_ptr;       /* [ceil(nsupers/npcol)]  in: A / partial sums, out: L     */
    slu_int **Ufstnz_br_ptr;      /* [ceil(nsupers/nprow)]                                   */
    double **Unzval_br_ptr;       /* [ceil(nsupers/nprow)]  in: A / partial sums, out: U     */
    /* dtrf3Dpartition_t (superlu_ddefs.h:317-337) */
    slu_int maxLvl;               /* log2(npdep)+1                                           */
    const slu_int *myTreeIdxs;    /* [maxLvl] forest index I hold at each Z-tree level       */
    const slu_int *myZeroTrIdxs;  /* [maxLvl] 1 = my copy of that forest starts as zeros     */
    slu_int nforests;             /* 2^maxLvl - 1                                            */
    const slu_b200_forest_t *forests; /* [nforests]                                          */
} slu_b200_lu_view_t;

typedef struct {
    int32_t device;               /* CUDA device ordinal (-1: current device)                */
    int32_t replace_tiny_pivot;   /* options->ReplaceTinyPivot (superlu_defs.h:707)          */
    double thresh;                /* smach_dist("Epsilon")*anorm (pdgstrf3d.c:132-133)       */
    int32_t verbose;              /* 0 silent                                                */
    int32_t pinned_host;          /* 1: caller's nzval arrays are page-locked (faster copies) */
    /* multi-GPU (npdep*nprow*npcol > 1): one NCCL communicator over the 3D grid replaces   */
    /* grid3d->comm for the panel / ancestor traffic (pd3dcomm.c:1046-1081).                 */
    int32_t world_size;           /* ranks in the 3D grid (1: no communication)              */
    int32_t world_rank;           /* my rank: mydep*(nprow*npcol) + myrow*npcol + mycol      */
    unsigned char nccl_id[128];   /* ncclUniqueId from slu_b200_nccl_unique_id on rank 0     */
    int32_t schur_variant;        /* 0 (default) = 4: 128x64 DMMA tiles, 2 CTAs/SM, running-pointer loader;
                                     5: the same with BK=32; 6: the round-1 general loader; 1: 128x128 tiles,
                                     1 CTA/SM; 3: general loader, BK=32 for wide supernodes */
    int32_t reserved[7];          /* [0] no look-ahead, [1] reference-style ancestors, [2] pdgstrf3d_b200 */
                                  /* uses slu_b200_factor_host (overlapped transfers), [3] level-by-  */
                                  /* level arena so that factor_host also overlaps the upload,        */
                                  /* [4] tcgen05 path for wide supernodes: int8 slices per operand    */
                                  /* (0 = default 7, 5..8, < 0 = off: FP64 DMMA only), [5] narrowest   */
                                  /* supernode that takes the tcgen05 path (0 = default 128)          */
} slu_b200_options_t;

typedef struct {
    double ops_fact;              /* flops, reference accounting (stat->ops[FACT]): diag LU  */
                                  /* pdgstrf2.c:578,590; U-TRSM trfAux.c:2303; Schur         */
                                  /* sec_structs.c:692-693.  Local to this rank.             */
    double ops_schur;             /* the 2*m*n*k part of ops_fact                            */
    double schur_bytes;           /* algorithmic bytes of the Schur updates (DESIGN.md)      */
    int64_t tiny_pivots;          /* stat->TinyPivots                                        */
    int64_t gpu_launches;         /* kernels launched by the last slu_b200_factor()          */
    double t_analyze_s;           /* host: structure analysis + device index build           */
    double t_upload_s;            /* H2D of L/U values                                       */
    double t_factor_s;            /* device time of the last factor (CUDA events)            */
    double t_download_s;          /* D2H of L/U values                                       */
    double t_diag_ms, t_trsm_ms, t_schur_setup_ms, t_schur_ms, t_reduce_ms; /* phase sums,   */
                                  /* only filled when options.verbose >= 2 (adds syncs)      */
    int64_t lu_device_bytes;      /* HBM held by L/U values                                  */
    int64_t index_device_bytes;   /* HBM held by index structures + workspace                */
    int64_t nnz_l, nnz_u;         /* elements (complex: pairs) in my L / U panels (device)   */
    int32_t nlevels;              /* level-synchronous steps executed                        */
    int32_t my_supernodes;        /* supernodes this rank factored                           */
    double reserved[8];           /* [0] ms spent slicing (verbose >= 2), [1] Schur flops taken by the */
                                  /* tcgen05 path, [2] bytes of its int8 workspace, [3] slices in use,  */
                                  /* [4] seconds of the last slu_b200_solve / slu_b200_z_solve,         */
                                  /* [5] its kernel launches                                            */
} slu_b200_stats_t;

typedef struct slu_b200_handle_s *slu_b200_handle_t;

int slu_b200_abi_version(void);
/* sizeof of {slu_b200_forest_t, slu_b200_lu_view_t, slu_b200_options_t, slu_b200_stats_t}: lets a
 * foreign-function binding (cgo / ctypes / Fortran) verify its struct mirrors before the first call */
void slu_b200_struct_sizes(int32_t out[4]);
const char *slu_b200_last_error(void);
/* number of visible CUDA devices (0 if none / driver missing); never throws */
int slu_b200_device_count(void);

/* Analyse the structure, allocate HBM, build device index structures.  Values are not read. */
int slu_b200_create(slu_b200_handle_t *h, const slu_b200_lu_view_t *lu,
                    const slu_b200_options_t *opt);
/* H2D: copy the view's Lnzval/Unzval (for the supernodes of my forests) into HBM. */
int slu_b200_upload(slu_b200_handle_t h);
/* Factor in HBM.  Collective over the NCCL communicator when world_size > 1. */
int slu_b200_factor(slu_b200_handle_t h, int *info);
/* upload + factor + download in one call with the D2H overlapped with the factorization: a panel is
 * final once the panel work of its level is done, so it is copied back on a second stream while the
 * upper levels are still being factored.  Same result as the three separate calls; needs page-locked
 * host arrays to actually overlap.  Patterns whose U skylines are not all full (unsymmetric patterns) and
 * Pr x Pc pieces take the plain upload / factor / download path inside this call: same results, no overlap. */
int slu_b200_factor_host(slu_b200_handle_t h, int *info);
/* D2H: write L and U back into the view's Lnzval/Unzval in the reference layout. */
int slu_b200_download(slu_b200_handle_t h);
/* Device-side distribution (the job of pddistribute3d, SRC/double/pddistribute3d.c:1357, on the GPU): instead of
 * slu_b200_upload of the caller's Lnzval/Unzval arrays, scatter the matrix itself into the panels.  A: n x n host CSR
 * (int32 indices, no duplicate entries); perm[old] = new is the final permutation of the factored matrix
 * (P (A) P^T, rows and columns alike).  12 bytes per nonzero cross PCIe instead of 8 bytes per factor entry; the value
 * arrays of the view may then be NULL-backed (never read) if the caller also skips slu_b200_download.  1 x 1 x Pz. */
int slu_b200_fill_csr(slu_b200_handle_t h, int n, const int32_t *rowptr, const int32_t *colind, const double *val,
                      const int32_t *perm);
/* Solve L U x = b with the factors still resident in HBM (after a successful slu_b200_factor / _factor_host on this
 * handle) -- the consumer of pdgstrf3d, pdgstrs3d (SRC/double/pdgstrs3d.c:6604), without the D2H/H2D round trip.
 * x: host, n x nrhs column-major (ldx >= n), in the ordering of the factored matrix (the caller applies the
 * permutations / scalings, as pdgssvx3d does around pdgstrs3d); holds b on entry, the solution on return.
 * 1 x 1 x Pz grids: collective, every rank passes the same b and receives the full x (NCCL all-reduces along Z
 * replace the ancestor reduce / dbroadcastAncestor3d, pd3dcomm.c:1145).  stats.reserved[4] = seconds of the call. */
int slu_b200_solve(slu_b200_handle_t h, double *x, int ldx, int nrhs);
int slu_b200_get_stats(slu_b200_handle_t h, slu_b200_stats_t *out);
void slu_b200_destroy(slu_b200_handle_t h);

/* The one-call drop-in for pdgstrf3d (pdgstrf3d.c:121): create+upload+factor+download+destroy. */
int pdgstrf3d_b200(const slu_b200_lu_view_t *lu, const slu_b200_options_t *opt,
                   slu_b200_stats_t *stats, int *info);

/* Fill `id` (128 bytes) with a fresh ncclUniqueId; rank 0 calls it and broadcasts the bytes. */
int slu_b200_nccl_unique_id(unsigned char id[128]);
/* The NCCL communicators (world + per-Z-level groups) built from an id are cached per process and reused by every
 * later create / pdgstrf3d_b200 with the same id and grid coordinates -- the counterpart of the MPI communicators
 * superlu_gridinit3d creates once (SRC/prec-independent/superlu_grid3d.c:47-63).  Destroy them explicitly: */
void slu_b200_comm_cache_clear(void);

/* Page-locked host allocation helpers for callers that want full-speed PCIe copies. */
void *slu_b200_host_alloc(size_t bytes);
void slu_b200_host_free(void *p);

/* Analysis only -- needs no device: fills stats (lu_device_bytes, index_device_bytes, ops_fact, nnz_l/u, nlevels,
 * my_supernodes) for this rank of a 1 x 1 x Pz grid, e.g. to size a run for 180 GB GPUs before allocating them
 * (the role of the reference's memory estimate dQuerySpace_dist, SRC/double/dmemory_dist.c). */
int slu_b200_plan(const slu_b200_lu_view_t *lu, const slu_b200_options_t *opt, slu_b200_stats_t *stats);

/* ---- kernel-level entry points (host pointers; used by tests and micro-benchmarks) ---------- */
/* In-place unpivoted LU of an ns x ns column-major block (Local_Dgstrf2, pdgstrf2.c:508-601). */
int slu_b200_k_diag_lu(double *a, int ns, int lda, int replace_tiny, double thresh, int col0,
                       int *info, int *tiny);
/* X <- X * U^-1, U = upper triangle (non-unit) of lu[ns x ns] (dLPanelTrSolve,
 * dtrfCommWrapper.c:120-223).  x is m x ns column-major. */
int slu_b200_k_trsm_l(const double *lu, int ldlu, int ns, double *x, int m, int ldx);
/* X <- L^-1 * X, L = unit lower triangle of lu (dUPanelTrSolve, dtrfCommWrapper.c:242-357).
 * x is ns x ncols column-major. */
int slu_b200_k_trsm_u(const double *lu, int ldlu, int ns, double *x, int ncols, int ldx);
/* C <- C - A*B with the Schur-update main loop (dblock_gemm_scatter, dscatter3d.c:82-189,
 * identity scatter).  Returns device milliseconds of the kernel in *ms if non-NULL. */
int slu_b200_k_gemm_sub(int m, int n, int k, const double *a, int lda, const double *b, int ldb,
                        double *c, int ldc, int reps, float *ms);
/* benchmark support (SURVEY 8a row a10): see slu_api.cu; device_lu receives the library's DeviceLU struct (device
 * pointers; layout in superlu_dist_b200/csrc/cuda/slu_device.cuh), nodes the level's supernodes with a big update.
 * Returns their count (< 0 on error). */
int slu_b200_k_level_export(slu_b200_handle_t h, int level, void *device_lu, int device_lu_bytes, int32_t *nodes, int max_nodes);
int slu_b200_k_rerun_schur(slu_b200_handle_t h, int level, int reps, float *ms);
/* ---- doublecomplex twins (SRC/complex16/pzgstrf3d.c:120; the reference's z* handle API,
 * SRC/include/superlu_upacked.h:84-97).  Same view/options/stats structs: the Lnzval_bc_ptr / Unzval_br_ptr
 * entries point at arrays of doublecomplex {double r, i} (SRC/include/dcomplex.h:30) and are declared double*
 * only to keep one struct; n, nsupr, lda ... count complex elements.  Supernodes up to 256 columns.
 * stats.ops_fact follows the reference's own complex accounting (pzgstrf2.c:578,590 for the diagonal blocks,
 * the precision-independent 2*m*n*k for the Schur update, sec_structs.c:692-693).
 * Validated on a B200 (GPUTEST_r01.json: kernels vs NumPy, cg20 vs the reference's pzgstrf3d factors, pzdrive3d
 * drop-in); gating tests in tests/test_gpu_variants_complex.py. */
typedef struct slu_b200_zhandle_s *slu_b200_zhandle_t;
int slu_b200_z_create(slu_b200_zhandle_t *h, const slu_b200_lu_view_t *lu, const slu_b200_options_t *opt);
int slu_b200_z_upload(slu_b200_zhandle_t h);
int slu_b200_z_factor(slu_b200_zhandle_t h, int *info);
int slu_b200_z_factor_host(slu_b200_zhandle_t h, int *info);
int slu_b200_z_download(slu_b200_zhandle_t h);
int slu_b200_z_get_stats(slu_b200_zhandle_t h, slu_b200_stats_t *out);
int slu_b200_z_plan(const slu_b200_lu_view_t *lu, const slu_b200_options_t *opt, slu_b200_stats_t *stats);
void slu_b200_z_destroy(slu_b200_zhandle_t h);
/* drop-in body of pzgstrf3d (complex16/pzgstrf3d.c:120-123): create + upload + factor + download + destroy */
int pzgstrf3d_b200(const slu_b200_lu_view_t *lu, const slu_b200_options_t *opt, slu_b200_stats_t *stats, int *info);
/* Device-side distribution, as slu_b200_fill_csr (the job of pzdistribute3d, SRC/complex16/pzdistribute3d.c:24):
 * val holds nnz (re, im) pairs; 20 bytes per nonzero cross PCIe instead of 16 bytes per factor entry.  1 x 1 x Pz. */
int slu_b200_z_fill_csr(slu_b200_zhandle_t h, int n, const int32_t *rowptr, const int32_t *colind,
                        const double *val, const int32_t *perm);
/* Solve L U x = b on the resident factors, as slu_b200_solve (the job of pzgstrs3d, SRC/complex16/pzgstrs3d.c:6694):
 * x holds n x nrhs (re, im) pairs column-major, ldx counts complex elements.  1 x 1 x Pz grids: collective, every rank
 * passes the same b and receives the full x.  stats.reserved[4] = seconds of the call, [5] = its kernel launches. */
int slu_b200_z_solve(slu_b200_zhandle_t h, double *x, int ldx, int nrhs);
void slu_b200_z_comm_cache_clear(void);   /* called by slu_b200_comm_cache_clear */
/* kernel-level test entries; arrays are interleaved (re, im), sizes in complex elements */
int slu_b200_z_k_diag_lu(double *a, int ns, int lda, int replace_tiny, double thresh, int col0, int *info, int *tiny);
int slu_b200_z_k_trsm_l(const double *lu, int ldlu, int ns, double *x, int m, int ldx);
int slu_b200_z_k_trsm_u(const double *lu, int ldlu, int ns, double *x, int ncols, int ldx);
int slu_b200_z_k_gemm_sub(int m, int n, int k, const double *a, int lda, const double *b, int ldb, double *c, int ldc,
                          int reps, float *ms);

#ifdef __cplusplus
}
#endif
#endif /* SLU_B200_H */
