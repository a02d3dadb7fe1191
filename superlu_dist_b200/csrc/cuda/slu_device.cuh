// slu_device.cuh -- data structures shared by the host orchestration (slu_api.cu) and the sm_100a
// kernels (slu_kernels.cu) of libslu_b200.so.
//
// HBM layout (DESIGN.md section 3).  One value arena `val` (double) holds, per Z-tree level of the
// forests this rank owns, first the L panels then the U panels of that forest:
//   L panel k : column-major nsupr x ns, lda = nsupr  -- byte-identical to Lnzval_bc_ptr[k]
//               (SRC/include/superlu_defs.h:156-178), so upload/download of L is a plain copy;
//   U panel k : DENSE-PACKED ns x ncols, ld = ns: only the columns with a non-empty skyline segment,
//               zero-padded above the segment.  This is the GEMM-ready form the reference re-creates
//               for every supernode in dRgather_U (SRC/double/dgather.c:256-398); here it is the
//               resident form and is converted from/to the skyline of Unzval_br_ptr[k] only at
//               upload/download.
// Index arenas (int32): per L panel the row ids in panel order (`lrows`) and a sorted copy with the
// panel position of each (`lsrow`,`lspos`) for destination lookups; per U panel the sorted global
// column ids of its packed columns (`ucols`) with first-nonzero row (`ufst`) and skyline offset
// (`useg`).
//
// The header (and slu_api.cu) is compiled twice: as is for double (namespace slu, pdgstrf3d) and with SLU_COMPLEX
// for doublecomplex (namespace sluz, pzgstrf3d; SURVEY 8a row a15: "identical algorithm on interleaved (r,i)
// pairs").  All offsets and lengths count ELEMENTS of val_t, so the host orchestration is the same source.
#pragma once
#include <cstdint>
#include <cuda_runtime.h>

#ifdef SLU_COMPLEX
#define SLU_NS sluz
#else
#define SLU_NS slu
#endif

namespace SLU_NS {

#ifdef SLU_COMPLEX
typedef double2 val_t;       // (re, im) = the reference's doublecomplex, SRC/include/dcomplex.h:30
#else
typedef double val_t;
#endif
constexpr int VAL_DOUBLES = (int)(sizeof(val_t) / sizeof(double));

struct NodeDesc {            // one per supernode (indexed by global supernode id); zero if not held
    int32_t held, ns, nsupr, m, ncols, nlb, nub, fsupc;
    int64_t lval, uval;      // offsets into val (elements)
    int64_t lrow, ucol;      // offsets into lrows/lsrow/lspos and ucols/ufst/useg
    int64_t lblk, ublk;      // offsets into the LBlk / UBlk arrays
    int64_t ws_row, ws_col;  // offsets into the per-level rowinfo / colinfo workspace
    int64_t ws_lrel, ws_urel;
    int64_t lrel_total, urel_total;
    int64_t ws_inv;          // offset into the per-level workspace of inverted 16x16 diagonal blocks
    int32_t urg_rows, urg_cols;  // look-ahead: leading rows / packed columns whose destination is factored at
                                 // the NEXT level (the parent supernode); tiles touching them are "urgent"
    // tcgen05 path (slu_ozaki.cu): per-level workspace of this supernode's int8 slices and scales
    int64_t ws_oza, ws_ozb;      // byte offsets into oz_i8: A tiles [rt][ks][s][4096], B tiles [ct][ks][s][OZ_NT*32]
    int64_t ws_ozs;              // element offset into oz_scale / oz_rexp: row scales [0, 128*RT), column scales after
};

struct LBlk {                // an off-diagonal L block of panel k
    int32_t ib, row0, nrows; // rows [row0, row0+nrows) of the m sub-diagonal rows
    int32_t colstart;        // first packed U column j of panel k with supno(col) > ib (U-destinations)
    int64_t urel_off;        // offset (within the node's urel table) of this block's column map
    int32_t shared, pad;     // 1: another supernode of the same level also updates panel ib (scatter must be atomic)
};
struct UBlk {                // a U block (packed columns [col0, col0+ncols)) of block row k
    int32_t jb, col0, ncols;
    int32_t rowstart;        // first sub-diagonal row i of panel k with supno(row) >= jb (L-destinations)
    int64_t lrel_off;
    int32_t shared, pad;     // 1: another supernode of the same level also updates panel jb
};

struct RowInfo {             // built per supernode by schur_setup_kernel
    int32_t ib, ldu;         // destination block row and its leading dimension (SuperSize(ib))
    int64_t ubase;           // val offset of element (row, first packed column) of U panel ib
    int64_t urel_off;        // urel[urel_off + j] = packed column position of source column j
    int32_t shared, pad;     // destination U panel ib is also updated by another supernode of this level
};
struct ColInfo {
    int32_t jb, pad;         // pad: 1 if destination L panel jb is also updated by another supernode of this level
    int64_t lbase;           // val offset of the top of destination column in L panel jb
    int64_t lrel_off;        // lrel[lrel_off + i] = row position of source row i in L panel jb
};

struct DeviceLU {            // everything the kernels need, passed by value
    val_t *val;
    const NodeDesc *nodes;
    const int32_t *xsup, *supno;
    const int32_t *lrows, *lsrow, *lspos;
    const int32_t *ucols, *ufst, *useg;
    const LBlk *lblk;
    const UBlk *ublk;
    RowInfo *rowinfo;
    ColInfo *colinfo;
    int32_t *lrel, *urel;
    int8_t *oz_i8;           // tcgen05 path: int8 slice tiles of the level's wide supernodes
    double *oz_scale;        //   2^(e-6) back-scales of their rows / columns
    int *oz_rexp;            //   row exponents (between the two slicing passes)
    int *info;               // min over zero pivots of (1-based global column); INT_MAX if none
    unsigned long long *tiny;
    int *err;                // debug: count of destination lookups that failed
};

struct Batch {               // one kernel launch over several supernodes
    const int32_t *nodes;    // supernode ids
    const int64_t *prefix;   // [count+1] cumulative CTA counts
    int32_t count;
};

constexpr int DIAG_NB = 16;
constexpr bool DIAG_CLUSTER_DEFAULT = true;   // 8-CTA cluster LU of 65..256-column diagonal blocks (SLU_B200_DIAG_CLUSTER=1|0 overrides)
constexpr int TRSM_NB = 16;
constexpr bool TRSM_RL_DEFAULT = false;      // right-looking register-blocked panel solve (SLU_B200_TRSM_RL=1|0 overrides)
constexpr int MAX_NS = 512;  // MAX_SUPER_SIZE, SRC/include/superlu_defs.h:154
#ifdef SLU_COMPLEX
constexpr int TRSM_STRIP = 32;      // vectors a TRSM CTA keeps in shared memory (16-byte elements)
constexpr int MAX_NS_HELD = 256;    // widest supernode the kernels accept (the default superlu_maxsup)
constexpr int TRSM_WIDE_NS = MAX_NS_HELD;   // no half-width strips in the doublecomplex build
constexpr int SCHUR_BN_TILE = 32;   // columns of a big Schur tile (complex columns: 64 real ones)
#else
constexpr int TRSM_STRIP = 64;
constexpr int MAX_NS_HELD = MAX_NS;  // MAX_SUPER_SIZE
constexpr int TRSM_WIDE_NS = 416;    // a 64-vector strip of a wider supernode does not fit 227 KB: those use 32-vector strips
constexpr int SCHUR_BN_TILE = 64;
#endif

// vectors per TRSM CTA for a supernode of ns columns (the CTA prefix of a level batch is built with this)
__host__ __device__ inline int trsm_strip_of(int ns) { return ns > TRSM_WIDE_NS ? TRSM_STRIP / 2 : TRSM_STRIP; }

// launchers (slu_kernels.cu).  Every launcher returns the number of kernels it launched.
// replace_tiny: 0 off, 1 replace and count in d.tiny, 2 replace without counting (replicated copy of a shared forest)
int launch_diag_lu(const DeviceLU &d, const Batch &b, int max_ns, int replace_tiny, double thresh,
                   cudaStream_t s);
// inverse of every 16x16 diagonal block of U_kk and L_kk: dinv[ws_inv + blk*512 + {0: inv U, 256: inv L}]
int launch_diag_inv(const DeviceLU &d, const Batch &b, int64_t ctas, val_t *dinv, cudaStream_t s);
int launch_trsm_l(const DeviceLU &d, const Batch &b, int64_t ctas, int max_ns, const val_t *dinv, cudaStream_t s);
int launch_trsm_u(const DeviceLU &d, const Batch &b, int64_t ctas, int max_ns, const val_t *dinv, cudaStream_t s);
int launch_schur_setup(const DeviceLU &d, const Batch &b, int64_t ctas, cudaStream_t s);
// variant 0 (default): 128x64 tiles, 256 threads, 2 CTAs/SM; variant 1: 128x128 tiles, 512 threads, 1 CTA/SM
// mode 0: every tile of each supernode; 1: only the urgent tiles (urg_rows/urg_cols); 2: only the others
// split_n/split_i: this rank takes tiles t with t % split_n == split_i (cooperative ancestor forests)
int launch_schur(const DeviceLU &d, const Batch &b, int64_t ctas, int big, int atomic, int variant, int mode, int split_n,
                 int split_i, int wide, cudaStream_t s);
// skyline (sky + sky_off[slot]) <-> dense-packed U panel of each node of the batch; 32 columns per CTA
int launch_u_convert(const DeviceLU &d, const Batch &b, int64_t ctas, int pack, val_t *sky,
                     const int64_t *sky_off, cudaStream_t s);
int launch_axpy(val_t *dst, const val_t *src, int64_t n, cudaStream_t s);
// dst += src with atomic adds (overlapped upload: races with the Schur scatter into the same panels)
int launch_axpy_atomic(val_t *dst, const val_t *src, int64_t n, cudaStream_t s);
struct UpSeg { int64_t dst, src, len; };  // a transfer chunk: arena offset, (unused), length in elements
// standalone kernel tests
int launch_gemm_sub(int m, int n, int k, const val_t *a, int lda, const val_t *b, int ldb, val_t *c,
                    int ldc, int variant, cudaStream_t s);

// slu_solve.cu / slu_solve_z.cu: triangular solves on the resident factors.  x: device, n x nrhs, ordering of the
// factored matrix
constexpr int SOLVE_TILE = 256;
int launch_solve_diag(const DeviceLU &d, const int32_t *nodes, int count, bool upper, val_t *x, int n, int nrhs, cudaStream_t s);
int launch_solve_update(const DeviceLU &d, const Batch &b, int64_t ctas, bool upper, val_t *x, int n, int nrhs, cudaStream_t s);
// x[entries of the listed supernodes] = src[...] (src == nullptr: 0)
int launch_solve_mask(const DeviceLU &d, const int32_t *nodes, int count, val_t *x, int n, int nrhs, const val_t *src, cudaStream_t s);
// device-side distribution of a CSR matrix (device arrays) into the arena; *err counts entries without a slot
int launch_fill_csr(const DeviceLU &d, int n, const int32_t *rowptr, const int32_t *colind, const val_t *aval, const int32_t *perm,
                    const int8_t *active, int *err, cudaStream_t s);

#ifndef SLU_COMPLEX
// slu_ozaki.cu: the Schur update of wide supernodes on tcgen05 (int8 slices, exact int32 accumulation in TMEM)
constexpr int OZ_NT = 32;             // columns of one CTA's tcgen05 Schur tile (rows: 128)
constexpr int OZ_CL = 1;              // CTAs per cluster sharing the A operand by multicast (2 and 4 measured SLOWER: r02_notes.md)
constexpr int OZ_NT_HOST = OZ_NT * OZ_CL;  // columns of the tile unit the host enumerates
constexpr int OZ_KSTEP = 32;          // int8 k per MMA instruction and per pipeline stage
constexpr int OZ_DEFAULT_SLICES = 7;  // 48 bits per operand: error ~1e-15 * k * rowmax * colmax (scripts/ozaki_emulate.py)
constexpr int OZ_DEFAULT_MIN_NS = 128;
constexpr bool OZ_PERSIST_DEFAULT = false;     // persistent warp-specialised tcgen05 Schur kernel (SLU_B200_TC_PERSIST=1|0)
constexpr bool OZ_NONATOMIC_DEFAULT = false;   // SLU_B200_TC_NONATOMIC=1|0 overrides
constexpr bool OZ_DEFAULT_ON = true;  // validated on hardware: profiles/r02_notes.md (options.reserved[4] = -1 / SLU_B200_TC_SLICES=0: off)
inline int64_t oz_a_bytes(int m, int ns, int S) { return (int64_t)((m + 127) / 128) * ((ns + OZ_KSTEP - 1) / OZ_KSTEP) * S * 4096; }
inline int64_t oz_b_bytes(int n, int ns, int S) { return (int64_t)((n + OZ_NT - 1) / OZ_NT) * ((ns + OZ_KSTEP - 1) / OZ_KSTEP) * S * OZ_NT * OZ_KSTEP; }
inline int64_t oz_scale_elems(int m, int n) { return (int64_t)((m + 127) / 128) * 128 + (int64_t)((n + OZ_NT - 1) / OZ_NT) * OZ_NT; }
// slice the L rows / U columns of the batch's supernodes (3 launches); prefixes: row tiles, row tiles x k-steps, 4-column groups
int launch_oz_slice(const DeviceLU &d, const int32_t *nodes, int count, const int64_t *p_rt, int64_t n_rt, const int64_t *p_ak,
                    int64_t n_ak, const int64_t *p_b, int64_t n_b, int S, cudaStream_t s);
// fused GEMM + scatter of the batch's 128 x OZ_NT tiles; mode / split as launch_schur
// nonatomic: destinations flagged exclusive (LBlk/UBlk.shared == 0) are updated with plain load/store instead of RED --
// the caller must then order this level's updates after ALL earlier levels' (no bulk update of level l-1 in flight)
int launch_oz_schur(const DeviceLU &d, const Batch &b, int64_t ctas, int mode, int split_n, int split_i, int S, int nonatomic,
                    cudaStream_t s);
// slu_ozaki.cu: C -= A*B through int8 slices on tcgen05 (variants 120..142: slices and tile width)
int launch_gemm_sub_ozaki(int m, int n, int k, const double *a, int lda, const double *b, int ldb, double *c, int ldc,
                          int variant, cudaStream_t s);
#endif

#ifdef SLU_COMPLEX
constexpr int SCHUR_BM_BIG = 128, SCHUR_BN_BIG = 32, SCHUR_BM_SMALL = 32, SCHUR_BN_SMALL = 16;
#else
constexpr int SCHUR_BM_BIG = 128, SCHUR_BN_BIG = 128, SCHUR_BM_SMALL = 32, SCHUR_BN_SMALL = 32;
#endif
constexpr int SETUP_THREADS = 256;

}  // namespace SLU_NS
