// slu_solve.cu -- triangular solves on the device-resident factors (SURVEY 8f row N2: the consumer of pdgstrf3d).
//
// The reference solves with pdgstrs3d (SRC/double/pdgstrs3d.c:6604): per supernode a dense triangular solve with the
// diagonal block and a GEMV-like update of the dependent rows, messages along the process grid, and along Z the
// ancestor contributions reduced pairwise / the ancestor solution broadcast back (dbroadcastAncestor3d,
// pd3dcomm.c:1145).  Here the factors never leave HBM: the same level batches that drove the factorization drive
//   forward   for every level, bottom-up:   x_k <- L_kk^-1 x_k ;  x[rows below] -= L(below,k) x_k     (atomic adds)
//   backward  for every level, top-down:    x_k <- x_k - U(k,:) x[cols] ;  x_k <- U_kk^-1 x_k
// with four small kernels per level; one right-hand side streams L and U once (HBM-bound: 8 bytes per stored entry,
// 16 in doublecomplex).
// x is a device vector in the ordering of the factored matrix (the caller applies the permutations, as pdgssvx3d does
// around pdgstrs3d).
//
// Compiled twice, like slu_api.cu: as is for double (namespace slu) and through slu_solve_z.cu with SLU_COMPLEX for
// doublecomplex (namespace sluz, the job of pzgstrs3d, SRC/complex16/pzgstrs3d.c:6694).  The kernels are written on
// val_t with the arithmetic helpers below; for double they expand to exactly the plain scalar operations.
#include "slu_device.cuh"
#define SLU_COMMON_HELPERS_ONLY
#include "slu_kernels_common.cuh"

namespace SLU_NS {

constexpr int SOLVE_ROWS = 256;   // rows of an L panel / columns of a U panel per CTA in the update kernels

// ---- val_t arithmetic ------------------------------------------------------------------------------------------
#ifdef SLU_COMPLEX
__device__ __forceinline__ void vmul_add(val_t &acc, val_t a, val_t b)   // acc += a * b
{
    acc.x += a.x * b.x - a.y * b.y;
    acc.y += a.x * b.y + a.y * b.x;
}
__device__ __forceinline__ void vmul_sub(val_t &acc, val_t a, val_t b)   // acc -= a * b
{
    acc.x -= a.x * b.x - a.y * b.y;
    acc.y -= a.x * b.y + a.y * b.x;
}
__device__ __forceinline__ void vadd(val_t &acc, val_t a) { acc.x += a.x; acc.y += a.y; }
__device__ __forceinline__ void vsub(val_t &acc, val_t a) { acc.x -= a.x; acc.y -= a.y; }
// 1 / p by Smith's scaling (no overflow of |p|^2): the reference's slud_z_div, as zrecip in slu_kernels_z.cu
__device__ __forceinline__ val_t vrecip(val_t p)
{
    if (fabs(p.x) >= fabs(p.y)) {
        const double r = p.y / p.x, den = p.x + p.y * r;
        return make_double2(1.0 / den, -r / den);
    }
    const double r = p.x / p.y, den = p.y + p.x * r;
    return make_double2(r / den, -1.0 / den);
}
__device__ __forceinline__ val_t vdiv(val_t a, val_t p)                  // a / p
{
    const val_t q = vrecip(p);
    return make_double2(a.x * q.x - a.y * q.y, a.x * q.y + a.y * q.x);
}
__device__ __forceinline__ val_t vshfl(val_t v, int lane)
{
    return make_double2(__shfl_sync(0xffffffffu, v.x, lane), __shfl_sync(0xffffffffu, v.y, lane));
}
// there is no double2 atomicAdd: the two halves are independent doubles (as the complex Schur epilogue does)
__device__ __forceinline__ void vatomic_sub(val_t *p, val_t a)
{
    atomicAdd(&p->x, -a.x);
    atomicAdd(&p->y, -a.y);
}
#else
__device__ __forceinline__ void vmul_add(val_t &acc, val_t a, val_t b) { acc += a * b; }
__device__ __forceinline__ void vmul_sub(val_t &acc, val_t a, val_t b) { acc -= a * b; }
__device__ __forceinline__ void vadd(val_t &acc, val_t a) { acc += a; }
__device__ __forceinline__ void vsub(val_t &acc, val_t a) { acc -= a; }
__device__ __forceinline__ val_t vdiv(val_t a, val_t p) { return a / p; }
__device__ __forceinline__ val_t vshfl(val_t v, int lane) { return __shfl_sync(0xffffffffu, v, lane); }
__device__ __forceinline__ void vatomic_sub(val_t *p, val_t a) { atomicAdd(p, -a); }
#endif
__device__ __forceinline__ val_t vzero() { return val_t{}; }

// x_k <- L_kk^-1 x_k (unit lower) or U_kk^-1 x_k (upper, non-unit): one CTA per supernode, column sweep in shared
// memory.  16-column blocks: warp 0 finishes the block's 16 unknowns with shuffles, then all threads apply them.
template <bool UPPER>
__global__ void __launch_bounds__(256) solve_diag_kernel(DeviceLU d, const int32_t *nodes, val_t *x, int n, int nrhs)
{
    __shared__ val_t xs[MAX_NS_HELD];
    const NodeDesc nd = d.nodes[nodes[blockIdx.x]];
    const int ns = nd.ns, lda = nd.nsupr, tid = threadIdx.x;
    const val_t *A = d.val + nd.lval;
    for (int rhs = 0; rhs < nrhs; ++rhs) {
        val_t *xk = x + (size_t)rhs * n + nd.fsupc;
        for (int r = tid; r < ns; r += 256) xs[r] = xk[r];
        __syncthreads();
        if (!UPPER) {
            for (int c0 = 0; c0 < ns; c0 += 16) {
                const int cb = min(16, ns - c0);
                if (tid < 32) {   // the 16 x 16 unit-lower block, lane r owns unknown c0 + r
                    val_t v = (tid < cb) ? xs[c0 + tid] : vzero();
                    for (int c = 0; c < cb; ++c) {
                        const val_t xc = vshfl(v, c);
                        if (tid > c && tid < cb) vmul_sub(v, A[(size_t)(c0 + c) * lda + c0 + tid], xc);
                    }
                    if (tid < cb) xs[c0 + tid] = v;
                }
                __syncthreads();
                for (int r = c0 + cb + tid; r < ns; r += 256) {
                    val_t acc = vzero();
                    for (int c = 0; c < cb; ++c) vmul_add(acc, A[(size_t)(c0 + c) * lda + r], xs[c0 + c]);
                    vsub(xs[r], acc);
                }
                __syncthreads();
            }
        } else {
            for (int c1 = ns; c1 > 0; c1 -= 16) {
                const int c0 = max(0, c1 - 16), cb = c1 - c0;
                if (tid < 32) {   // upper block, solved from its last unknown up
                    val_t v = (tid < cb) ? xs[c0 + tid] : vzero();
                    for (int c = cb - 1; c >= 0; --c) {
                        const val_t piv = A[(size_t)(c0 + c) * lda + c0 + c];
                        val_t xc = vshfl(v, c);
                        xc = vdiv(xc, piv);
                        if (tid == c) v = xc;
                        if (tid < c) vmul_sub(v, A[(size_t)(c0 + c) * lda + c0 + tid], xc);
                    }
                    if (tid < cb) xs[c0 + tid] = v;
                }
                __syncthreads();
                for (int r = tid; r < c0; r += 256) {
                    val_t acc = vzero();
                    for (int c = 0; c < cb; ++c) vmul_add(acc, A[(size_t)(c0 + c) * lda + r], xs[c0 + c]);
                    vsub(xs[r], acc);
                }
                __syncthreads();
            }
        }
        for (int r = tid; r < ns; r += 256) xk[r] = xs[r];
        __syncthreads();
    }
}

// x[rows below] -= L(below, k) x_k: CTA = 256 rows of one panel, thread = row (coalesced down the columns)
__global__ void __launch_bounds__(SOLVE_ROWS) solve_update_l_kernel(DeviceLU d, Batch b, val_t *x, int n, int nrhs)
{
    __shared__ val_t xs[MAX_NS_HELD];
    const int slot = find_slot(b.prefix, b.count, blockIdx.x);
    const NodeDesc nd = d.nodes[b.nodes[slot]];
    const int i = (int)(blockIdx.x - b.prefix[slot]) * SOLVE_ROWS + threadIdx.x;
    const int ns = nd.ns, lda = nd.nsupr;
    const val_t *L = d.val + nd.lval + ns;
    const int row = i < nd.m ? d.lrows[nd.lrow + ns + i] : 0;
    for (int rhs = 0; rhs < nrhs; ++rhs) {
        __syncthreads();
        for (int c = threadIdx.x; c < ns; c += SOLVE_ROWS) xs[c] = x[(size_t)rhs * n + nd.fsupc + c];
        __syncthreads();
        if (i < nd.m) {
            val_t acc = vzero();
#pragma unroll 8
            for (int c = 0; c < ns; ++c) vmul_add(acc, L[(size_t)c * lda + i], xs[c]);
            vatomic_sub(x + (size_t)rhs * n + row, acc);
        }
    }
}

// x_k -= U(k, cols) x[cols]: CTA = 256 packed columns of one U panel; warp w sweeps columns w, w+8, ..., lanes over rows
__global__ void __launch_bounds__(256) solve_update_u_kernel(DeviceLU d, Batch b, val_t *x, int n, int nrhs)
{
    __shared__ val_t part[8][MAX_NS_HELD];
    const int slot = find_slot(b.prefix, b.count, blockIdx.x);
    const NodeDesc nd = d.nodes[b.nodes[slot]];
    const int j0 = (int)(blockIdx.x - b.prefix[slot]) * SOLVE_ROWS, j1 = min(nd.ncols, j0 + SOLVE_ROWS);
    const int ns = nd.ns, warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const val_t *U = d.val + nd.uval;
    const int32_t *cols = d.ucols + nd.ucol;
    for (int rhs = 0; rhs < nrhs; ++rhs) {
        val_t acc[MAX_NS_HELD / 32];
#pragma unroll
        for (int t = 0; t < MAX_NS_HELD / 32; ++t) acc[t] = vzero();
        for (int j = j0 + warp; j < j1; j += 8) {
            const val_t xj = x[(size_t)rhs * n + cols[j]];
            const val_t *col = U + (size_t)j * ns;
#pragma unroll
            for (int t = 0; t < MAX_NS_HELD / 32; ++t) {
                const int r = t * 32 + lane;
                if (r < ns) vmul_add(acc[t], col[r], xj);
            }
        }
#pragma unroll
        for (int t = 0; t < MAX_NS_HELD / 32; ++t) {
            const int r = t * 32 + lane;
            if (r < ns) part[warp][r] = acc[t];
        }
        __syncthreads();
        for (int r = threadIdx.x; r < ns; r += 256) {
            val_t sum = vzero();
#pragma unroll
            for (int w = 0; w < 8; ++w) vadd(sum, part[w][r]);
            vatomic_sub(x + (size_t)rhs * n + nd.fsupc + r, sum);
        }
        __syncthreads();
    }
}

// keep / zero the entries of the supernodes in a node list (multi-GPU ownership masks)
__global__ void solve_mask_kernel(DeviceLU d, const int32_t *nodes, int count, val_t *x, int n, int nrhs, const val_t *src)
{
    for (int t = blockIdx.x; t < count; t += gridDim.x) {
        const NodeDesc nd = d.nodes[nodes[t]];
        for (int rhs = 0; rhs < nrhs; ++rhs)
            for (int r = threadIdx.x; r < nd.ns; r += blockDim.x)
                x[(size_t)rhs * n + nd.fsupc + r] = src ? src[(size_t)rhs * n + nd.fsupc + r] : vzero();
    }
}

// ---------------------------------------------------------------------------------------------------------------
// Device-side distribution (SURVEY 8f row N1): scatter P A P^T from a CSR copy in HBM straight into the L / U panels
// of the arena -- the job pddistribute3d (SRC/double/pddistribute3d.c:1357; pzdistribute3d in doublecomplex) does on
// the host, without the per-factor-entry host arrays and their H2D.  One thread per row of A; an entry (i, j) of the
// permuted matrix belongs to the L panel of supno(j) if i is at or below that supernode's first row, else to the U
// panel of supno(i).  `active[k]` = 0 for panels this rank does not hold or holds as zero-initialised replicated
// ancestors.
__global__ void fill_csr_kernel(DeviceLU d, int n, const int32_t *__restrict__ rowptr, const int32_t *__restrict__ colind,
                                const val_t *__restrict__ aval, const int32_t *__restrict__ perm, const int8_t *__restrict__ active,
                                int *err)
{
    const int r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= n) return;
    const int pi = perm[r];
    for (int p = rowptr[r]; p < rowptr[r + 1]; ++p) {
        const int pj = perm[colind[p]];
        const int ks = d.supno[pj];
        if (pi >= d.xsup[ks]) {                       // L panel of block column ks (diagonal block included)
            if (!active[ks]) continue;
            const NodeDesc *nd = d.nodes + ks;
            const int32_t *srow = d.lsrow + nd->lrow;
            const int q = lower_bound_i32(srow, nd->nsupr, pi);
            if (q >= nd->nsupr || srow[q] != pi) { atomicAdd(err, 1); continue; }
            d.val[nd->lval + (int64_t)(pj - nd->fsupc) * nd->nsupr + d.lspos[nd->lrow + q]] = aval[p];
        } else {                                      // U panel of block row supno(i)
            const int kr = d.supno[pi];
            if (!active[kr]) continue;
            const NodeDesc *nd = d.nodes + kr;
            const int32_t *uc = d.ucols + nd->ucol;
            const int q = lower_bound_i32(uc, nd->ncols, pj);
            if (q >= nd->ncols || uc[q] != pj) { atomicAdd(err, 1); continue; }
            d.val[nd->uval + (int64_t)q * nd->ns + (pi - nd->fsupc)] = aval[p];
        }
    }
}
int launch_fill_csr(const DeviceLU &d, int n, const int32_t *rowptr, const int32_t *colind, const val_t *aval, const int32_t *perm,
                    const int8_t *active, int *err, cudaStream_t s)
{
    fill_csr_kernel<<<(n + 127) / 128, 128, 0, s>>>(d, n, rowptr, colind, aval, perm, active, err);
    return 1;
}

int launch_solve_diag(const DeviceLU &d, const int32_t *nodes, int count, bool upper, val_t *x, int n, int nrhs, cudaStream_t s)
{
    if (count <= 0) return 0;
    if (upper) solve_diag_kernel<true><<<count, 256, 0, s>>>(d, nodes, x, n, nrhs);
    else solve_diag_kernel<false><<<count, 256, 0, s>>>(d, nodes, x, n, nrhs);
    return 1;
}
int launch_solve_update(const DeviceLU &d, const Batch &b, int64_t ctas, bool upper, val_t *x, int n, int nrhs, cudaStream_t s)
{
    if (b.count <= 0 || ctas <= 0) return 0;
    if (upper) solve_update_u_kernel<<<(unsigned)ctas, 256, 0, s>>>(d, b, x, n, nrhs);
    else solve_update_l_kernel<<<(unsigned)ctas, SOLVE_ROWS, 0, s>>>(d, b, x, n, nrhs);
    return 1;
}
int launch_solve_mask(const DeviceLU &d, const int32_t *nodes, int count, val_t *x, int n, int nrhs, const val_t *src, cudaStream_t s)
{
    if (count <= 0) return 0;
    solve_mask_kernel<<<std::min(count, 148 * 8), 128, 0, s>>>(d, nodes, count, x, n, nrhs, src);
    return 1;
}

}  // namespace SLU_NS
