// slu_api.cu -- C-ABI (include/slu_b200.h) and host orchestration of the B200 pdgstrf3d.
//
// The level loop mirrors pdgstrf3d (SRC/double/pdgstrf3d.c:333-385): for every Z-tree level this
// rank takes part in, factor its elimination sub-forest, combining the replicated ancestor copies
// along Z.  Inside a forest the reference walks supernodes one at a time with a look-ahead pipeline
// (dsparseTreeFactor_ASYNC, SRC/double/dtreeFactorization.c:295-716); here all supernodes of one
// topological level are processed by a handful of batched kernel launches (diagonal LU -> panel
// solves -> destination maps -> fused GEMM+scatter), the whole L/U resident in HBM, with
//   * look-ahead: panel work + "urgent" Schur tiles on a high-priority stream, the bulk on a second one;
//   * multi-GPU: either the reference's pairwise ancestor reduction, or (default) cooperative ancestors --
//     one NCCL all-reduce per topological level over the Z group, Schur tiles dealt round-robin;
//   * Pr x Pc > 1: block-cyclic pieces in, whole panels replicated per layer, same cooperative schedule;
//   * slu_b200_factor_host: D2H of every level overlapped with the factorization of the upper levels.
// No host compute touches the values.
//
// This file is compiled twice (see slu_device.cuh): as is for double, and through slu_api_z.cu with SLU_COMPLEX for
// doublecomplex, where the exported names become slu_b200_z_* / pzgstrf3d_b200 and the value pointers of the view
// are read as (re, im) pairs.
#include "slu_b200.h"
#include "slu_device.cuh"

#ifdef SLU_COMPLEX
#define slu_b200_handle_s slu_b200_zhandle_s
#define slu_b200_handle_t slu_b200_zhandle_t
#define slu_b200_create slu_b200_z_create
#define slu_b200_upload slu_b200_z_upload
#define slu_b200_factor slu_b200_z_factor
#define slu_b200_factor_host slu_b200_z_factor_host
#define slu_b200_download slu_b200_z_download
#define slu_b200_get_stats slu_b200_z_get_stats
#define slu_b200_destroy slu_b200_z_destroy
#define slu_b200_plan slu_b200_z_plan
#define slu_b200_solve slu_b200_z_solve
#define slu_b200_fill_csr slu_b200_z_fill_csr
#define pdgstrf3d_b200 pzgstrf3d_b200
#define slu_b200_k_diag_lu slu_b200_z_k_diag_lu
#define slu_b200_k_trsm_l slu_b200_z_k_trsm_l
#define slu_b200_k_trsm_u slu_b200_z_k_trsm_u
#define slu_b200_k_gemm_sub slu_b200_z_k_gemm_sub
#endif

#include <dlfcn.h>
#include <omp.h>

#include <algorithm>
#include <array>
#include <map>
#include <mutex>
#include <chrono>
#include <climits>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <string>
#include <vector>

using namespace SLU_NS;

// one error string for both precisions (slu_b200_last_error)
#ifdef SLU_COMPLEX
extern thread_local std::string slu_b200_err_storage;
#else
thread_local std::string slu_b200_err_storage;
#endif
#define g_err slu_b200_err_storage

namespace {

int fail(const char *fmt, ...)
{
    char buf[1024];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    g_err = buf;
    return -1;
}
#define CU(call)                                                                                   \
    do {                                                                                           \
        cudaError_t e_ = (call);                                                                   \
        if (e_ != cudaSuccess) return fail("%s:%d %s: %s", __FILE__, __LINE__, #call, cudaGetErrorString(e_)); \
    } while (0)

double now_s()
{
    return std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count();
}

constexpr int BC_HEADER = 2, LB_DESCRIPTOR = 2, BR_HEADER = 3, UB_DESCRIPTOR = 2;

// ---- NCCL through dlopen: no link-time dependency, the caller's (torch's) libnccl.so.2 is reused ---
}  // namespace

// the by-value ncclUniqueId argument of ncclCommInitRank needs a real 128-byte struct type
struct slu_nccl_id { char internal[128]; };

namespace {
struct NcclApi {
    void *so = nullptr;
    int (*GetUniqueId)(slu_nccl_id *) = nullptr;
    int (*CommInitRank)(void **, int, slu_nccl_id, int) = nullptr;
    int (*CommDestroy)(void *) = nullptr;
    int (*Send)(const void *, size_t, int, int, void *, cudaStream_t) = nullptr;
    int (*Recv)(void *, size_t, int, int, void *, cudaStream_t) = nullptr;
    int (*AllReduce)(const void *, void *, size_t, int, int, void *, cudaStream_t) = nullptr;
    int (*CommSplit)(void *, int, int, void **, void *) = nullptr;
    int (*AllGather)(const void *, void *, size_t, int, void *, cudaStream_t) = nullptr;
    const char *(*GetErrorString)(int) = nullptr;
    bool load()
    {
        if (so) return true;
        const char *names[] = {getenv("SLU_B200_NCCL"), "libnccl.so.2", "libnccl.so"};
        for (const char *n : names) {
            if (!n) continue;
            so = dlopen(n, RTLD_NOW | RTLD_GLOBAL);
            if (so) break;
        }
        if (!so) return false;
        GetUniqueId = (decltype(GetUniqueId))dlsym(so, "ncclGetUniqueId");
        CommInitRank = (decltype(CommInitRank))dlsym(so, "ncclCommInitRank");
        CommDestroy = (decltype(CommDestroy))dlsym(so, "ncclCommDestroy");
        Send = (decltype(Send))dlsym(so, "ncclSend");
        Recv = (decltype(Recv))dlsym(so, "ncclRecv");
        AllReduce = (decltype(AllReduce))dlsym(so, "ncclAllReduce");
        CommSplit = (decltype(CommSplit))dlsym(so, "ncclCommSplit");
        AllGather = (decltype(AllGather))dlsym(so, "ncclAllGather");
        GetErrorString = (decltype(GetErrorString))dlsym(so, "ncclGetErrorString");
        return GetUniqueId && CommInitRank && CommDestroy && Send && Recv && AllReduce;
    }
} g_nccl;
constexpr int NCCL_INT32 = 2, NCCL_FLOAT64 = 8, NCCL_SUM = 0, NCCL_MIN = 3;
#define NC(call)                                                                                   \
    do {                                                                                           \
        int r_ = (call);                                                                           \
        if (r_ != 0) return fail("%s:%d %s: NCCL error %d %s", __FILE__, __LINE__, #call, r_,      \
                                 g_nccl.GetErrorString ? g_nccl.GetErrorString(r_) : "");          \
    } while (0)

// NCCL communicators outlive a factorization, as the reference's MPI communicators do (superlu_gridinit3d creates
// them once, pdgstrf3d only uses them): the 128-byte NCCL id names the clique, and the world communicator plus the
// per-Z-level group communicators built from it are cached per process under (id, grid shape, my coordinates).
// Repeated pdgstrf3d_b200 calls with the same id reuse them; slu_b200_comm_cache_clear() destroys them.
struct CommSet {
    void *comm = nullptr;
    std::vector<void *> gcomm;
};
std::mutex g_comm_mu;
std::map<std::string, CommSet> g_comm_cache;

// slu_b200_plan: run the analysis without touching a device -- buffers record their sizes only
thread_local bool g_plan_only = false;

template <class T>
struct DevBuf {
    T *p = nullptr;
    size_t n = 0;
    int alloc(size_t count)
    {
        release();
        n = count;
        if (g_plan_only) return 0;
        if (count == 0) count = 1;
        cudaError_t e = cudaMalloc((void **)&p, count * sizeof(T));
        if (e != cudaSuccess) return fail("cudaMalloc(%zu bytes): %s", count * sizeof(T), cudaGetErrorString(e));
        return 0;
    }
    int upload(const std::vector<T> &h)
    {
        if (alloc(h.size())) return -1;
        if (g_plan_only) return 0;
        if (!h.empty()) CU(cudaMemcpy(p, h.data(), h.size() * sizeof(T), cudaMemcpyHostToDevice));
        return 0;
    }
    void release() { if (p) cudaFree(p); p = nullptr; n = 0; }
    size_t bytes() const { return n * sizeof(T); }
    DevBuf() = default;
    DevBuf(const DevBuf &) = delete;
    DevBuf &operator=(const DevBuf &) = delete;
    ~DevBuf() { release(); }   // the CU()/NC() early returns must not leak HBM
};

struct EventSet {            // timing events with the same guarantee
    cudaEvent_t e[6] = {};
    int create() { for (auto &x : e) if (cudaEventCreate(&x) != cudaSuccess) return -1; return 0; }
    ~EventSet() { for (auto x : e) if (x) cudaEventDestroy(x); }
    cudaEvent_t &operator[](int i) { return e[i]; }
};

struct LevelPlan {
    int zlvl = 0, count = 0, max_ns = 0, atomic = 1;
    int64_t nodes_off = 0;
    int64_t trsml_prefix = 0, trsml_ctas = 0, trsmu_prefix = 0, trsmu_ctas = 0, setup_prefix = 0, setup_ctas = 0;
    int64_t inv_prefix = 0, inv_ctas = 0;
    int64_t urg_prefix = 0, urg_ctas = 0, bulk_prefix = 0, bulk_ctas = 0;  // look-ahead split of the big batch
    int64_t slab_begin = 0, slab_end = 0;  // val range of this level's panels (contiguous in cooperative forests)
    int big_count = 0, small_count = 0;
    int64_t big_nodes = 0, big_prefix = 0, big_ctas = 0, small_nodes = 0, small_prefix = 0, small_ctas = 0;
    // tcgen05 path: the wide supernodes of the level (slu_ozaki.cu)
    int tc_count = 0;
    int64_t tc_nodes = 0, tc_prefix = 0, tc_ctas = 0, tc_urg_prefix = 0, tc_urg_ctas = 0, tc_bulk_prefix = 0, tc_bulk_ctas = 0;
    int64_t tc_p_rt = 0, tc_n_rt = 0, tc_p_ak = 0, tc_n_ak = 0, tc_p_b = 0, tc_n_b = 0;
    int64_t sl_prefix = 0, sl_ctas = 0, su_prefix = 0, su_ctas = 0;   // triangular solve: 256-row / 256-column tiles
};

}  // namespace

struct slu_b200_handle_s {
    slu_b200_lu_view_t view;
    slu_b200_options_t opt;
    int nsupers = 0, n = 0, max_lvl = 1;
    std::vector<int32_t> xsup, my_tree, my_zero;
    std::vector<NodeDesc> nodes;          // host copy
    std::vector<std::vector<int32_t>> znodes;  // held nodes per Z level, arena order
    std::vector<int64_t> chunk_start;     // val offsets per Z level (L part, U part interleaved): [maxLvl+1]
    std::vector<int64_t> sky_len;         // skyline nnz of each held U panel (host side)
    std::vector<char> u_full;             // 1 if the skyline of U panel k equals its dense-packed form
    std::vector<LevelPlan> levels;
    // device
    DevBuf<val_t> val, stage, d_inv;
    DevBuf<NodeDesc> d_nodes;
    DevBuf<int32_t> d_xsup, d_supno, d_lrows, d_lsrow, d_lspos, d_ucols, d_ufst, d_useg, d_pool_i32, d_lrel, d_urel;
    DevBuf<int64_t> d_pool_i64;
    DevBuf<LBlk> d_lblk;
    DevBuf<UBlk> d_ublk;
    DevBuf<RowInfo> d_rowinfo;
    DevBuf<ColInfo> d_colinfo;
    DevBuf<int8_t> d_oz_i8;               // tcgen05 path: int8 slice workspace (two level parities)
    DevBuf<double> d_oz_scale;
    DevBuf<int> d_oz_rexp;
    int tc_slices = 0, tc_min_ns = 0;     // 0 slices: tcgen05 path off
    bool tc_force_off = false, tc_alloc_failed = false;   // slice workspace did not fit: analysed again without the tcgen05 path
    int tc_nonatomic = 0;                 // plain load/store scatter for destinations only one supernode of a level updates
    DevBuf<val_t> d_x, d_x2;              // triangular solve: right-hand sides / solution
    std::vector<int64_t> z_nodes_off;     // [zl] offset into d_pool_i32 of the forest's node list (solve masks)
    bool factored = false;
    DevBuf<int> d_flags;                  // [0]=info [1]=err
    DevBuf<unsigned long long> d_tiny;
    DeviceLU dev{};
    cudaStream_t stream = nullptr, stream2 = nullptr;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    std::vector<cudaEvent_t> ev_panel, ev_bulk;
    cudaStream_t s_down = nullptr;                       // overlapped D2H (slu_b200_factor_host)
    cudaStream_t s_up = nullptr;                         // overlapped H2D (options.reserved[3])
    std::vector<cudaEvent_t> ev_up;                      // [li] level li's panels have arrived in the arena
    std::vector<int32_t> h_pool_i32;                     // host copy of the level node lists
    bool grouped = false;                                // every forest laid out level by level
    std::vector<UpSeg> h_segs;                           // download chunks (arena offset, -, length), by release level
    std::vector<val_t *> h_seg_host;                     // host address of each chunk
    std::vector<std::array<int64_t, 2>> lvl_segs;         // [li] -> [first, last) chunk released after level li
    bool pipe_ready = false;
    int64_t ws_max[4] = {0, 0, 0, 0};
    void *comm = nullptr;
    bool coop = false;                    // cooperative ancestors: all ranks of a Z group factor the shared forest
    int P2 = 1;                           // nprow * npcol: ranks of one layer (2D input: panels replicated per layer)
    void *lcomm = nullptr;                // communicator of my layer (structure exchange)
    std::vector<const slu_int *> Lidx, Uidx;        // [nsupers] index arrays of the FULL panels
    std::vector<std::vector<slu_int>> fullL, fullU; // their storage when merged from the 2D pieces
    struct Piece { int64_t dev; val_t *host; int64_t width, height, spitch, dpitch; };
    std::vector<Piece> pieces;            // my local blocks <-> their place in the replicated panels
    std::vector<LBlk> h_lblk;
    std::vector<UBlk> h_ublk;
    std::vector<void *> gcomm;            // [zl] communicator of my Z group at level zl (2^zl ranks)
    slu_b200_stats_t st{};
    bool uploaded = false;
};

namespace {

int device_setup(const slu_b200_options_t *opt)
{
    if (opt->device >= 0) CU(cudaSetDevice(opt->device));
    CU(cudaFree(0));
    return 0;
}

// ------------------------------------------------------------------------------------------------
// analysis: parse the reference index arrays, lay out HBM, plan the level batches
// ------------------------------------------------------------------------------------------------
int analyze(slu_b200_handle_s *H)
{
    const slu_b200_lu_view_t &v = H->view;
    const int nsupers = v.nsupers, n = v.n;
    if (H->P2 > 1 && !H->coop)
        return fail("Pr x Pc > 1 needs the cooperative schedule (options.reserved[1] must be 0)");
    if (v.npdep < 1 || (v.npdep & (v.npdep - 1))) return fail("npdep must be a power of two");
    int max_lvl = 1;
    while ((1 << (max_lvl - 1)) < v.npdep) ++max_lvl;
    if (v.maxLvl != max_lvl) return fail("maxLvl %d does not match npdep %d", v.maxLvl, v.npdep);
    if (v.nforests != (1 << max_lvl) - 1) return fail("nforests must be 2^maxLvl - 1");
    H->nsupers = nsupers; H->n = n; H->max_lvl = max_lvl;
    H->xsup.assign(v.xsup, v.xsup + nsupers + 1);
    H->my_tree.assign(v.myTreeIdxs, v.myTreeIdxs + max_lvl);
    H->my_zero.assign(v.myZeroTrIdxs, v.myZeroTrIdxs + max_lvl);
    const std::vector<int32_t> &xsup = H->xsup;
    std::vector<int32_t> supno((size_t)n);
    for (int k = 0; k < nsupers; ++k) {
        if (xsup[k + 1] - xsup[k] > MAX_NS_HELD) return fail("supernode %d wider than %d columns is not supported", k, MAX_NS_HELD);
        for (int c = xsup[k]; c < xsup[k + 1]; ++c) supno[c] = k;
    }

    const bool timing = getenv("SLU_B200_TIMING") != nullptr;
    double tmark = now_s();
    auto lap = [&](const char *what) { if (timing) { double t = now_s(); fprintf(stderr, "analyze: %-28s %.3f s\n", what, t - tmark); tmark = t; } };
    H->nodes.assign(nsupers, NodeDesc{});
    H->znodes.assign(max_lvl, {});
    std::vector<int> forest_of(nsupers, -1), zl_of(nsupers, -1);
    for (int zl = 0; zl < max_lvl; ++zl) {
        const slu_b200_forest_t &f = v.forests[H->my_tree[zl]];
        for (int t = 0; t < f.nNodes; ++t) {
            int k = f.nodeList[t];
            if (k < 0 || k >= nsupers || zl_of[k] != -1) return fail("bad forest node list");
            zl_of[k] = zl;
            H->znodes[zl].push_back(k);
        }
    }

    // topological levels inside each forest (a supernode precedes every block it updates); the node lists are
    // valid elimination orders, so one sweep suffices
    std::vector<int> lev(nsupers, 0);
    for (int zl = 0; zl < max_lvl; ++zl)
        for (int k : H->znodes[zl]) {
            const slu_int *li = H->Lidx[k], *ui = H->Uidx[k];
            if (!li) return fail("supernode %d of my forest has no L panel", k);
            int w = BC_HEADER;
            for (int b = 0; b < li[0]; ++b) {
                int t = li[w];
                if (b > 0 && t >= 0 && t < nsupers && zl_of[t] == zl) lev[t] = std::max(lev[t], lev[k] + 1);
                w += LB_DESCRIPTOR + li[w + 1];
            }
            if (!ui) continue;
            int u = BR_HEADER;
            for (int b = 0; b < ui[0]; ++b) {
                int t = ui[u];
                if (t < 0 || t >= nsupers) return fail("U panel %d: bad block id", k);
                int jns = xsup[t + 1] - xsup[t];
                bool nonempty = false;
                for (int c = 0; c < jns && !nonempty; ++c) nonempty = ui[u + UB_DESCRIPTOR + c] < xsup[k + 1];
                if (nonempty && zl_of[t] == zl) lev[t] = std::max(lev[t], lev[k] + 1);
                u += UB_DESCRIPTOR + jns;
            }
        }
    lap("forests + topological levels");
    // cooperative ancestors (world_size > 1): every rank of a Z group factors the shared forest; its panels are
    // laid out level by level so that the panels due at one topological level are one contiguous slab
    const bool coop = H->coop;
    // options.reserved[3] (overlapped upload): the same level-by-level layout for every forest, so that the panels
    // are needed in arena order
    H->grouped = H->opt.reserved[3] && H->P2 == 1;
    if (coop || H->grouped)
        for (int zl = ((H->P2 > 1 || H->grouped) ? 0 : 1); zl < max_lvl; ++zl)
            std::stable_sort(H->znodes[zl].begin(), H->znodes[zl].end(), [&](int a, int b) { return lev[a] < lev[b]; });

    // pass 1: sizes and offsets.  Three sweeps over the held supernodes in arena order: (a) parallel -- count rows,
    // blocks and non-empty U columns of each panel; (b) serial -- prefix sums give every panel its place in the value
    // arena and in the index arenas; (c) parallel -- fill the index arenas, cross maps and flop counts.
    std::vector<int32_t> lrows, lsrow, lspos, ucols, ufst, useg;
    std::vector<LBlk> lblk;
    std::vector<UBlk> ublk;
    H->sky_len.assign(nsupers, 0);
    H->u_full.assign(nsupers, 1);
    H->chunk_start.assign(max_lvl + 1, 0);
    int64_t voff = 0;
    double ops = 0, ops_schur = 0, bytes_schur = 0;
    int64_t nnz_l = 0, nnz_u = 0;
    // arena order: per Z level, per group (the whole forest, or one topological level of a cooperatively factored /
    // grouped forest), first the L panels of the group, then its U panels
    std::vector<int32_t> order;                       // held supernodes in the order their L panels are laid out
    std::vector<std::pair<int64_t, int64_t>> groups;  // [begin, end) into order
    std::vector<int> group_zl;
    order.reserve(nsupers);
    for (int zl = 0; zl < max_lvl; ++zl) {
        const bool split = (coop && (zl >= 1 || H->P2 > 1)) || H->grouped;
        int64_t g0 = (int64_t)order.size();
        for (size_t t = 0; t < H->znodes[zl].size(); ++t) {
            const int k = H->znodes[zl][t];
            if (split && t > 0 && lev[H->znodes[zl][t - 1]] != lev[k]) {
                groups.emplace_back(g0, (int64_t)order.size()); group_zl.push_back(zl);
                g0 = (int64_t)order.size();
            }
            order.push_back(k);
        }
        if ((int64_t)order.size() > g0) { groups.emplace_back(g0, (int64_t)order.size()); group_zl.push_back(zl); }
    }
    const int64_t nheld = (int64_t)order.size();
    std::vector<int32_t> cnt_ucols(nheld, 0), cnt_ublk(nheld, 0);
    std::vector<char> bad(1, 0);
    std::string badmsg;
    auto flag = [&](const char *fmt, int a1, int a2 = 0, int a3 = 0) {
#pragma omp critical(slu_analyze_err)
        if (!bad[0]) { char buf[256]; snprintf(buf, sizeof buf, fmt, a1, a2, a3); badmsg = buf; bad[0] = 1; }
    };
    // a handful of threads is enough (and 8 ranks of one box share the cores)
    const int nth = std::max(1, std::min(omp_get_max_threads(), 16));
    // (a) counts
#pragma omp parallel for schedule(dynamic, 64) num_threads(nth)
    for (int64_t t = 0; t < nheld; ++t) {
        const int k = order[t];
        const slu_int *li = H->Lidx[k], *ui = H->Uidx[k];
        NodeDesc &nd = H->nodes[k];
        nd.held = 1; nd.fsupc = xsup[k]; nd.ns = xsup[k + 1] - xsup[k];
        nd.nsupr = li[1]; nd.m = nd.nsupr - nd.ns;
        const int nblk = li[0];
        if (nblk < 1 || li[BC_HEADER] != k || li[BC_HEADER + 1] != nd.ns) { flag("L panel %d: the diagonal block must come first and be full", k); continue; }
        nd.nlb = nblk - 1;
        if (!ui) continue;
        const int nb = ui[0], klst = xsup[k + 1];
        int u = BR_HEADER, ncols = 0, nub = 0;
        for (int bq = 0; bq < nb; ++bq) {
            const int jb = ui[u];
            if (jb < 0 || jb >= nsupers) { flag("U panel %d: bad block id", k); break; }
            const int jns = xsup[jb + 1] - xsup[jb];
            int c2 = 0;
            for (int c = 0; c < jns; ++c) c2 += ui[u + UB_DESCRIPTOR + c] < klst;
            ncols += c2; nub += c2 > 0;
            u += UB_DESCRIPTOR + jns;
        }
        cnt_ucols[t] = ncols; cnt_ublk[t] = nub;
    }
    if (bad[0]) return fail("%s", badmsg.c_str());
    // (b) offsets
    std::vector<int64_t> off_lrow(nheld + 1, 0), off_lblk(nheld + 1, 0), off_ucol(nheld + 1, 0), off_ublk(nheld + 1, 0);
    for (int64_t t = 0; t < nheld; ++t) {
        const NodeDesc &nd = H->nodes[order[t]];
        off_lrow[t + 1] = off_lrow[t] + nd.nsupr;
        off_lblk[t + 1] = off_lblk[t] + nd.nlb;
        off_ucol[t + 1] = off_ucol[t] + cnt_ucols[t];
        off_ublk[t + 1] = off_ublk[t] + cnt_ublk[t];
    }
    {
        int last_zl = -1;
        for (size_t g = 0; g < groups.size(); ++g) {
            if (group_zl[g] != last_zl) { for (int z = last_zl + 1; z <= group_zl[g]; ++z) H->chunk_start[z] = voff; last_zl = group_zl[g]; }
            for (int64_t t = groups[g].first; t < groups[g].second; ++t) {
                NodeDesc &nd = H->nodes[order[t]];
                nd.lval = voff; voff += (int64_t)nd.nsupr * nd.ns;
                nnz_l += (int64_t)nd.nsupr * nd.ns;
            }
            for (int64_t t = groups[g].first; t < groups[g].second; ++t) {
                NodeDesc &nd = H->nodes[order[t]];
                nd.ncols = cnt_ucols[t];
                nd.uval = voff; voff += (int64_t)nd.ns * nd.ncols;
                nnz_u += (int64_t)nd.ns * nd.ncols;
            }
        }
        for (int z = last_zl + 1; z < max_lvl; ++z) H->chunk_start[z] = voff;
    }
    lrows.resize((size_t)off_lrow[nheld]); lsrow.resize(lrows.size()); lspos.resize(lrows.size());
    ucols.resize((size_t)off_ucol[nheld]); ufst.resize(ucols.size()); useg.resize(ucols.size());
    lblk.resize((size_t)off_lblk[nheld]); ublk.resize((size_t)off_ublk[nheld]);
    // (c) fill
#pragma omp parallel reduction(+ : ops, ops_schur, bytes_schur) num_threads(nth)
    {
        std::vector<std::pair<int32_t, int32_t>> tmp;
#pragma omp for schedule(dynamic, 32)
        for (int64_t t = 0; t < nheld; ++t) {
            const int k = order[t];
            const int zl = zl_of[k];
            const slu_int *li = H->Lidx[k];
            NodeDesc &nd = H->nodes[k];
            nd.lrow = off_lrow[t]; nd.lblk = off_lblk[t]; nd.ucol = off_ucol[t]; nd.ublk = off_ublk[t];
            const int nblk = li[0];
            {
                int w = BC_HEADER, row0 = 0, last_ib = -1;
                int64_t lr = nd.lrow, lbq = nd.lblk;
                bool okp = true;
                tmp.clear();
                for (int bq = 0; bq < nblk && okp; ++bq) {
                    int ib = li[w], nb = li[w + 1];
                    if (ib <= last_ib) { flag("L panel %d: row blocks are not in ascending order", k); okp = false; break; }
                    last_ib = ib;
                    if (row0 + nb > nd.nsupr) { flag("L panel %d: row count mismatch", k); okp = false; break; }
                    for (int q = 0; q < nb; ++q) {
                        int r = li[w + 2 + q];
                        if (r < xsup[ib] || r >= xsup[ib + 1]) { flag("L panel %d: row %d outside block %d", k, r, ib); okp = false; break; }
                        if (bq == 0 && r != xsup[k] + q) { flag("L panel %d: diagonal block rows must be sorted", k); okp = false; break; }
                        tmp.emplace_back(r, row0 + q);
                        lrows[lr++] = r;
                    }
                    if (bq > 0) lblk[lbq++] = LBlk{ib, row0 - nd.ns, nb, 0, 0};
                    row0 += nb;
                    w += LB_DESCRIPTOR + nb;
                }
                if (!okp) continue;
                if (row0 != nd.nsupr) { flag("L panel %d: row count mismatch", k); continue; }
                std::sort(tmp.begin(), tmp.end());
                for (size_t q = 0; q < tmp.size(); ++q) { lsrow[nd.lrow + q] = tmp[q].first; lspos[nd.lrow + q] = tmp[q].second; }
            }
            const slu_int *ui = H->Uidx[k];
            int ldu = 0;
            double utrsm = 0;
            if (ui) {
                const int nb = ui[0], klst = xsup[k + 1];
                int u = BR_HEADER, seg = 0, last_jb = k, col = 0;
                int64_t uc = nd.ucol, ubq = nd.ublk;
                bool oku = true, full = true;
                for (int bq = 0; bq < nb && oku; ++bq) {
                    int jb = ui[u];
                    if (jb <= last_jb || jb >= nsupers) { flag("U panel %d: column blocks are not ascending", k); oku = false; break; }
                    last_jb = jb;
                    int jns = xsup[jb + 1] - xsup[jb], col0 = col, cnt = 0;
                    for (int c = 0; c < jns; ++c) {
                        int fst = ui[u + UB_DESCRIPTOR + c];
                        if (fst >= klst) continue;
                        if (fst < xsup[k]) { flag("U panel %d: fstnz below the supernode", k); oku = false; break; }
                        ucols[uc] = xsup[jb] + c; ufst[uc] = fst; useg[uc] = seg; ++uc;
                        int len = klst - fst;
                        seg += len; ldu = std::max(ldu, len);
                        utrsm += (double)len * (len + 1);
                        if (len != nd.ns) full = false;
                        ++cnt;
                    }
                    if (cnt) ublk[ubq++] = UBlk{jb, col0, cnt, 0, 0};
                    col += cnt;
                    u += UB_DESCRIPTOR + jns;
                }
                if (!oku) continue;
                if (seg != ui[1]) { flag("U panel %d: nnz mismatch (%d vs %d)", k, seg, ui[1]); continue; }
                H->sky_len[k] = seg;
                H->u_full[k] = full ? 1 : 0;
            }
            nd.nub = cnt_ublk[t];
            // cross maps: colstart per L block, rowstart per U block
            const int32_t *ucp = ucols.data() + nd.ucol;
            int64_t uoff = 0;
            for (int bq = 0; bq < nd.nlb; ++bq) {
                LBlk &lb = lblk[nd.lblk + bq];
                lb.colstart = (int)(std::lower_bound(ucp, ucp + nd.ncols, xsup[lb.ib + 1]) - ucp);
                lb.urel_off = uoff;
                uoff += nd.ncols - lb.colstart;
            }
            nd.urel_total = uoff;
            int64_t loff = 0;
            int q0 = 0;                                   // both block lists ascend: one merge sweep
            for (int bq = 0; bq < nd.nub; ++bq) {
                UBlk &ub = ublk[nd.ublk + bq];
                while (q0 < nd.nlb && lblk[nd.lblk + q0].ib < ub.jb) ++q0;
                ub.rowstart = q0 < nd.nlb ? lblk[nd.lblk + q0].row0 : nd.m;
                ub.lrel_off = loff;
                loff += nd.m - ub.rowstart;
            }
            nd.lrel_total = loff;
            // flops in the reference's accounting
            double diag = 0;
#ifdef SLU_COMPLEX
            for (int j = 0; j < nd.ns; ++j) { double r = nd.ns - j - 1; diag += (6 * r + 10) + 8 * r * r; }  // pzgstrf2.c:578,590
#else
            for (int j = 0; j < nd.ns; ++j) { double r = nd.ns - j - 1; diag += r + 2 * r * r; }
#endif
            double sch = 2.0 * nd.m * (double)ldu * nd.ncols;
            if (H->my_zero[zl]) continue;  // replicated ancestor copy: counted by its owner layer only
            if (H->P2 > 1 && (k % v.nprow != v.myrow || k % v.npcol != v.mycol)) continue;  // ... and by the diagonal owner
            ops += diag + utrsm + sch;
            ops_schur += sch;
            bytes_schur += VAL_DOUBLES * (8.0 * ((double)nd.m * nd.ns + (double)nd.ns * nd.ncols) + 16.0 * nd.m * (double)nd.ncols) +
                           4.0 * (nd.m + nd.ncols);
        }
    }
    if (bad[0]) return fail("%s", badmsg.c_str());
    H->chunk_start[max_lvl] = voff;
    lap("pass 1 (index arrays)");

    // every destination of a held supernode must be held too
    for (int zl = 0; zl < max_lvl; ++zl)
        for (int k : H->znodes[zl]) {
            const NodeDesc &nd = H->nodes[k];
            for (int b = 0; b < nd.nlb; ++b)
                if (!H->nodes[lblk[nd.lblk + b].ib].held) return fail("supernode %d updates block row %d which this rank does not hold", k, lblk[nd.lblk + b].ib);
            for (int b = 0; b < nd.nub; ++b)
                if (!H->nodes[ublk[nd.ublk + b].jb].held) return fail("supernode %d updates block column %d which this rank does not hold", k, ublk[nd.ublk + b].jb);
        }

    // level batches
    std::vector<int32_t> seen_by(nsupers, -1), stamp(nsupers, -1), ndest(nsupers, 0);
    std::vector<int32_t> pool_i32;
    std::vector<int64_t> pool_i64;
    int64_t ws_row_max = 0, ws_col_max = 0, ws_lrel_max = 0, ws_urel_max = 0, ws_inv_max = 0;
    int64_t ws_oz_i8_max = 0, ws_oz_s_max = 0;
    double ops_tc = 0;
#ifndef SLU_COMPLEX
    // tcgen05 path (slu_ozaki.cu): options.reserved[4] = int8 slices per operand (0: default, < 0: off),
    // options.reserved[5] = narrowest supernode that takes it (0: default)
    H->tc_slices = H->opt.reserved[4] < 0 ? 0 : (H->opt.reserved[4] == 0 ? (OZ_DEFAULT_ON ? OZ_DEFAULT_SLICES : 0) : std::min(8, std::max(5, (int)H->opt.reserved[4])));
    H->tc_min_ns = H->opt.reserved[5] > 0 ? H->opt.reserved[5] : OZ_DEFAULT_MIN_NS;
    if (getenv("SLU_B200_TC_SLICES")) { int v = atoi(getenv("SLU_B200_TC_SLICES")); H->tc_slices = v <= 0 ? 0 : std::min(8, std::max(5, v)); }
    if (getenv("SLU_B200_TC_MIN_NS")) H->tc_min_ns = std::max(1, atoi(getenv("SLU_B200_TC_MIN_NS")));
    if (H->tc_force_off) H->tc_slices = 0;
    H->tc_nonatomic = getenv("SLU_B200_TC_NONATOMIC") ? atoi(getenv("SLU_B200_TC_NONATOMIC")) : (OZ_NONATOMIC_DEFAULT ? 1 : 0);
#endif
    H->levels.clear();
    for (int zl = 0; zl < max_lvl; ++zl) {
        int maxlev = -1;
        for (int k : H->znodes[zl]) maxlev = std::max(maxlev, lev[k]);
        std::vector<std::vector<int32_t>> by(maxlev + 1);
        for (int k : H->znodes[zl]) by[lev[k]].push_back(k);
        for (auto &nodes : by) {
            if (nodes.empty()) continue;
            LevelPlan L;
            L.zlvl = zl; L.count = (int)nodes.size(); L.atomic = 1;  // RED.ADD.F64 beats a load/store read-modify-write here (profiles/r01_notes.md)
            L.nodes_off = (int64_t)pool_i32.size();
            pool_i32.insert(pool_i32.end(), nodes.begin(), nodes.end());
            // which destination panels are updated by MORE than one supernode of this level?  Only those need atomic
            // scatters; an exclusive destination is updated tile-disjointly by its single source (slu_ozaki.cu).
            for (int k : nodes) {
                const NodeDesc &nd = H->nodes[k];
                if (nd.m <= 0 || nd.ncols <= 0) continue;
                auto touch = [&](int t) {
                    if (seen_by[t] == k) return;
                    seen_by[t] = k;
                    if (stamp[t] != (int)H->levels.size()) { stamp[t] = (int)H->levels.size(); ndest[t] = 0; }
                    ++ndest[t];
                };
                for (int q = 0; q < nd.nlb; ++q) touch(lblk[nd.lblk + q].ib);
                for (int q = 0; q < nd.nub; ++q) touch(ublk[nd.ublk + q].jb);
            }
            for (int k : nodes) {
                const NodeDesc &nd = H->nodes[k];
                if (nd.m <= 0 || nd.ncols <= 0) continue;
                for (int q = 0; q < nd.nlb; ++q) { LBlk &lb = lblk[nd.lblk + q]; lb.shared = ndest[lb.ib] >= 2; }
                for (int q = 0; q < nd.nub; ++q) { UBlk &ub = ublk[nd.ublk + q]; ub.shared = ndest[ub.jb] >= 2; }
            }
            std::vector<int32_t> big, small, tc;
            std::vector<int64_t> p_l{0}, p_u{0}, p_s{0}, p_big{0}, p_small{0}, p_inv{0}, p_urg{0}, p_bulk{0};
            std::vector<int64_t> p_tc{0}, p_tc_urg{0}, p_tc_bulk{0}, p_tc_rt{0}, p_tc_ak{0}, p_tc_b{0}, p_sl{0}, p_su{0};
            int64_t wr = 0, wc = 0, wl = 0, wu = 0, woz = 0, wozs = 0;
            L.slab_begin = INT64_MAX;
            for (int k : nodes) {
                NodeDesc &nd = H->nodes[k];
                L.slab_begin = std::min(L.slab_begin, nd.lval);
                L.slab_end = std::max(L.slab_end, std::max(nd.lval + (int64_t)nd.nsupr * nd.ns, nd.uval + (int64_t)nd.ns * nd.ncols));
                L.max_ns = std::max(L.max_ns, nd.ns);
                const int strip = trsm_strip_of(nd.ns);
                p_l.push_back(p_l.back() + (nd.m + strip - 1) / strip);
                p_u.push_back(p_u.back() + (nd.ncols + strip - 1) / strip);
                p_sl.push_back(p_sl.back() + (nd.m + 255) / 256);
                p_su.push_back(p_su.back() + (nd.ncols + 255) / 256);
                nd.ws_inv = p_inv.back() * 512;
                p_inv.push_back(p_inv.back() + (nd.ns + 15) / 16);
                bool has_schur = nd.m > 0 && nd.ncols > 0;
                int64_t tasks = has_schur ? (int64_t)nd.m + nd.ncols + nd.lrel_total + nd.urel_total : 0;
                p_s.push_back(p_s.back() + (tasks + SETUP_THREADS - 1) / SETUP_THREADS);
                nd.ws_row = wr; nd.ws_col = wc; nd.ws_lrel = wl; nd.ws_urel = wu;
                if (has_schur) {
                    wr += nd.m; wc += nd.ncols; wl += nd.lrel_total; wu += nd.urel_total;
                    if (nd.m >= 96 && nd.ncols >= 96) {
                        bool use_tc = false;
                        int bn = H->opt.schur_variant != 1 ? SCHUR_BN_TILE : SCHUR_BN_BIG;
#ifndef SLU_COMPLEX
                        use_tc = H->tc_slices > 0 && nd.ns >= H->tc_min_ns && nd.ns <= 512;
                        if (use_tc) bn = OZ_NT_HOST;
#endif
                        (use_tc ? tc : big).push_back(k);
                        const int64_t tiles_m = (nd.m + SCHUR_BM_BIG - 1) / SCHUR_BM_BIG, tiles_n = (nd.ncols + bn - 1) / bn;
                        p_big.push_back(p_big.back() + tiles_m * tiles_n);
                        // look-ahead: which destinations are factored at the very next level of this forest?
                        int r1 = 0, c1 = 0;
                        bool other = false;
                        for (int q = 0; q < nd.nlb; ++q) {
                            const LBlk &lb = lblk[nd.lblk + q];
                            if (zl_of[lb.ib] == zl && lev[lb.ib] == lev[k] + 1) { if (q == 0) r1 = lb.nrows; else other = true; }
                        }
                        for (int q = 0; q < nd.nub; ++q) {
                            const UBlk &ub = ublk[nd.ublk + q];
                            if (zl_of[ub.jb] == zl && lev[ub.jb] == lev[k] + 1) { if (q == 0) c1 = ub.ncols; else other = true; }
                        }
                        if (other) { r1 = nd.m; c1 = nd.ncols; }
                        nd.urg_rows = r1; nd.urg_cols = c1;
                        const int64_t tru = (r1 + SCHUR_BM_BIG - 1) / SCHUR_BM_BIG, tcu = (c1 + bn - 1) / bn;
                        if (use_tc) {
#ifndef SLU_COMPLEX
                            p_big.pop_back();
                            p_tc.push_back(p_tc.back() + tiles_m * tiles_n);
                            p_tc_urg.push_back(p_tc_urg.back() + tiles_m * tcu + tru * (tiles_n - tcu));
                            p_tc_bulk.push_back(p_tc_bulk.back() + (tiles_m - tru) * (tiles_n - tcu));
                            const int S = H->tc_slices, KS = (nd.ns + OZ_KSTEP - 1) / OZ_KSTEP;
                            p_tc_rt.push_back(p_tc_rt.back() + tiles_m);
                            p_tc_ak.push_back(p_tc_ak.back() + tiles_m * KS);
                            p_tc_b.push_back(p_tc_b.back() + ((nd.ncols + OZ_NT - 1) / OZ_NT * OZ_NT + 3) / 4);
                            nd.ws_oza = woz; woz += oz_a_bytes(nd.m, nd.ns, S);
                            nd.ws_ozb = woz; woz += oz_b_bytes(nd.ncols, nd.ns, S);
                            nd.ws_ozs = wozs; wozs += oz_scale_elems(nd.m, nd.ncols);
                            if (!H->my_zero[zl]) ops_tc += 2.0 * nd.m * (double)nd.ns * nd.ncols;
#endif
                            continue;
                        }
                        p_urg.push_back(p_urg.back() + tiles_m * tcu + tru * (tiles_n - tcu));
                        p_bulk.push_back(p_bulk.back() + (tiles_m - tru) * (tiles_n - tcu));
                    } else {
                        small.push_back(k);
                        p_small.push_back(p_small.back() + (int64_t)((nd.m + SCHUR_BM_SMALL - 1) / SCHUR_BM_SMALL) * ((nd.ncols + SCHUR_BN_SMALL - 1) / SCHUR_BN_SMALL));
                    }
                }
            }
            ws_row_max = std::max(ws_row_max, wr); ws_col_max = std::max(ws_col_max, wc);
            ws_lrel_max = std::max(ws_lrel_max, wl); ws_urel_max = std::max(ws_urel_max, wu);
            ws_inv_max = std::max(ws_inv_max, p_inv.back() * 512);
            ws_oz_i8_max = std::max(ws_oz_i8_max, woz); ws_oz_s_max = std::max(ws_oz_s_max, wozs);
            auto put64 = [&](const std::vector<int64_t> &p) { int64_t o = (int64_t)pool_i64.size(); pool_i64.insert(pool_i64.end(), p.begin(), p.end()); return o; };
            L.trsml_prefix = put64(p_l); L.trsml_ctas = p_l.back();
            L.trsmu_prefix = put64(p_u); L.trsmu_ctas = p_u.back();
            L.setup_prefix = put64(p_s); L.setup_ctas = p_s.back();
            L.inv_prefix = put64(p_inv); L.inv_ctas = p_inv.back();
            L.sl_prefix = put64(p_sl); L.sl_ctas = p_sl.back();
            L.su_prefix = put64(p_su); L.su_ctas = p_su.back();
            L.big_count = (int)big.size(); L.big_nodes = (int64_t)pool_i32.size();
            pool_i32.insert(pool_i32.end(), big.begin(), big.end());
            L.big_prefix = put64(p_big); L.big_ctas = p_big.back();
            L.urg_prefix = put64(p_urg); L.urg_ctas = p_urg.back();
            L.bulk_prefix = put64(p_bulk); L.bulk_ctas = p_bulk.back();
            L.tc_count = (int)tc.size(); L.tc_nodes = (int64_t)pool_i32.size();
            pool_i32.insert(pool_i32.end(), tc.begin(), tc.end());
            L.tc_prefix = put64(p_tc); L.tc_ctas = p_tc.back();
            L.tc_urg_prefix = put64(p_tc_urg); L.tc_urg_ctas = p_tc_urg.back();
            L.tc_bulk_prefix = put64(p_tc_bulk); L.tc_bulk_ctas = p_tc_bulk.back();
            L.tc_p_rt = put64(p_tc_rt); L.tc_n_rt = p_tc_rt.back();
            L.tc_p_ak = put64(p_tc_ak); L.tc_n_ak = p_tc_ak.back();
            L.tc_p_b = put64(p_tc_b); L.tc_n_b = p_tc_b.back();
            L.small_count = (int)small.size(); L.small_nodes = (int64_t)pool_i32.size();
            pool_i32.insert(pool_i32.end(), small.begin(), small.end());
            L.small_prefix = put64(p_small); L.small_ctas = p_small.back();
            const int64_t lim = 2147483647LL;
            if (L.trsml_ctas > lim || L.trsmu_ctas > lim || L.setup_ctas > lim || L.big_ctas > lim || L.small_ctas > lim)
                return fail("a level needs more than 2^31 CTAs in one launch");
            H->levels.push_back(L);
        }
    }

    H->z_nodes_off.assign(max_lvl, 0);
    for (int zl = 0; zl < max_lvl; ++zl) {
        H->z_nodes_off[zl] = (int64_t)pool_i32.size();
        pool_i32.insert(pool_i32.end(), H->znodes[zl].begin(), H->znodes[zl].end());
    }
    lap("level batches");
    // the Schur workspace is double-buffered by level parity: with look-ahead the bulk update of level l still
    // reads its maps while level l+1 builds its own
    H->ws_max[0] = ws_row_max; H->ws_max[1] = ws_col_max; H->ws_max[2] = ws_lrel_max; H->ws_max[3] = ws_urel_max;
    for (size_t li = 0; li < H->levels.size(); ++li) {
        if (!(li & 1)) continue;
        const LevelPlan &L = H->levels[li];
        for (int t = 0; t < L.count; ++t) {
            NodeDesc &nd = H->nodes[pool_i32[L.nodes_off + t]];
            nd.ws_row += ws_row_max; nd.ws_col += ws_col_max; nd.ws_lrel += ws_lrel_max; nd.ws_urel += ws_urel_max;
            nd.ws_oza += ws_oz_i8_max; nd.ws_ozb += ws_oz_i8_max; nd.ws_ozs += ws_oz_s_max;
        }
    }
    // upload the index structures
    if (H->val.alloc((size_t)voff)) return -1;
    if (H->d_nodes.upload(H->nodes) || H->d_xsup.upload(H->xsup) || H->d_supno.upload(supno) ||
        H->d_lrows.upload(lrows) || H->d_lsrow.upload(lsrow) || H->d_lspos.upload(lspos) ||
        H->d_ucols.upload(ucols) || H->d_ufst.upload(ufst) || H->d_useg.upload(useg) ||
        H->d_lblk.upload(lblk) || H->d_ublk.upload(ublk) || H->d_pool_i32.upload(pool_i32) ||
        H->d_pool_i64.upload(pool_i64))
        return -1;
    if (H->d_rowinfo.alloc((size_t)ws_row_max * 2) || H->d_colinfo.alloc((size_t)ws_col_max * 2) ||
        H->d_lrel.alloc((size_t)ws_lrel_max * 2) || H->d_urel.alloc((size_t)ws_urel_max * 2) || H->d_flags.alloc(2) ||
        H->d_inv.alloc((size_t)ws_inv_max) ||
        H->d_tiny.alloc(1))
        return -1;
    if (ws_oz_i8_max > 0 &&
        (H->d_oz_i8.alloc((size_t)ws_oz_i8_max * 2) || H->d_oz_scale.alloc((size_t)ws_oz_s_max * 2) || H->d_oz_rexp.alloc((size_t)ws_oz_s_max * 2))) {
        H->tc_alloc_failed = true;
        H->d_oz_i8.release(); H->d_oz_scale.release(); H->d_oz_rexp.release();
        return fail("tcgen05 path: cannot allocate %.1f GB of int8 slice workspace (options.reserved[4] = -1 turns the path off): %s",
                    2e-9 * ws_oz_i8_max, g_err.c_str());
    }
    lap("device alloc + index upload");
    H->h_lblk = lblk;
    H->h_ublk = ublk;
    H->h_pool_i32 = pool_i32;
    DeviceLU &d = H->dev;
    d.val = H->val.p; d.nodes = H->d_nodes.p; d.xsup = H->d_xsup.p; d.supno = H->d_supno.p;
    d.lrows = H->d_lrows.p; d.lsrow = H->d_lsrow.p; d.lspos = H->d_lspos.p;
    d.ucols = H->d_ucols.p; d.ufst = H->d_ufst.p; d.useg = H->d_useg.p;
    d.lblk = H->d_lblk.p; d.ublk = H->d_ublk.p; d.rowinfo = H->d_rowinfo.p; d.colinfo = H->d_colinfo.p;
    d.oz_i8 = H->d_oz_i8.p; d.oz_scale = H->d_oz_scale.p; d.oz_rexp = H->d_oz_rexp.p;
    d.lrel = H->d_lrel.p; d.urel = H->d_urel.p; d.info = H->d_flags.p; d.err = H->d_flags.p + 1; d.tiny = H->d_tiny.p;

    slu_b200_stats_t &st = H->st;
    st.ops_fact = ops; st.ops_schur = ops_schur; st.schur_bytes = bytes_schur;
    st.nnz_l = nnz_l; st.nnz_u = nnz_u; st.nlevels = (int)H->levels.size();
    st.lu_device_bytes = (int64_t)H->val.bytes();
    st.reserved[1] = ops_tc;                                   // Schur flops taken by the tcgen05 path
    st.reserved[2] = (double)(H->d_oz_i8.bytes() + H->d_oz_scale.bytes() + H->d_oz_rexp.bytes());
    st.reserved[3] = (double)H->tc_slices;
    st.index_device_bytes = (int64_t)(H->d_nodes.bytes() + H->d_xsup.bytes() + H->d_supno.bytes() + H->d_lrows.bytes() * 3 +
                                      H->d_ucols.bytes() * 3 + H->d_lblk.bytes() + H->d_ublk.bytes() + H->d_pool_i32.bytes() +
                                      H->d_pool_i64.bytes() + H->d_rowinfo.bytes() + H->d_colinfo.bytes() + H->d_lrel.bytes() +
                                      H->d_urel.bytes() + H->d_oz_i8.bytes() + H->d_oz_scale.bytes() + H->d_oz_rexp.bytes());
    int mine = 0;
    for (int zl = 0; zl < max_lvl; ++zl)
        if (!H->my_zero[zl]) mine += (int)H->znodes[zl].size();
    st.my_supernodes = mine;
    return 0;
}

// ------------------------------------------------------------------------------------------------
// Pr x Pc > 1.  The caller's panels are block-cyclic pieces (block (I,J) on process (I mod Pr, J mod Pc),
// SRC/include/superlu_defs.h:270-279).  Here every rank of a layer keeps the WHOLE panels of the layer's forests
// and the cooperative schedule does the rest: each rank uploads only its own blocks into a zeroed arena, the
// per-level all-reduce makes the panels complete, the Schur tiles are dealt over the Pr*Pc*2^level ranks of the
// group, and the local blocks are copied back at the end.  What the reference does with per-supernode panel and
// diagonal broadcasts (dIBcast_LPanel/UPanel, dcommunication_aux.c:29-283) becomes one NVSwitch all-reduce per level.
// ------------------------------------------------------------------------------------------------
int gather_structure(slu_b200_handle_s *H)
{
    const slu_b200_lu_view_t &v = H->view;
    const int nsupers = v.nsupers;
    H->Lidx.assign(nsupers, nullptr);
    H->Uidx.assign(nsupers, nullptr);
    if (H->P2 == 1) {
        for (int k = 0; k < nsupers; ++k) { H->Lidx[k] = v.Lrowind_bc_ptr[k]; H->Uidx[k] = v.Ufstnz_br_ptr[k]; }
        return 0;
    }
    const slu_int *xsup = v.xsup;
    // serialise my pieces of the supernodes of my forests: [type, k, len, payload]
    std::vector<int32_t> mine;
    std::vector<char> inforest(nsupers, 0);
    for (int zl = 0; zl < v.maxLvl; ++zl) {
        const slu_b200_forest_t &f = v.forests[v.myTreeIdxs[zl]];
        for (int t = 0; t < f.nNodes; ++t) inforest[f.nodeList[t]] = 1;
    }
    for (int k = 0; k < nsupers; ++k) {
        if (!inforest[k]) continue;
        if (k % v.npcol == v.mycol) {
            const slu_int *li = v.Lrowind_bc_ptr[k / v.npcol];
            if (li) {
                int len = BC_HEADER + li[0] * LB_DESCRIPTOR + li[1];
                mine.push_back(0); mine.push_back(k); mine.push_back(len);
                mine.insert(mine.end(), li, li + len);
            }
        }
        if (k % v.nprow == v.myrow) {
            const slu_int *ui = v.Ufstnz_br_ptr[k / v.nprow];
            if (ui) {
                mine.push_back(1); mine.push_back(k); mine.push_back(ui[2]);
                mine.insert(mine.end(), ui, ui + ui[2]);
            }
        }
    }
    // all-gather over my layer
    if (!g_nccl.AllGather) return fail("this NCCL has no ncclAllGather");
    const int P2 = H->P2;
    DevBuf<int32_t> dsz, dall, dsend, drecv;
    std::vector<int32_t> sizes(P2, 0), one{(int32_t)mine.size()};
    if (dsz.upload(one) || dall.alloc(P2)) return -1;
    NC(g_nccl.AllGather(dsz.p, dall.p, 1, NCCL_INT32, H->lcomm, H->stream));
    CU(cudaStreamSynchronize(H->stream));
    CU(cudaMemcpy(sizes.data(), dall.p, P2 * sizeof(int32_t), cudaMemcpyDeviceToHost));
    size_t maxn = 1;
    for (int s2 : sizes) maxn = std::max(maxn, (size_t)s2);
    std::vector<int32_t> padded(maxn, 0), all(maxn * P2);
    std::copy(mine.begin(), mine.end(), padded.begin());
    if (dsend.upload(padded) || drecv.alloc(maxn * P2)) return -1;
    NC(g_nccl.AllGather(dsend.p, drecv.p, maxn, NCCL_INT32, H->lcomm, H->stream));
    CU(cudaStreamSynchronize(H->stream));
    CU(cudaMemcpy(all.data(), drecv.p, all.size() * sizeof(int32_t), cudaMemcpyDeviceToHost));
    dsz.release(); dall.release(); dsend.release(); drecv.release();
    // merge
    struct Blk { int id; const int32_t *body; int len; };
    std::vector<std::vector<Blk>> lb(nsupers), ub(nsupers);
    for (int r = 0; r < P2; ++r) {
        const int32_t *p = all.data() + (size_t)r * maxn, *e = p + sizes[r];
        while (p < e) {
            int type = p[0], k = p[1], len = p[2];
            const int32_t *idx = p + 3;
            if (k < 0 || k >= nsupers) return fail("bad structure message");
            if (type == 0) {
                int w = BC_HEADER;
                for (int b = 0; b < idx[0]; ++b) { lb[k].push_back(Blk{idx[w], idx + w, LB_DESCRIPTOR + idx[w + 1]}); w += LB_DESCRIPTOR + idx[w + 1]; }
            } else {
                int u = BR_HEADER;
                for (int b = 0; b < idx[0]; ++b) {
                    int jns = xsup[idx[u] + 1] - xsup[idx[u]];
                    ub[k].push_back(Blk{idx[u], idx + u, UB_DESCRIPTOR + jns});
                    u += UB_DESCRIPTOR + jns;
                }
            }
            p += 3 + len;
        }
    }
    H->fullL.assign(nsupers, {});
    H->fullU.assign(nsupers, {});
    auto byid = [](const Blk &a, const Blk &b) { return a.id < b.id; };
    for (int k = 0; k < nsupers; ++k) {
        if (!inforest[k]) continue;
        if (!lb[k].empty()) {
            std::sort(lb[k].begin(), lb[k].end(), byid);
            std::vector<slu_int> &f = H->fullL[k];
            f.assign(BC_HEADER, 0);
            int nrows = 0;
            for (auto &b : lb[k]) { f.insert(f.end(), b.body, b.body + b.len); nrows += b.body[1]; }
            f[0] = (slu_int)lb[k].size(); f[1] = nrows;
            H->Lidx[k] = f.data();
        }
        if (!ub[k].empty()) {
            std::sort(ub[k].begin(), ub[k].end(), byid);
            std::vector<slu_int> &f = H->fullU[k];
            f.assign(BR_HEADER, 0);
            int nnz = 0;
            for (auto &b : ub[k]) { f.insert(f.end(), b.body, b.body + b.len); nnz += b.body[1]; }
            f[0] = (slu_int)ub[k].size(); f[1] = nnz; f[2] = (slu_int)f.size();
            H->Uidx[k] = f.data();
        }
    }
    return 0;
}

// where my local blocks sit inside the replicated panels
int build_pieces(slu_b200_handle_s *H)
{
    const slu_b200_lu_view_t &v = H->view;
    H->pieces.clear();
    if (H->P2 == 1) return 0;
    const slu_int *xsup = v.xsup;
    for (auto &zn : H->znodes)
        for (int k : zn) {
            const NodeDesc &nd = H->nodes[k];
            if (k % v.npcol == v.mycol && v.Lrowind_bc_ptr[k / v.npcol]) {
                const slu_int *li = v.Lrowind_bc_ptr[k / v.npcol];
                val_t *lv = (val_t *)v.Lnzval_bc_ptr[k / v.npcol];
                if (!lv) return fail("L piece %d has no values", k);
                // row offset of every block of the full panel
                const slu_int *fi = H->Lidx[k];
                int w = BC_HEADER, lo = 0;
                for (int b = 0; b < li[0]; ++b) {
                    int ib = li[w], nb = li[w + 1], fw = BC_HEADER, fo = 0, found = 0;
                    for (int q = 0; q < fi[0]; ++q) {
                        if (fi[fw] == ib) { found = 1; break; }
                        fo += fi[fw + 1]; fw += LB_DESCRIPTOR + fi[fw + 1];
                    }
                    if (!found) return fail("L piece %d: block %d missing from the merged panel", k, ib);
                    H->pieces.push_back({nd.lval + fo, lv + lo, nb, nd.ns, li[1], nd.nsupr});
                    lo += nb; w += LB_DESCRIPTOR + nb;
                }
            }
            if (k % v.nprow == v.myrow && v.Ufstnz_br_ptr[k / v.nprow]) {
                const slu_int *ui = v.Ufstnz_br_ptr[k / v.nprow];
                val_t *uv = (val_t *)v.Unzval_br_ptr[k / v.nprow];
                const int klst = xsup[k + 1];
                int u = BR_HEADER;
                int64_t lo = 0;
                for (int b = 0; b < ui[0]; ++b) {
                    int jb = ui[u], jns = xsup[jb + 1] - xsup[jb], cnt = 0;
                    for (int c = 0; c < jns; ++c) {
                        int fst = ui[u + UB_DESCRIPTOR + c];
                        if (fst >= klst) continue;
                        if (klst - fst != nd.ns) return fail("Pr x Pc > 1 needs U panels whose skyline segments are all full");
                        ++cnt;
                    }
                    if (cnt) {
                        int64_t col0 = -1;
                        for (int q = 0; q < nd.nub; ++q)
                            if (H->h_ublk[nd.ublk + q].jb == jb) { col0 = H->h_ublk[nd.ublk + q].col0; break; }
                        if (col0 < 0) return fail("U piece %d: block %d missing from the merged panel", k, jb);
                        if (!uv) return fail("U piece %d has no values", k);
                        H->pieces.push_back({nd.uval + col0 * nd.ns, uv + lo, (int64_t)cnt * nd.ns, 1, (int64_t)cnt * nd.ns, (int64_t)cnt * nd.ns});
                        lo += (int64_t)cnt * nd.ns;
                    }
                    u += UB_DESCRIPTOR + jns;
                }
            }
        }
    return 0;
}

int transfer_2d(slu_b200_handle_s *H, bool to_device)
{
    if (to_device) CU(cudaMemsetAsync(H->val.p, 0, H->val.bytes(), H->stream));
    for (const auto &p : H->pieces) {
        if (to_device)
            CU(cudaMemcpy2DAsync(H->val.p + p.dev, (size_t)p.dpitch * sizeof(val_t), p.host, (size_t)p.spitch * sizeof(val_t), (size_t)p.width * sizeof(val_t),
                                 (size_t)p.height, cudaMemcpyHostToDevice, H->stream));
        else
            CU(cudaMemcpy2DAsync(p.host, (size_t)p.spitch * sizeof(val_t), H->val.p + p.dev, (size_t)p.dpitch * sizeof(val_t), (size_t)p.width * sizeof(val_t),
                                 (size_t)p.height, cudaMemcpyDeviceToHost, H->stream));
    }
    CU(cudaStreamSynchronize(H->stream));
    return 0;
}

// copy a list of (device offset, host pointer, length) runs, merging neighbours
struct Run { int64_t dev; val_t *host; int64_t len; };
int copy_runs(slu_b200_handle_s *H, std::vector<Run> &runs, bool to_device)
{
    size_t i = 0;
    while (i < runs.size()) {
        Run r = runs[i];
        size_t j = i + 1;
        while (j < runs.size() && runs[j].dev == r.dev + r.len && runs[j].host == r.host + r.len) { r.len += runs[j].len; ++j; }
        if (r.len > 0) {
            if (to_device) CU(cudaMemcpyAsync(H->val.p + r.dev, r.host, (size_t)r.len * sizeof(val_t), cudaMemcpyHostToDevice, H->stream));
            else CU(cudaMemcpyAsync(r.host, H->val.p + r.dev, (size_t)r.len * sizeof(val_t), cudaMemcpyDeviceToHost, H->stream));
        }
        i = j;
    }
    return 0;
}

// skyline <-> dense-packed conversion of the U panels that are not already identical
int convert_u(slu_b200_handle_s *H, bool to_device)
{
    const size_t STAGE = (size_t)32 << 20;  // elements (256 MB of doubles) per round
    std::vector<int32_t> pend;
    for (auto &zn : H->znodes)
        for (int k : zn)
            if (!H->u_full[k] && H->nodes[k].ncols > 0) pend.push_back(k);
    if (pend.empty()) return 0;
    size_t need = 0;
    for (int k : pend) need = std::max(need, (size_t)H->sky_len[k]);
    if (H->stage.n < std::max(need, std::min(STAGE, need * 64))) {
        if (H->stage.alloc(std::max(need, std::min(STAGE, need * 64)))) return -1;
    }
    size_t i = 0;
    DevBuf<int32_t> dn;
    DevBuf<int64_t> dp, ds;
    while (i < pend.size()) {
        std::vector<int32_t> nodes;
        std::vector<int64_t> prefix{0}, soff;
        size_t used = 0;
        while (i < pend.size() && used + (size_t)H->sky_len[pend[i]] <= H->stage.n) {
            int k = pend[i++];
            nodes.push_back(k);
            soff.push_back((int64_t)used);
            used += (size_t)H->sky_len[k];
            prefix.push_back(prefix.back() + (H->nodes[k].ncols + 31) / 32);
        }
        if (dn.upload(nodes) || dp.upload(prefix) || ds.upload(soff)) return -1;
        Batch b{dn.p, dp.p, (int)nodes.size()};
        if (to_device) {
            for (size_t t = 0; t < nodes.size(); ++t)
                CU(cudaMemcpyAsync(H->stage.p + soff[t], H->view.Unzval_br_ptr[nodes[t]], (size_t)H->sky_len[nodes[t]] * sizeof(val_t),
                                   cudaMemcpyHostToDevice, H->stream));
            launch_u_convert(H->dev, b, prefix.back(), 0, H->stage.p, ds.p, H->stream);
        } else {
            launch_u_convert(H->dev, b, prefix.back(), 1, H->stage.p, ds.p, H->stream);
            for (size_t t = 0; t < nodes.size(); ++t)
                CU(cudaMemcpyAsync(H->view.Unzval_br_ptr[nodes[t]], H->stage.p + soff[t], (size_t)H->sky_len[nodes[t]] * sizeof(val_t),
                                   cudaMemcpyDeviceToHost, H->stream));
        }
        CU(cudaStreamSynchronize(H->stream));
        CU(cudaGetLastError());
    }
    dn.release(); dp.release(); ds.release();
    return 0;
}

int transfer(slu_b200_handle_s *H, bool to_device)
{
    if (H->P2 > 1) return transfer_2d(H, to_device);
    std::vector<Run> runs;
    for (auto &zn : H->znodes) {
        for (int k : zn) {
            const NodeDesc &nd = H->nodes[k];
            runs.push_back(Run{nd.lval, (val_t *)H->view.Lnzval_bc_ptr[k], (int64_t)nd.nsupr * nd.ns});
        }
        for (int k : zn) {
            const NodeDesc &nd = H->nodes[k];
            if (H->u_full[k] && nd.ncols > 0) runs.push_back(Run{nd.uval, (val_t *)H->view.Unzval_br_ptr[k], (int64_t)nd.ns * nd.ncols});
        }
    }
    for (auto &r : runs)
        if (r.len > 0 && !r.host) return fail("a held panel has a NULL value pointer");
    if (copy_runs(H, runs, to_device)) return -1;
    if (convert_u(H, to_device)) return -1;
    CU(cudaStreamSynchronize(H->stream));
    return 0;
}

int reduce_ancestors(slu_b200_handle_s *H, int zl)
{
    // dreduceAllAncestors3d (pd3dcomm.c:1046-1081): layers with z % 2^(zl+1) != 0 send all their
    // ancestor panels to z - 2^zl, which adds them.  The ancestor forests are one contiguous slab.
    const int z = H->view.mydep;
    const int64_t begin = H->chunk_start[zl + 1], end = H->chunk_start[H->max_lvl];
    const int64_t total = end - begin;
    if (total <= 0) return 0;
    const size_t CH = (size_t)64 << 20;  // elements per message (512 MB of doubles)
    if (z % (1 << (zl + 1)) != 0) {
        const int peer = z - (1 << zl);
        for (int64_t o = 0; o < total; o += (int64_t)CH) {
            size_t len = (size_t)std::min<int64_t>(CH, total - o);
            NC(g_nccl.Send(H->val.p + begin + o, len * VAL_DOUBLES, NCCL_FLOAT64, peer, H->comm, H->stream));
        }
    } else {
        const int peer = z + (1 << zl);
        if (H->stage.n < std::min<size_t>(CH, (size_t)total))
            if (H->stage.alloc(std::min<size_t>(CH, (size_t)total))) return -1;
        for (int64_t o = 0; o < total; o += (int64_t)CH) {
            size_t len = (size_t)std::min<int64_t>(CH, total - o);
            NC(g_nccl.Recv(H->stage.p, len * VAL_DOUBLES, NCCL_FLOAT64, peer, H->comm, H->stream));
            H->st.gpu_launches += launch_axpy(H->val.p + begin + o, H->stage.p, (int64_t)len, H->stream);
        }
    }
    return 0;
}

// ---- overlapped download ------------------------------------------------------------------------------------
// A panel is final as soon as the panel work of its level is done (nothing updates a factored panel), so its D2H
// can run on a copy stream while the upper levels are still being factored.  The arena is cut into chunks that are
// contiguous on both sides (host arrays of consecutive supernodes are usually adjacent); a chunk is released after
// the last level any of its panels belongs to.
int pipe_prepare(slu_b200_handle_s *H)
{
    if (H->pipe_ready) return 0;
    if (H->P2 > 1) return fail("overlapped transfers are not available for Pr x Pc > 1");
    for (auto &zn : H->znodes)
        for (int k : zn)
            if (!H->u_full[k] && H->nodes[k].ncols > 0)
                return fail("overlapped transfers need U panels whose skyline segments are all full");
    std::vector<int32_t> pool(H->d_pool_i32.n);
    CU(cudaMemcpy(pool.data(), H->d_pool_i32.p, pool.size() * sizeof(int32_t), cudaMemcpyDeviceToHost));
    std::vector<int> level_of(H->nsupers, -1);
    for (size_t li = 0; li < H->levels.size(); ++li)
        for (int t = 0; t < H->levels[li].count; ++t) level_of[pool[H->levels[li].nodes_off + t]] = (int)li;
    // panels in arena order, merged into chunks of <= 32M elements (256 MB of doubles)
    const int64_t CH = (int64_t)32 << 20;
    H->h_segs.clear(); H->h_seg_host.clear();
    std::vector<int> seg_level;
    bool fresh = true;       // never merge across a Z-level boundary: with reference-style ancestors a layer with
                             // my_zero[zl+1] never runs that level, and a chunk spanning both would never be released
    auto add = [&](int64_t dev, val_t *host, int64_t len, int lvl) {
        if (len <= 0) return;
        if (!H->h_segs.empty() && !fresh) {
            UpSeg &b2 = H->h_segs.back();
            if (b2.dst + b2.len == dev && H->h_seg_host.back() + b2.len == host && b2.len + len <= CH) {
                b2.len += len;
                seg_level.back() = std::max(seg_level.back(), lvl);
                return;
            }
        }
        H->h_segs.push_back(UpSeg{dev, 0, len});
        H->h_seg_host.push_back(host);
        seg_level.push_back(lvl);
        fresh = false;
    };
    for (auto &zn : H->znodes) {
        fresh = true;
        for (int k : zn) add(H->nodes[k].lval, (val_t *)H->view.Lnzval_bc_ptr[k], (int64_t)H->nodes[k].nsupr * H->nodes[k].ns, level_of[k]);
        for (int k : zn) add(H->nodes[k].uval, (val_t *)H->view.Unzval_br_ptr[k], (int64_t)H->nodes[k].ns * H->nodes[k].ncols, level_of[k]);
    }
    // bucket the chunks by release level
    H->lvl_segs.assign(H->levels.size(), {0, 0});
    std::vector<size_t> order(H->h_segs.size());
    for (size_t i = 0; i < order.size(); ++i) order[i] = i;
    std::stable_sort(order.begin(), order.end(), [&](size_t x, size_t y) { return seg_level[x] < seg_level[y]; });
    std::vector<UpSeg> segs2;
    std::vector<val_t *> host2;
    for (size_t i : order) {
        if (seg_level[i] < 0) continue;
        segs2.push_back(H->h_segs[i]);
        host2.push_back(H->h_seg_host[i]);
        H->lvl_segs[seg_level[i]][1] = (int64_t)segs2.size();
    }
    int64_t prev = 0;
    for (auto &r : H->lvl_segs) { r[0] = prev; if (r[1] < prev) r[1] = prev; prev = r[1]; }
    H->h_segs.swap(segs2);
    H->h_seg_host.swap(host2);
    if (!H->s_down && cudaStreamCreateWithFlags(&H->s_down, cudaStreamNonBlocking) != cudaSuccess)
        return fail("cannot create the download stream");
    H->pipe_ready = true;
    return 0;
}

// D2H of the chunks whose panels are all final once level li's panel work is done
int pipe_download_level(slu_b200_handle_s *H, size_t li)
{
    const int64_t a = H->lvl_segs[li][0], b = H->lvl_segs[li][1];
    if (a >= b) return 0;
    CU(cudaStreamWaitEvent(H->s_down, H->ev_panel[li], 0));
    for (int64_t q = a; q < b; ++q)
        CU(cudaMemcpyAsync(H->h_seg_host[q], H->val.p + H->h_segs[q].dst, (size_t)H->h_segs[q].len * sizeof(val_t), cudaMemcpyDeviceToHost, H->s_down));
    return 0;
}

// ---- overlapped upload (options.reserved[3]) ---------------------------------------------------------------
// With the level-by-level layout the panels are needed in arena order.  The arena is zeroed, every level's host
// panels are copied through a staging buffer and ADDED to the arena with atomic adds on a copy stream (a Schur
// update scattered into an ancestor before that ancestor's A values arrive commutes with the addition), and the
// panel work of level li waits for the event of level li only: the H2D of the upper levels -- most of the bytes --
// runs under the factorization of the lower ones.
int upload_pipe_issue(slu_b200_handle_s *H)
{
    if (!H->grouped) return fail("overlapped upload needs options.reserved[3] at create time and Pr x Pc = 1");
    for (auto &zn : H->znodes)
        for (int k : zn)
            if (!H->u_full[k] && H->nodes[k].ncols > 0)
                return fail("overlapped transfers need U panels whose skyline segments are all full");
    const size_t CAP = (size_t)32 << 20;  // elements per staging round
    if (H->stage.n < CAP && H->stage.alloc(CAP)) return -1;
    if (!H->s_up && cudaStreamCreateWithFlags(&H->s_up, cudaStreamNonBlocking) != cudaSuccess)
        return fail("cannot create the upload stream");
    if (H->ev_up.size() != H->levels.size()) {
        for (auto e : H->ev_up) if (e) cudaEventDestroy(e);
        H->ev_up.assign(H->levels.size(), nullptr);
        for (auto &e : H->ev_up) cudaEventCreateWithFlags(&e, cudaEventDisableTiming);
    }
    cudaStream_t su = H->s_up;
    CU(cudaMemsetAsync(H->val.p, 0, H->val.bytes(), su));
    for (size_t li = 0; li < H->levels.size(); ++li) {
        const LevelPlan &L = H->levels[li];
        const int32_t *nodes = H->h_pool_i32.data() + L.nodes_off;
        int64_t off = L.slab_begin;   // next arena element to receive
        size_t fill = 0;
        auto flush = [&]() -> int {
            if (!fill) return 0;
            H->st.gpu_launches += launch_axpy_atomic(H->val.p + off, H->stage.p, (int64_t)fill, su);
            off += (int64_t)fill;
            fill = 0;
            return 0;
        };
        for (int pass = 0; pass < 2; ++pass)  // the L panels of the level, then its U panels (arena order)
            for (int t = 0; t < L.count; ++t) {
                const int k = nodes[t];
                const NodeDesc &nd = H->nodes[k];
                const int64_t dev = pass ? nd.uval : nd.lval;
                const int64_t len = pass ? (int64_t)nd.ns * nd.ncols : (int64_t)nd.nsupr * nd.ns;
                const val_t *host = (const val_t *)(pass ? H->view.Unzval_br_ptr[k] : H->view.Lnzval_bc_ptr[k]);
                if (len <= 0) continue;
                if (dev != off + (int64_t)fill) return fail("internal: level %zu is not contiguous in the arena", li);
                if (!host) return fail("a held panel has a NULL value pointer");
                int64_t pos = 0;
                while (pos < len) {
                    const size_t take = (size_t)std::min<int64_t>(len - pos, (int64_t)(CAP - fill));
                    CU(cudaMemcpyAsync(H->stage.p + fill, host + pos, take * sizeof(val_t), cudaMemcpyHostToDevice, su));
                    fill += take; pos += (int64_t)take;
                    if (fill == CAP && flush()) return -1;
                }
            }
        if (flush()) return -1;
        CU(cudaEventRecord(H->ev_up[li], su));
    }
    return 0;
}

}  // namespace

// ------------------------------------------------------------------------------------------------
// C-ABI
// ------------------------------------------------------------------------------------------------
extern "C" {

#ifndef SLU_COMPLEX
int slu_b200_abi_version(void) { return SLU_B200_ABI_VERSION; }
void slu_b200_struct_sizes(int32_t out[4])
{
    out[0] = (int32_t)sizeof(slu_b200_forest_t); out[1] = (int32_t)sizeof(slu_b200_lu_view_t);
    out[2] = (int32_t)sizeof(slu_b200_options_t); out[3] = (int32_t)sizeof(slu_b200_stats_t);
}
const char *slu_b200_last_error(void) { return g_err.c_str(); }
int slu_b200_device_count(void)
{
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
    return n;
}

int slu_b200_nccl_unique_id(unsigned char id[128])
{
    if (!g_nccl.load()) return fail("cannot load libnccl.so.2");
    slu_nccl_id u;
    NC(g_nccl.GetUniqueId(&u));
    memcpy(id, u.internal, 128);
    return 0;
}

void *slu_b200_host_alloc(size_t bytes)
{
    void *p = nullptr;
    if (cudaHostAlloc(&p, bytes ? bytes : 1, cudaHostAllocDefault) != cudaSuccess) { cudaGetLastError(); return nullptr; }
    return p;
}
void slu_b200_host_free(void *p) { if (p) cudaFreeHost(p); }
#endif  // !SLU_COMPLEX

#ifdef SLU_COMPLEX
void slu_b200_z_comm_cache_clear(void)
#else
void slu_b200_z_comm_cache_clear(void);
static void comm_cache_clear_d(void)
#endif
{
    std::lock_guard<std::mutex> lock(g_comm_mu);
    for (auto &kv : g_comm_cache) {
        for (void *c : kv.second.gcomm) if (c && g_nccl.CommDestroy) g_nccl.CommDestroy(c);
        if (kv.second.comm && g_nccl.CommDestroy) g_nccl.CommDestroy(kv.second.comm);
    }
    g_comm_cache.clear();
}
#ifndef SLU_COMPLEX
void slu_b200_comm_cache_clear(void)
{
    comm_cache_clear_d();
    slu_b200_z_comm_cache_clear();
}
#endif

void slu_b200_destroy(slu_b200_handle_t H)
{
    if (!H) return;
    // the NCCL communicators belong to the per-process cache (slu_b200_comm_cache_clear)
    if (H->ev0) cudaEventDestroy(H->ev0);
    if (H->ev1) cudaEventDestroy(H->ev1);
    if (H->stream) cudaStreamDestroy(H->stream);
    if (H->stream2) cudaStreamDestroy(H->stream2);
    if (H->s_down) cudaStreamDestroy(H->s_down);
    if (H->s_up) cudaStreamDestroy(H->s_up);
    for (auto e : H->ev_up) if (e) cudaEventDestroy(e);
    for (auto e : H->ev_panel) if (e) cudaEventDestroy(e);
    for (auto e : H->ev_bulk) if (e) cudaEventDestroy(e);
    H->val.release(); H->stage.release(); H->d_inv.release(); H->d_nodes.release(); H->d_xsup.release(); H->d_supno.release();
    H->d_lrows.release(); H->d_lsrow.release(); H->d_lspos.release(); H->d_ucols.release(); H->d_ufst.release();
    H->d_useg.release(); H->d_pool_i32.release(); H->d_pool_i64.release(); H->d_lrel.release(); H->d_urel.release();
    H->d_lblk.release(); H->d_ublk.release(); H->d_rowinfo.release(); H->d_colinfo.release(); H->d_flags.release();
    H->d_x.release(); H->d_x2.release();
    H->d_tiny.release(); H->d_oz_i8.release(); H->d_oz_scale.release(); H->d_oz_rexp.release();
    delete H;
}

int slu_b200_create(slu_b200_handle_t *out, const slu_b200_lu_view_t *lu, const slu_b200_options_t *opt)
{
    if (!out || !lu || !opt) return fail("null argument");
    *out = nullptr;
    if (slu_b200_device_count() < 1) return fail("no CUDA device: libslu_b200 has no CPU fallback");
    if (device_setup(opt)) return -1;
    slu_b200_handle_s *H = new slu_b200_handle_s;
    H->view = *lu;
    H->opt = *opt;
    H->coop = opt->world_size > 1 && !opt->reserved[1];
    H->P2 = lu->nprow * lu->npcol;
    double t0 = now_s();
    if (lu->npdep < 1 || (lu->npdep & (lu->npdep - 1)) || H->P2 < 1) { slu_b200_destroy(H); return fail("bad process grid"); }
    H->max_lvl = 1;
    while ((1 << (H->max_lvl - 1)) < lu->npdep) ++H->max_lvl;
    if (cudaStreamCreate(&H->stream) != cudaSuccess || cudaEventCreate(&H->ev0) != cudaSuccess ||
        cudaEventCreate(&H->ev1) != cudaSuccess) {
        slu_b200_destroy(H);
        return fail("cannot create stream/events");
    }
    if (opt->world_size > 1) {
        if (opt->world_size != lu->npdep * H->P2) { slu_b200_destroy(H); return fail("world_size does not match the process grid"); }
        if (!g_nccl.load()) { slu_b200_destroy(H); return fail("cannot load libnccl.so.2"); }
        std::string key((const char *)opt->nccl_id, 128);
        const int32_t shape[9] = {opt->world_size, opt->world_rank, lu->nprow, lu->npcol, lu->npdep, lu->myrow, lu->mycol, lu->mydep, (int32_t)H->coop};
        key.append((const char *)shape, sizeof shape);
        std::lock_guard<std::mutex> lock(g_comm_mu);
        CommSet &cs = g_comm_cache[key];
        if (!cs.comm) {
            slu_nccl_id id;
            memcpy(id.internal, opt->nccl_id, 128);
            int r = g_nccl.CommInitRank(&cs.comm, opt->world_size, id, opt->world_rank);
            if (r != 0) { g_comm_cache.erase(key); slu_b200_destroy(H); return fail("ncclCommInitRank failed: %d", r); }
            cs.gcomm.assign(H->max_lvl, nullptr);
            if (H->coop) {
                if (!g_nccl.CommSplit) { g_comm_cache.erase(key); slu_b200_destroy(H); return fail("this NCCL has no ncclCommSplit (need >= 2.18)"); }
                // my group at Z level zl: the Pr*Pc ranks of each of the 2^zl layers sharing forest my_tree[zl]
                for (int zl = (H->P2 > 1 ? 0 : 1); zl < H->max_lvl; ++zl) {
                    r = g_nccl.CommSplit(cs.comm, lu->mydep >> zl, opt->world_rank, &cs.gcomm[zl], nullptr);
                    if (r != 0) { g_comm_cache.erase(key); slu_b200_destroy(H); return fail("ncclCommSplit failed: %d", r); }
                }
            }
        }
        H->comm = cs.comm;
        H->gcomm = cs.gcomm;
        if (H->coop) H->lcomm = H->gcomm[0];
    } else if (lu->npdep > 1 || H->P2 > 1) {
        slu_b200_destroy(H);
        return fail("a process grid with more than one rank needs world_size == nprow*npcol*npdep and an NCCL id");
    }
    if (gather_structure(H)) { slu_b200_destroy(H); return -1; }
    if (analyze(H)) {
        // the int8 slice workspace of the tcgen05 path did not fit beside the L/U arena: plan again without it (FP64 DMMA only)
        if (!H->tc_alloc_failed) { slu_b200_destroy(H); return -1; }
        cudaGetLastError();
        H->tc_force_off = true;
        H->tc_alloc_failed = false;
        if (analyze(H)) { slu_b200_destroy(H); return -1; }
    }
    if (build_pieces(H)) { slu_b200_destroy(H); return -1; }
    {
        int lo = 0, hi = 0;
        cudaDeviceGetStreamPriorityRange(&lo, &hi);  // hi = numerically lowest = highest priority
        cudaStreamDestroy(H->stream);
        H->stream = nullptr;
        if (cudaStreamCreateWithPriority(&H->stream, cudaStreamNonBlocking, hi) != cudaSuccess ||
            cudaStreamCreateWithPriority(&H->stream2, cudaStreamNonBlocking, lo) != cudaSuccess) {
            slu_b200_destroy(H);
            return fail("cannot create the look-ahead streams");
        }
        H->ev_panel.resize(H->levels.size());
        H->ev_bulk.resize(H->levels.size());
        for (size_t i = 0; i < H->levels.size(); ++i) {
            cudaEventCreateWithFlags(&H->ev_panel[i], cudaEventDisableTiming);
            cudaEventCreateWithFlags(&H->ev_bulk[i], cudaEventDisableTiming);
        }
    }
    H->st.t_analyze_s = now_s() - t0;
    *out = H;
    return 0;
}

int slu_b200_upload(slu_b200_handle_t H)
{
    if (!H) return fail("null handle");
    double t0 = now_s();
    H->factored = false;
    if (transfer(H, true)) return -1;
    H->st.t_upload_s = now_s() - t0;
    H->uploaded = true;
    return 0;
}

int slu_b200_download(slu_b200_handle_t H)
{
    if (!H) return fail("null handle");
    double t0 = now_s();
    if (transfer(H, false)) return -1;
    H->st.t_download_s = now_s() - t0;
    return 0;
}

static int factor_impl(slu_b200_handle_t H, int *info, bool pipelined, bool up_pipe = false)
{
    if (!H || !info) return fail("null argument");
    if (!H->uploaded) return fail("slu_b200_factor before slu_b200_upload");
    if (pipelined && pipe_prepare(H)) return -1;
    cudaStream_t s = H->stream;
    const DeviceLU &d = H->dev;
    int init[2] = {INT_MAX, 0};
    CU(cudaMemcpyAsync(H->d_flags.p, init, sizeof init, cudaMemcpyHostToDevice, s));
    CU(cudaMemsetAsync(H->d_tiny.p, 0, sizeof(unsigned long long), s));
    H->st.gpu_launches = 0;
    const bool prof = H->opt.verbose >= 2 && !pipelined;
    float t_diag = 0, t_trsm = 0, t_setup = 0, t_schur = 0, t_red = 0;

    EventSet pe;
    if (prof && pe.create()) return fail("cannot create the profiling events");
    CU(cudaEventRecord(H->ev0, s));
    // Look-ahead (the role of dsparseTreeFactor_ASYNC's pipeline, dtreeFactorization.c:430-454,598-706): the
    // critical path (panel work of level l, then the "urgent" Schur tiles that feed the panels of level l+1) runs on
    // a high-priority stream; the bulk of the Schur update of level l runs on a second stream, concurrently with the
    // panel work of level l+1.  All updates are atomic adds, so bulk(l) and anything of level l+1 commute; the only
    // ordering needed is panel(l) after bulk(l-2) (in-order stream: after every earlier bulk).
    const bool lookahead = !prof && !H->opt.reserved[0];
    cudaStream_t s2 = H->stream2;
    size_t li = 0;
    for (int zl = 0; zl < H->max_lvl; ++zl) {
        const bool coopz = H->coop && (zl >= 1 || H->P2 > 1);
        if (H->my_zero[zl] && !coopz) continue;  // pdgstrf3d.c:336
        const int split_n = coopz ? (H->P2 << zl) : 1;
        const int split_i = coopz ? ((H->view.mydep & ((1 << zl) - 1)) * H->P2 + H->view.myrow * H->view.npcol + H->view.mycol) : 0;
        size_t first = (size_t)-1, last = (size_t)-1;
        for (; li < H->levels.size() && H->levels[li].zlvl <= zl; ++li) {
            const LevelPlan &L = H->levels[li];
            if (L.zlvl < zl) continue;
            if (first == (size_t)-1) first = li;
            last = li;
            const int32_t *nodes = H->d_pool_i32.p + L.nodes_off;
            const int64_t *p64 = H->d_pool_i64.p;
            Batch all{nodes, p64 + L.trsml_prefix, L.count};
            if (lookahead && li >= first + 2) CU(cudaStreamWaitEvent(s, H->ev_bulk[li - 2], 0));
            if (up_pipe) CU(cudaStreamWaitEvent(s, H->ev_up[li], 0));  // this level's A values are in the arena
            if (coopz && L.slab_end > L.slab_begin) {
                // every rank of the Z group holds a partial sum of this level's panels (its own Schur contributions,
                // plus A on the group leader): one in-place all-reduce makes them complete and identical everywhere.
                // Replaces dreduceAllAncestors3d's pairwise Send/Recv (pd3dcomm.c:1046-1081) for this forest.
                if (prof) cudaEventRecord(pe[5], s);
                NC(g_nccl.AllReduce(H->val.p + L.slab_begin, H->val.p + L.slab_begin, (size_t)(L.slab_end - L.slab_begin) * VAL_DOUBLES,
                                    NCCL_FLOAT64, NCCL_SUM, H->gcomm[zl], s));
                if (prof) { cudaEventRecord(pe[0], s); cudaEventSynchronize(pe[0]); float ms; cudaEventElapsedTime(&ms, pe[5], pe[0]); t_red += ms; }
            }
            if (prof) cudaEventRecord(pe[0], s);
            // tiny-pivot replacements are counted once: by the layer that owns the forest (not by the replicated
            // copies of a cooperative group) and by one rank of its 2D grid (stat->TinyPivots is MPI_SUMmed there,
            // pdgssvx3d.c:1149)
            const bool count_tiny = !H->my_zero[zl] && (H->P2 == 1 || (H->view.myrow == 0 && H->view.mycol == 0));
            H->st.gpu_launches += launch_diag_lu(d, all, L.max_ns, H->opt.replace_tiny_pivot ? (count_tiny ? 1 : 2) : 0, H->opt.thresh, s);
            if (prof) cudaEventRecord(pe[1], s);
            H->st.gpu_launches += launch_diag_inv(d, Batch{nodes, p64 + L.inv_prefix, L.count}, L.inv_ctas, H->d_inv.p, s);
            H->st.gpu_launches += launch_trsm_l(d, Batch{nodes, p64 + L.trsml_prefix, L.count}, L.trsml_ctas, L.max_ns, H->d_inv.p, s);
            H->st.gpu_launches += launch_trsm_u(d, Batch{nodes, p64 + L.trsmu_prefix, L.count}, L.trsmu_ctas, L.max_ns, H->d_inv.p, s);
            if (prof) cudaEventRecord(pe[2], s);
            H->st.gpu_launches += launch_schur_setup(d, Batch{nodes, p64 + L.setup_prefix, L.count}, L.setup_ctas, s);
#ifndef SLU_COMPLEX
            const int32_t *tcn = H->d_pool_i32.p + L.tc_nodes;
            if (L.tc_count > 0)      // int8 slices of the level's wide panels (final after the TRSMs above)
                H->st.gpu_launches += launch_oz_slice(d, tcn, L.tc_count, p64 + L.tc_p_rt, L.tc_n_rt, p64 + L.tc_p_ak, L.tc_n_ak,
                                                      p64 + L.tc_p_b, L.tc_n_b, H->tc_slices, s);
#endif
            if (prof) cudaEventRecord(pe[3], s);
            const int32_t *bign = H->d_pool_i32.p + L.big_nodes;
            if (lookahead || pipelined) CU(cudaEventRecord(H->ev_panel[li], s));
            if (pipelined && pipe_download_level(H, li)) return -1;
            // non-atomic scatter of exclusive destinations (tcgen05 path): this level's updates must not overlap the bulk
            // update of the level before (it targets the same ancestors); the panel work above still did
            const int tc_na = (H->tc_nonatomic && !up_pipe) ? 1 : 0;
            if (tc_na && lookahead && li >= first + 1 && (L.tc_count > 0 || H->levels[li - 1].tc_count > 0))
                CU(cudaStreamWaitEvent(s, H->ev_bulk[li - 1], 0));
            if (lookahead) {
                H->st.gpu_launches += launch_schur(d, Batch{bign, p64 + L.urg_prefix, L.big_count}, L.urg_ctas, 1, L.atomic, H->opt.schur_variant, 1, split_n, split_i, H->opt.schur_variant == 3 && L.max_ns >= 128, s);
                H->st.gpu_launches += launch_schur(d, Batch{H->d_pool_i32.p + L.small_nodes, p64 + L.small_prefix, L.small_count}, L.small_ctas, 0, L.atomic, H->opt.schur_variant, 0, split_n, split_i, H->opt.schur_variant == 3 && L.max_ns >= 128, s);
#ifndef SLU_COMPLEX
                H->st.gpu_launches += launch_oz_schur(d, Batch{tcn, p64 + L.tc_urg_prefix, L.tc_count}, L.tc_urg_ctas, 1, split_n, split_i, H->tc_slices, tc_na, s);
#endif
                CU(cudaStreamWaitEvent(s2, H->ev_panel[li], 0));
#ifndef SLU_COMPLEX
                H->st.gpu_launches += launch_oz_schur(d, Batch{tcn, p64 + L.tc_bulk_prefix, L.tc_count}, L.tc_bulk_ctas, 2, split_n, split_i, H->tc_slices, tc_na, s2);
#endif
                H->st.gpu_launches += launch_schur(d, Batch{bign, p64 + L.bulk_prefix, L.big_count}, L.bulk_ctas, 1, L.atomic, H->opt.schur_variant, 2, split_n, split_i, H->opt.schur_variant == 3 && L.max_ns >= 128, s2);
                CU(cudaEventRecord(H->ev_bulk[li], s2));
            } else {
#ifndef SLU_COMPLEX
                H->st.gpu_launches += launch_oz_schur(d, Batch{tcn, p64 + L.tc_prefix, L.tc_count}, L.tc_ctas, 0, split_n, split_i, H->tc_slices, tc_na, s);
#endif
                H->st.gpu_launches += launch_schur(d, Batch{bign, p64 + L.big_prefix, L.big_count}, L.big_ctas, 1, L.atomic, H->opt.schur_variant, 0, split_n, split_i, H->opt.schur_variant == 3 && L.max_ns >= 128, s);
                H->st.gpu_launches += launch_schur(d, Batch{H->d_pool_i32.p + L.small_nodes, p64 + L.small_prefix, L.small_count}, L.small_ctas, 0, L.atomic, H->opt.schur_variant, 0, split_n, split_i, H->opt.schur_variant == 3 && L.max_ns >= 128, s);
            }
            if (prof) {
                cudaEventRecord(pe[4], s);
                cudaEventSynchronize(pe[4]);
                float ms;
                cudaEventElapsedTime(&ms, pe[0], pe[1]); t_diag += ms;
                cudaEventElapsedTime(&ms, pe[1], pe[2]); t_trsm += ms;
                cudaEventElapsedTime(&ms, pe[2], pe[3]); t_setup += ms;
                cudaEventElapsedTime(&ms, pe[3], pe[4]); t_schur += ms;
            }
        }
        if (lookahead && last != (size_t)-1) {  // join the bulk stream before anything that reads the ancestors
            CU(cudaStreamWaitEvent(s, H->ev_bulk[last], 0));
            if (last > first) CU(cudaStreamWaitEvent(s, H->ev_bulk[last - 1], 0));
        }
        if (zl < H->max_lvl - 1 && !H->coop) {
            if (prof) cudaEventRecord(pe[0], s);
            // the pairwise reduction adds non-atomically: every upload into the ancestors must have landed
            if (up_pipe && !H->ev_up.empty()) CU(cudaStreamWaitEvent(s, H->ev_up.back(), 0));
            if (reduce_ancestors(H, zl)) return -1;
            if (prof) { cudaEventRecord(pe[1], s); cudaEventSynchronize(pe[1]); float ms; cudaEventElapsedTime(&ms, pe[0], pe[1]); t_red += ms; }
        }
    }
    if (H->comm)  // pdgstrf3d.c:388-392: MPI_Allreduce(info, MIN) over the 3D grid
        NC(g_nccl.AllReduce(H->d_flags.p, H->d_flags.p, 1, NCCL_INT32, NCCL_MIN, H->comm, s));
    CU(cudaEventRecord(H->ev1, s));
    CU(cudaStreamSynchronize(s));
    if (pipelined) CU(cudaStreamSynchronize(H->s_down));
    if (up_pipe) CU(cudaStreamSynchronize(H->s_up));
    CU(cudaGetLastError());
    float ms = 0;
    CU(cudaEventElapsedTime(&ms, H->ev0, H->ev1));
    H->st.t_factor_s = ms * 1e-3;
    int flags[2];
    unsigned long long tiny = 0;
    CU(cudaMemcpy(flags, H->d_flags.p, sizeof flags, cudaMemcpyDeviceToHost));
    CU(cudaMemcpy(&tiny, H->d_tiny.p, sizeof tiny, cudaMemcpyDeviceToHost));
    if (prof) {
        H->st.t_diag_ms = t_diag; H->st.t_trsm_ms = t_trsm; H->st.t_schur_setup_ms = t_setup; H->st.t_schur_ms = t_schur; H->st.t_reduce_ms = t_red;
    }
    H->st.tiny_pivots = (int64_t)tiny;
    if (flags[1]) return fail("%d Schur-update destinations were not found in the L/U structure", flags[1]);
    *info = flags[0] == INT_MAX ? 0 : flags[0];
    H->factored = *info == 0;
    return 0;
}

int slu_b200_factor(slu_b200_handle_t H, int *info) { return factor_impl(H, info, false); }

int slu_b200_factor_host(slu_b200_handle_t H, int *info)
{
    if (!H || !info) return fail("null argument");
    // The overlapped transfers move whole panels between the caller's arrays and the arena, which needs the U
    // skylines to equal their dense-packed form (symmetric patterns) and 1 x 1 x Pz pieces.  Anything else -- the
    // unsymmetric patterns SuperLU exists for, Pr x Pc pieces -- takes the plain path: upload (with the skyline
    // conversion), factor, download.  Same results, no overlap.
    bool overlappable = H->P2 == 1;
    for (size_t zl = 0; zl < H->znodes.size() && overlappable; ++zl)
        for (int k : H->znodes[zl])
            if (!H->u_full[k] && H->nodes[k].ncols > 0) { overlappable = false; break; }
    if (!overlappable) {
        if (slu_b200_upload(H)) return -1;
        int rc2 = factor_impl(H, info, false);
        return rc2 ? rc2 : slu_b200_download(H);
    }
    if (H->grouped) {                      // options.reserved[3]: H2D, factorization and D2H all overlapped
        H->factored = false;
        if (pipe_prepare(H) || upload_pipe_issue(H)) return -1;
        H->uploaded = true;
        H->st.t_upload_s = 0;
        int rc3 = factor_impl(H, info, true, true);
        H->st.t_download_s = 0;
        return rc3;
    }
    if (slu_b200_upload(H)) return -1;
    int rc = factor_impl(H, info, true);   // downloads every level as soon as it is final
    H->st.t_download_s = 0;
    return rc;
}

// Device-side distribution (SURVEY 8f row N1): A arrives as host CSR (the caller's matrix, perm[old] = new as
// ScalePermstruct->perm_c after sp_colorder), is copied to HBM once (12 bytes per nonzero instead of 8 bytes per FACTOR
// entry; 20 instead of 16 in doublecomplex) and scattered into the panels by a kernel -- what pddistribute3d /
// pzdistribute3d (SRC/complex16/pzdistribute3d.c:24) do on the host.  Replicated ancestors of other layers start at
// zero (dinit3DLUstructForest, pdgssvx3d.c:948).  Replaces slu_b200_upload.  Both precisions: val holds nnz elements of
// val_t ((re, im) pairs in doublecomplex).
int slu_b200_fill_csr(slu_b200_handle_t H, int n, const int32_t *rowptr, const int32_t *colind, const double *val, const int32_t *perm)
{
    if (!H || !rowptr || !colind || !val || !perm) return fail("null argument");
    if (n != H->n) return fail("matrix order %d does not match the handle's %d", n, H->n);
    if (H->P2 > 1) return fail("slu_b200_fill_csr handles 1 x 1 x Pz grids");
    double t0 = now_s();
    const int64_t nnz = rowptr[n];
    DevBuf<int32_t> drp, dci, dperm;
    DevBuf<val_t> dv;
    DevBuf<int8_t> dact;
    std::vector<int8_t> act(H->nsupers, 0);
    for (int zl = 0; zl < H->max_lvl; ++zl)
        if (!H->my_zero[zl])
            for (int k : H->znodes[zl]) act[k] = 1;
    if (drp.alloc((size_t)n + 1) || dci.alloc((size_t)nnz) || dv.alloc((size_t)nnz) || dperm.alloc((size_t)n) || dact.upload(act)) return -1;
    cudaStream_t s = H->stream;
    CU(cudaMemcpyAsync(drp.p, rowptr, ((size_t)n + 1) * sizeof(int32_t), cudaMemcpyHostToDevice, s));
    CU(cudaMemcpyAsync(dci.p, colind, (size_t)nnz * sizeof(int32_t), cudaMemcpyHostToDevice, s));
    CU(cudaMemcpyAsync(dv.p, val, (size_t)nnz * sizeof(val_t), cudaMemcpyHostToDevice, s));
    CU(cudaMemcpyAsync(dperm.p, perm, (size_t)n * sizeof(int32_t), cudaMemcpyHostToDevice, s));
    CU(cudaMemsetAsync(H->val.p, 0, H->val.bytes(), s));
    CU(cudaMemsetAsync(H->d_flags.p + 1, 0, sizeof(int), s));
    launch_fill_csr(H->dev, n, drp.p, dci.p, dv.p, dperm.p, dact.p, H->d_flags.p + 1, s);
    int bad = 0;
    CU(cudaMemcpyAsync(&bad, H->d_flags.p + 1, sizeof(int), cudaMemcpyDeviceToHost, s));
    CU(cudaStreamSynchronize(s));
    CU(cudaGetLastError());
    if (bad) return fail("%d entries of A have no slot in the L/U structure (wrong permutation or symbolic structure)", bad);
    H->st.t_upload_s = now_s() - t0;
    H->uploaded = true;
    H->factored = false;
    return 0;
}

// Triangular solves on the resident factors (the job of pdgstrs3d, SRC/double/pdgstrs3d.c:6604, and of pzgstrs3d,
// SRC/complex16/pzgstrs3d.c:6694, for factors that never left HBM); xh holds n x nrhs elements of val_t.  Along Z:
// forward, the partial vectors climb the Z tree -- an all-reduce over the group of each level, after which only the
// group's owner layer keeps the vector (the reference reduces the ancestor contributions pairwise); backward, the
// owner's solution is spread to its group the same way (dbroadcastAncestor3d, pd3dcomm.c:1145); a last all-reduce of
// the owned pieces gives every rank the full solution.
int slu_b200_solve(slu_b200_handle_t H, double *xh, int ldx, int nrhs)
{
    if (!H || !xh) return fail("null argument");
    if (!H->factored) return fail("slu_b200_solve needs a successful slu_b200_factor on this handle first");
    if (nrhs < 1 || ldx < H->n) return fail("bad nrhs / ldx");
    if (H->P2 > 1) return fail("slu_b200_solve: Pr x Pc > 1 is not supported yet (1 x 1 x Pz only)");
    if (H->comm && !H->coop) return fail("slu_b200_solve: the Z-distributed solve needs the cooperative schedule (options.reserved[1] = 0)");
    const int n = H->n;
    const size_t len = (size_t)n * nrhs;
    if (H->d_x.n < len && (H->d_x.alloc(len) || H->d_x2.alloc(len))) return -1;
    cudaStream_t s = H->stream;
    const DeviceLU &d = H->dev;
    val_t *x = H->d_x.p, *x2 = H->d_x2.p;
    double t0 = now_s();
    CU(cudaMemcpy2DAsync(x2, (size_t)n * sizeof(val_t), xh, (size_t)ldx * sizeof(val_t), (size_t)n * sizeof(val_t), (size_t)nrhs,
                         cudaMemcpyHostToDevice, s));
    const bool multi = H->comm != nullptr;
    int launches = 0;
    auto forest_nodes = [&](int zl) { return H->d_pool_i32.p + H->z_nodes_off[zl]; };
    if (multi) {      // start from the entries this rank owns: b on the owner layer of every forest, 0 elsewhere
        CU(cudaMemsetAsync(x, 0, len * sizeof(val_t), s));
        for (int zl = 0; zl < H->max_lvl; ++zl)
            if (!H->my_zero[zl]) launches += launch_solve_mask(d, forest_nodes(zl), (int)H->znodes[zl].size(), x, n, nrhs, x2, s);
    } else {
        CU(cudaMemcpyAsync(x, x2, len * sizeof(val_t), cudaMemcpyDeviceToDevice, s));
    }
    const int64_t *p64 = H->d_pool_i64.p;
    // forward: L y = b
    size_t li = 0;
    for (int zl = 0; zl < H->max_lvl; ++zl) {
        if (multi && zl >= 1) {
            NC(g_nccl.AllReduce(x, x, len * VAL_DOUBLES, NCCL_FLOAT64, NCCL_SUM, H->gcomm[zl], s));
            if (H->my_zero[zl]) CU(cudaMemsetAsync(x, 0, len * sizeof(val_t), s));
        }
        for (; li < H->levels.size() && H->levels[li].zlvl <= zl; ++li) {
            const LevelPlan &L = H->levels[li];
            if (L.zlvl < zl || H->my_zero[zl]) continue;
            const int32_t *nodes = H->d_pool_i32.p + L.nodes_off;
            launches += launch_solve_diag(d, nodes, L.count, false, x, n, nrhs, s);
            launches += launch_solve_update(d, Batch{nodes, p64 + L.sl_prefix, L.count}, L.sl_ctas, false, x, n, nrhs, s);
        }
    }
    // backward: U x = y
    li = H->levels.size();
    for (int zl = H->max_lvl - 1; zl >= 0; --zl) {
        size_t lo = li;
        while (lo > 0 && H->levels[lo - 1].zlvl >= zl) --lo;
        if (!H->my_zero[zl])
            for (size_t q = li; q-- > lo;) {
                const LevelPlan &L = H->levels[q];
                if (L.zlvl != zl) continue;
                const int32_t *nodes = H->d_pool_i32.p + L.nodes_off;
                launches += launch_solve_update(d, Batch{nodes, p64 + L.su_prefix, L.count}, L.su_ctas, true, x, n, nrhs, s);
                launches += launch_solve_diag(d, nodes, L.count, true, x, n, nrhs, s);
            }
        li = lo;
        if (multi && zl >= 1) {
            if (H->my_zero[zl]) CU(cudaMemsetAsync(x, 0, len * sizeof(val_t), s));
            NC(g_nccl.AllReduce(x, x, len * VAL_DOUBLES, NCCL_FLOAT64, NCCL_SUM, H->gcomm[zl], s));
        }
    }
    val_t *result = x;
    if (multi) {      // every rank contributes the entries it owns: the full solution everywhere
        CU(cudaMemsetAsync(x2, 0, len * sizeof(val_t), s));
        for (int zl = 0; zl < H->max_lvl; ++zl)
            if (!H->my_zero[zl]) launches += launch_solve_mask(d, forest_nodes(zl), (int)H->znodes[zl].size(), x2, n, nrhs, x, s);
        NC(g_nccl.AllReduce(x2, x2, len * VAL_DOUBLES, NCCL_FLOAT64, NCCL_SUM, H->comm, s));
        result = x2;
    }
    CU(cudaMemcpy2DAsync(xh, (size_t)ldx * sizeof(val_t), result, (size_t)n * sizeof(val_t), (size_t)n * sizeof(val_t), (size_t)nrhs,
                         cudaMemcpyDeviceToHost, s));
    CU(cudaStreamSynchronize(s));
    CU(cudaGetLastError());
    H->st.reserved[4] = now_s() - t0;      // seconds of the last solve (H2D of b and D2H of x included)
    H->st.reserved[5] = (double)launches;
    return 0;
}

#ifndef SLU_COMPLEX
// ---- benchmark support (SURVEY 8a row a10: the reference's GPU Schur path is "to be beaten") ------------------------
// Export what an EXTERNAL baseline needs to redo one level's Schur updates on this handle's device data: the DeviceLU
// struct (device pointers) and the ids of the level's supernodes with a big (>= 96 x 96) update.  oracle/ref_gpu_schur.cu
// uses it to time cublasDgemm into a bigV buffer + a restatement of the reference's Scatter_GPU_kernel on exactly the
// same operands; slu_b200_k_rerun_schur times this library's fused kernel on them.
int slu_b200_k_level_export(slu_b200_handle_t H, int level, void *device_lu, int device_lu_bytes, int32_t *nodes, int max_nodes)
{
    if (!H || level < 0 || level >= (int)H->levels.size()) return fail("bad handle / level");
    if (device_lu && device_lu_bytes == (int)sizeof(DeviceLU)) memcpy(device_lu, &H->dev, sizeof(DeviceLU));
    else if (device_lu) return fail("DeviceLU is %d bytes", (int)sizeof(DeviceLU));
    const LevelPlan &L = H->levels[level];
    int cnt = 0;
    for (int pass = 0; pass < 2; ++pass) {
        const int64_t off = pass ? L.tc_nodes : L.big_nodes;
        const int c = pass ? L.tc_count : L.big_count;
        for (int t = 0; t < c; ++t, ++cnt)
            if (nodes && cnt < max_nodes) nodes[cnt] = H->h_pool_i32[off + t];
    }
    return cnt;
}
// Re-run the destination maps + the fused Schur kernels of one level `reps` times on whatever the arena holds (timing
// only: the values are updated again and again); *ms = mean device time of the Schur launches of the level.
int slu_b200_k_rerun_schur(slu_b200_handle_t H, int level, int reps, float *ms)
{
    if (!H || level < 0 || level >= (int)H->levels.size() || reps < 1 || !ms) return fail("bad argument");
    const LevelPlan &L = H->levels[level];
    cudaStream_t s = H->stream;
    const DeviceLU &d = H->dev;
    const int32_t *nodes = H->d_pool_i32.p + L.nodes_off;
    const int64_t *p64 = H->d_pool_i64.p;
    EventSet ev;
    if (ev.create()) return fail("cannot create events");
    launch_schur_setup(d, Batch{nodes, p64 + L.setup_prefix, L.count}, L.setup_ctas, s);
    const int32_t *tcn = H->d_pool_i32.p + L.tc_nodes;
    if (L.tc_count > 0)
        launch_oz_slice(d, tcn, L.tc_count, p64 + L.tc_p_rt, L.tc_n_rt, p64 + L.tc_p_ak, L.tc_n_ak, p64 + L.tc_p_b, L.tc_n_b, H->tc_slices, s);
    for (int r = -1; r < reps; ++r) {
        if (r == 0) CU(cudaEventRecord(ev[0], s));
        launch_oz_schur(d, Batch{tcn, p64 + L.tc_prefix, L.tc_count}, L.tc_ctas, 0, 1, 0, H->tc_slices, 0, s);
        launch_schur(d, Batch{H->d_pool_i32.p + L.big_nodes, p64 + L.big_prefix, L.big_count}, L.big_ctas, 1, L.atomic, H->opt.schur_variant, 0, 1, 0, 0, s);
    }
    CU(cudaEventRecord(ev[1], s));
    CU(cudaStreamSynchronize(s));
    CU(cudaGetLastError());
    float t = 0;
    CU(cudaEventElapsedTime(&t, ev[0], ev[1]));
    *ms = t / reps;
    return 0;
}
#endif

int slu_b200_get_stats(slu_b200_handle_t H, slu_b200_stats_t *out)
{
    if (!H || !out) return fail("null argument");
    *out = H->st;
    return 0;
}

int pdgstrf3d_b200(const slu_b200_lu_view_t *lu, const slu_b200_options_t *opt, slu_b200_stats_t *stats, int *info)
{
    slu_b200_handle_t H = nullptr;
    if (slu_b200_create(&H, lu, opt)) return -1;
    int rc;
    if (opt->reserved[2]) {
        rc = slu_b200_factor_host(H, info);   // overlapped H2D / factor / D2H
    } else {
        rc = slu_b200_upload(H);
        if (!rc) rc = slu_b200_factor(H, info);
        if (!rc) rc = slu_b200_download(H);
    }
    if (stats) *stats = H->st;
    slu_b200_destroy(H);
    return rc;
}

// Analysis only, no device needed: HBM bytes, flops in the reference's accounting, level count ... for one rank of a
// 1 x 1 x Pz grid -- what a caller needs to size a run for 180 GB GPUs before it allocates them.  Also checks the
// level-by-level layout that the overlapped upload (options.reserved[3]) relies on.
int slu_b200_plan(const slu_b200_lu_view_t *lu, const slu_b200_options_t *opt, slu_b200_stats_t *stats)
{
    if (!lu || !opt || !stats) return fail("null argument");
    if (lu->nprow * lu->npcol != 1) return fail("slu_b200_plan handles 1 x 1 x Pz grids (a Pr x Pc layer needs its peers' index pieces)");
    struct Guard { Guard() { g_plan_only = true; } ~Guard() { g_plan_only = false; } } guard;
    slu_b200_handle_s *H = new slu_b200_handle_s;
    H->view = *lu;
    H->opt = *opt;
    H->coop = opt->world_size > 1 && !opt->reserved[1];
    H->P2 = 1;
    int rc = (gather_structure(H) || analyze(H)) ? -1 : 0;
    if (!rc && H->grouped)
        for (size_t li = 0; li < H->levels.size() && !rc; ++li) {
            const LevelPlan &L = H->levels[li];
            const int32_t *nodes = H->h_pool_i32.data() + L.nodes_off;
            int64_t off = L.slab_begin;
            for (int pass = 0; pass < 2 && !rc; ++pass)
                for (int t = 0; t < L.count; ++t) {
                    const NodeDesc &nd = H->nodes[nodes[t]];
                    const int64_t dev = pass ? nd.uval : nd.lval;
                    const int64_t len = pass ? (int64_t)nd.ns * nd.ncols : (int64_t)nd.nsupr * nd.ns;
                    if (len <= 0) continue;
                    if (dev != off) { rc = fail("level %zu is not contiguous in the arena", li); break; }
                    off += len;
                }
            if (!rc && off != L.slab_end) rc = fail("level %zu: slab end mismatch", li);
        }
    if (!rc) *stats = H->st;
    delete H;
    return rc;
}

// ---- kernel-level entry points -----------------------------------------------------------------
namespace {
struct MiniLU {  // a one-supernode DeviceLU around a caller-provided block
    DevBuf<val_t> val;
    DevBuf<NodeDesc> nodes;
    DevBuf<int32_t> ids;
    DevBuf<int64_t> prefix;
    DevBuf<int> flags;
    DevBuf<unsigned long long> tiny;
    DevBuf<val_t> inv;
    DeviceLU d{};
    int init(const NodeDesc &nd, size_t nval, const std::vector<int64_t> &pre)
    {
        if (val.alloc(nval) || nodes.upload(std::vector<NodeDesc>{nd}) || ids.upload(std::vector<int32_t>{0}) ||
            prefix.upload(pre) || flags.alloc(2) || tiny.alloc(1))
            return -1;
        int init[2] = {INT_MAX, 0};
        cudaMemcpy(flags.p, init, sizeof init, cudaMemcpyHostToDevice);
        cudaMemset(tiny.p, 0, 8);
        d.val = val.p; d.nodes = nodes.p; d.info = flags.p; d.err = flags.p + 1; d.tiny = tiny.p;
        return 0;
    }
    ~MiniLU() { val.release(); nodes.release(); ids.release(); prefix.release(); flags.release(); tiny.release(); inv.release(); }
};
}  // namespace

int slu_b200_k_diag_lu(double *a, int ns, int lda, int replace_tiny, double thresh, int col0, int *info, int *tiny)
{
    if (slu_b200_device_count() < 1) return fail("no CUDA device");
    if (ns < 1 || ns > MAX_NS_HELD || lda < ns) return fail("bad size");
    MiniLU M;
    NodeDesc nd{}; nd.held = 1; nd.ns = ns; nd.nsupr = lda; nd.fsupc = col0; nd.lval = 0;
    if (M.init(nd, (size_t)lda * ns, {0, 1})) return -1;
    CU(cudaMemcpy(M.val.p, a, (size_t)lda * ns * sizeof(val_t), cudaMemcpyHostToDevice));
    launch_diag_lu(M.d, Batch{M.ids.p, M.prefix.p, 1}, ns, replace_tiny, thresh, 0);
    CU(cudaDeviceSynchronize());
    CU(cudaGetLastError());
    CU(cudaMemcpy(a, M.val.p, (size_t)lda * ns * sizeof(val_t), cudaMemcpyDeviceToHost));
    int flags[2]; unsigned long long t;
    CU(cudaMemcpy(flags, M.flags.p, sizeof flags, cudaMemcpyDeviceToHost));
    CU(cudaMemcpy(&t, M.tiny.p, 8, cudaMemcpyDeviceToHost));
    if (info) *info = flags[0] == INT_MAX ? 0 : flags[0];
    if (tiny) *tiny = (int)t;
    return 0;
}

static int k_trsm(bool ucase, const double *lu_, int ldlu, int ns, double *x_, int nvec, int ldx)
{
    const val_t *lu = (const val_t *)lu_;
    val_t *x = (val_t *)x_;
    if (slu_b200_device_count() < 1) return fail("no CUDA device");
    if (ns < 1 || ns > MAX_NS_HELD || ldlu < ns || nvec < 0) return fail("bad size");
    // assemble a panel: L case [diag (ns rows) ; x (m rows)] with lda = ns + m; U case diag + packed U
    MiniLU M;
    NodeDesc nd{}; nd.held = 1; nd.ns = ns; nd.lval = 0;
    size_t nval;
    std::vector<val_t> h;
    if (!ucase) {
        nd.nsupr = ns + nvec; nd.m = nvec;
        nval = (size_t)nd.nsupr * ns;
        h.assign(nval, val_t{});
        for (int c = 0; c < ns; ++c) {
            for (int r = 0; r < ns; ++r) h[(size_t)c * nd.nsupr + r] = lu[(size_t)c * ldlu + r];
            for (int r = 0; r < nvec; ++r) h[(size_t)c * nd.nsupr + ns + r] = x[(size_t)c * ldx + r];
        }
    } else {
        nd.nsupr = ns; nd.m = 0; nd.ncols = nvec; nd.uval = (int64_t)ns * ns;
        nval = (size_t)ns * ns + (size_t)ns * nvec;
        h.assign(nval, val_t{});
        for (int c = 0; c < ns; ++c)
            for (int r = 0; r < ns; ++r) h[(size_t)c * ns + r] = lu[(size_t)c * ldlu + r];
        for (int c = 0; c < nvec; ++c)
            for (int r = 0; r < ns; ++r) h[(size_t)ns * ns + (size_t)c * ns + r] = x[(size_t)c * ldx + r];
    }
    int64_t ctas = (nvec + trsm_strip_of(ns) - 1) / trsm_strip_of(ns);
    if (M.init(nd, nval, {0, ctas})) return -1;
    CU(cudaMemcpy(M.val.p, h.data(), nval * sizeof(val_t), cudaMemcpyHostToDevice));
    Batch b{M.ids.p, M.prefix.p, 1};
    const int nb16 = (ns + 15) / 16;
    DevBuf<int64_t> pinv;
    if (M.inv.alloc((size_t)nb16 * 512) || pinv.upload(std::vector<int64_t>{0, nb16})) return -1;
    launch_diag_inv(M.d, Batch{M.ids.p, pinv.p, 1}, nb16, M.inv.p, 0);
    if (ucase) launch_trsm_u(M.d, b, ctas, ns, M.inv.p, 0); else launch_trsm_l(M.d, b, ctas, ns, M.inv.p, 0);
    CU(cudaDeviceSynchronize());
    pinv.release();
    CU(cudaDeviceSynchronize());
    CU(cudaGetLastError());
    CU(cudaMemcpy(h.data(), M.val.p, nval * sizeof(val_t), cudaMemcpyDeviceToHost));
    if (!ucase) {
        for (int c = 0; c < ns; ++c)
            for (int r = 0; r < nvec; ++r) x[(size_t)c * ldx + r] = h[(size_t)c * nd.nsupr + ns + r];
    } else {
        for (int c = 0; c < nvec; ++c)
            for (int r = 0; r < ns; ++r) x[(size_t)c * ldx + r] = h[(size_t)ns * ns + (size_t)c * ns + r];
    }
    return 0;
}
int slu_b200_k_trsm_l(const double *lu, int ldlu, int ns, double *x, int m, int ldx) { return k_trsm(false, lu, ldlu, ns, x, m, ldx); }
int slu_b200_k_trsm_u(const double *lu, int ldlu, int ns, double *x, int ncols, int ldx) { return k_trsm(true, lu, ldlu, ns, x, ncols, ldx); }

int slu_b200_k_gemm_sub(int m, int n, int k, const double *a, int lda, const double *b, int ldb, double *c, int ldc,
                        int reps, float *ms)
{
    const int variant = getenv("SLU_B200_GEMM_VARIANT") ? atoi(getenv("SLU_B200_GEMM_VARIANT")) : 0;
    if (slu_b200_device_count() < 1) return fail("no CUDA device");
    DevBuf<val_t> da, db, dc;
    if (da.alloc((size_t)lda * k) || db.alloc((size_t)ldb * n) || dc.alloc((size_t)ldc * n)) return -1;
    CU(cudaMemcpy(da.p, a, (size_t)lda * k * sizeof(val_t), cudaMemcpyHostToDevice));
    CU(cudaMemcpy(db.p, b, (size_t)ldb * n * sizeof(val_t), cudaMemcpyHostToDevice));
    CU(cudaMemcpy(dc.p, c, (size_t)ldc * n * sizeof(val_t), cudaMemcpyHostToDevice));
    EventSet ev;
    if (ev.create()) return fail("cannot create events");
    cudaEvent_t e0 = ev[0], e1 = ev[1];
#ifndef SLU_COMPLEX
    auto launch_gemm_sub = [](int m_, int n_, int k_, const val_t *a_, int lda_, const val_t *b_, int ldb_, val_t *c_, int ldc_,
                              int variant_, cudaStream_t s_) {
        if (variant_ >= 100) return launch_gemm_sub_ozaki(m_, n_, k_, a_, lda_, b_, ldb_, c_, ldc_, variant_, s_);
        return SLU_NS::launch_gemm_sub(m_, n_, k_, a_, lda_, b_, ldb_, c_, ldc_, variant_, s_);
    };
    if (variant >= 100 && k > 512) return fail("the tcgen05 path handles k <= 512 (MAX_SUPER_SIZE)");
#endif
    launch_gemm_sub(m, n, k, da.p, lda, db.p, ldb, dc.p, ldc, variant, 0);
    CU(cudaDeviceSynchronize());
    CU(cudaGetLastError());
    CU(cudaMemcpy(c, dc.p, (size_t)ldc * n * sizeof(val_t), cudaMemcpyDeviceToHost));
    if (reps > 0) {
        cudaEventRecord(e0, 0);
        for (int r = 0; r < reps; ++r) launch_gemm_sub(m, n, k, da.p, lda, db.p, ldb, dc.p, ldc, variant, 0);
        cudaEventRecord(e1, 0);
        CU(cudaEventSynchronize(e1));
        float t = 0;
        cudaEventElapsedTime(&t, e0, e1);
        if (ms) *ms = t / reps;
    }
    return 0;
}

}  // extern "C"
