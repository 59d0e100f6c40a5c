// dhqr_api.cu — context, workspace, panel/update drivers and the C-ABI of libdhqr.so.
// See include/dhqr.h for the contract; each entry point names the reference method it replaces
// (S:n = /root/reference/src/DistributedHouseholderQR.jl:n).
#include "../../include/dhqr.h"

#include <cuda_runtime.h>
#include <dlfcn.h>
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <time.h>

#include <algorithm>
#include <memory>
#include <utility>
#include <vector>

#include "dhqr_kernels.cuh"
#include "dhqr_wide.cuh"
#include "dhqr_complex.cuh"

using namespace dhqr;

// ------------------------------------------------------------------------------------------------
// errors
// ------------------------------------------------------------------------------------------------
static thread_local char g_err[512] = "";
static int set_err(int code, const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
    return code;
}
#define CU(call)                                                                                         \
    do {                                                                                                 \
        cudaError_t e_ = (call);                                                                         \
        if (e_ != cudaSuccess)                                                                           \
            return set_err(1000 + (int)e_, "%s failed at %s:%d: %s", #call, __FILE__, __LINE__, cudaGetErrorString(e_)); \
    } while (0)
#define TRY(call)          \
    do {                   \
        int rc_ = (call);  \
        if (rc_) return rc_; \
    } while (0)

// ------------------------------------------------------------------------------------------------
// NCCL, loaded lazily so that single-GPU use needs no NCCL at all
// ------------------------------------------------------------------------------------------------
typedef struct ncclComm* ncclComm_t;
typedef struct { char internal[128]; } ncclUniqueId;
typedef int ncclResult_t;
enum { ncclFloat64 = 8, ncclInt64 = 4, ncclSum = 0 };
struct NcclApi {
    void* lib = nullptr;
    ncclResult_t (*GetUniqueId)(ncclUniqueId*) = nullptr;
    ncclResult_t (*CommInitRank)(ncclComm_t*, int, ncclUniqueId, int) = nullptr;
    ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
    ncclResult_t (*Broadcast)(const void*, void*, size_t, int, int, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*AllGather)(const void*, void*, size_t, int, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*Send)(const void*, size_t, int, int, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*Recv)(void*, size_t, int, int, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*GroupStart)() = nullptr;
    ncclResult_t (*GroupEnd)() = nullptr;
    const char* (*GetErrorString)(ncclResult_t) = nullptr;
};
static NcclApi g_nccl;
static int load_nccl() {
    if (g_nccl.lib) return 0;
    // An already-loaded libnccl.so.2 (e.g. the one bundled with torch) is reused by soname.
    const char* names[] = {"libnccl.so.2", "libnccl.so"};
    for (const char* nm : names) {
        g_nccl.lib = dlopen(nm, RTLD_NOW | RTLD_GLOBAL);
        if (g_nccl.lib) break;
    }
    if (!g_nccl.lib) return set_err(2001, "cannot dlopen libnccl.so.2: %s", dlerror());
#define SYM(field, name)                                                       \
    *(void**)(&g_nccl.field) = dlsym(g_nccl.lib, name);                        \
    if (!g_nccl.field) return set_err(2002, "libnccl lacks symbol %s", name);
    SYM(GetUniqueId, "ncclGetUniqueId")
    SYM(CommInitRank, "ncclCommInitRank")
    SYM(CommDestroy, "ncclCommDestroy")
    SYM(Broadcast, "ncclBroadcast")
    SYM(AllGather, "ncclAllGather")
    SYM(Send, "ncclSend")
    SYM(Recv, "ncclRecv")
    SYM(GroupStart, "ncclGroupStart")
    SYM(GroupEnd, "ncclGroupEnd")
    SYM(GetErrorString, "ncclGetErrorString")
#undef SYM
    return 0;
}
#define NC(call)                                                                                              \
    do {                                                                                                      \
        ncclResult_t r_ = (call);                                                                             \
        if (r_ != 0) return set_err(3000 + (int)r_, "%s failed at %s:%d: %s", #call, __FILE__, __LINE__, g_nccl.GetErrorString(r_)); \
    } while (0)

// ------------------------------------------------------------------------------------------------
// context
// ------------------------------------------------------------------------------------------------
static inline int64_t rup(int64_t x, int64_t a) { return (x + a - 1) / a * a; }

static constexpr int CU_STREAMS = 3;   // catch-up streams of dhqr_qr_host_f64, each with its own V buffer and workspace set

// Owners of the handle's CUDA resources: each releases what it holds when it goes, so neither a failed call nor
// dhqr_destroy has to know the list of buffers, streams and events.
template <typename T>
class DevBuf {   // one zero-filled cudaMalloc allocation and its element count
  public:
    DevBuf() = default;
    DevBuf(DevBuf&& o) noexcept : p_(o.p_), n_(o.n_) { o.p_ = nullptr; o.n_ = 0; }
    ~DevBuf() { if (p_) cudaFree(p_); }
    operator T*() const { return p_; }
    size_t size() const { return n_; }
    // at least `need` elements: a smaller allocation is freed first and replaced by a zero-filled one of exactly `need`;
    // *grown says whether that happened
    int grow(size_t need, bool* grown = nullptr) {
        if (grown) *grown = false;
        if (n_ >= need && p_) return 0;
        if (p_) CU(cudaFree(p_));
        p_ = nullptr;
        n_ = 0;
        CU(cudaMalloc((void**)&p_, need * sizeof(T)));
        CU(cudaMemset(p_, 0, need * sizeof(T)));
        n_ = need;
        if (grown) *grown = true;
        return 0;
    }
  private:
    T* p_ = nullptr;
    size_t n_ = 0;
};
class Stream {   // a non-blocking stream
  public:
    Stream() = default;
    Stream(const Stream&) = delete;
    Stream& operator=(const Stream&) = delete;
    ~Stream() { if (s_) cudaStreamDestroy(s_); }
    operator cudaStream_t() const { return s_; }
    cudaError_t create() { return cudaStreamCreateWithFlags(&s_, cudaStreamNonBlocking); }
    cudaError_t create(int priority) { return cudaStreamCreateWithPriority(&s_, cudaStreamNonBlocking, priority); }
  private:
    cudaStream_t s_ = nullptr;
};
class Event {   // may go as soon as the work it orders is enqueued; a std::vector<Event> is the event list of one call
  public:
    Event() = default;
    Event(Event&& o) noexcept : e_(o.e_) { o.e_ = nullptr; }
    Event& operator=(Event&& o) noexcept { std::swap(e_, o.e_); return *this; }
    ~Event() { if (e_) cudaEventDestroy(e_); }
    operator cudaEvent_t() const { return e_; }
    cudaError_t create(unsigned flags) { *this = Event(); return cudaEventCreateWithFlags(&e_, flags); }
  private:
    cudaEvent_t e_ = nullptr;
};

struct dhqr_context {
    int device = 0, sms = 0;
    int rank = 0, nranks = 1;
    ncclComm_t comm = nullptr;
    // options
    int nb = 128, sync = 0;
    // workspace
    // three V buffers (panels k, k+1 and the one being broadcast live at the same time under look-ahead) and two
    // workspace sets (set 0: trailing update on the caller's stream; set 1: panel chain on the high-priority stream)
    DevBuf<double> vpk2[3 + CU_STREAMS];                                // packed V [chunk][128][68]; [3..]: catch-up of late column chunks (host entry)
    struct WSet {
        DevBuf<double> wpart;                                           // gemm_vta partials
        DevBuf<double> wsum;                                            // reduced Wext
        DevBuf<double> ypk;                                             // packed Y = -T'W
        DevBuf<double> linv;                                            // [128*128]
    } ws[3 + CU_STREAMS];                                               // [2]: the chain's second apply (columns of panel k+2) on its own stream; [3..]: catch-up (host entry)
    DevBuf<double> linv_all;                                            // T' of every outer panel of the factorisation in flight (look-ahead): slot k = panel k
    double* tslot(int k) const { return linv_all + (size_t)k * 128 * 128; }
    Stream hp_stream;                                                   // stream of the panel chain (high priority)
    Stream comm_stream;                                                 // collectives of the look-ahead schedule (high priority)
    Stream aux_stream;                                                  // small side kernels of the wide chain (Rt = R2 R1, k_trecon), high priority
    Event ev_aux[4];
    Stream hp2_stream;                                                  // the chain's second apply (V_k -> columns of panel k+2), high priority
    int host_trace = 0;                                                 // option: print a stage timeline of dhqr_qr_host_f64 to stderr
    int lookahead = 1;
    DevBuf<unsigned long long> cells;                                   // panel exchange cells [IB+1][MAXG+1][IB][2]
    uint32_t ll_epoch = 0;
    DevBuf<unsigned long long> cells2;                                  // exchange cells of the panel kernel's fast path
    DevBuf<int> fast_stats;                                             // [2] fast / fallback panel counters
    int panel_fast = 1;
    int bs_wave_max_ctas = 0;                                           // co-residency limit of k_backsolve_wave on this device
    DevBuf<unsigned long long> bs_cells;                                // x cells of the wavefront ([block][32][2 words])
    uint32_t bs_epoch = 0;
    DevBuf<unsigned int> uw_flags; unsigned int uw_epoch = 0;           // k_unblocked_wave column flags
    // 128-column panel chain (dhqr_wide.cuh)
    int wide_panel = 1;                                                 // option: factor full aligned outer panels with CholeskyQR2 + reconstruction
    DevBuf<WideCtl> wctl;                                               // device control words (first refused panel, guards of the panel in flight)
    DevBuf<double> wbuf;                                                // R1, R2, X2, Rt, Y3 (plain 128x128) + XL, XL3 (rmul operand layout)
    int64_t wide_panels = 0, wide_redone = 0;                           // statistics: panels factored by the wide chain / factorisations restarted
    double wide_kappa = 1000.0;                                         // guard on ||D R1^{-1}||_F of the first Cholesky factor (option "wide_kappa")
    // Q'b / Qb with one right-hand side: T' of every local panel (computed before the sweep), per-CTA partials of V'b, y, ticket
    DevBuf<double> qt_T;
    DevBuf<double> qt_part; DevBuf<unsigned int> qt_ticket;
    int qt_vec = 1;                                                     // option: use it (0: the GEMM-shaped block update also for one right-hand side)
    DevBuf<double> v1;                                                  // unblocked path: v
    DevBuf<double> xbuf;                                                // back-substitution output
    DevBuf<double> hostA;                                               // device staging for _host_ entry points
    DevBuf<double> hostB;
    DevBuf<int64_t> d_i64;                                              // small int64 scratch (partition exchange)
    int64_t launches = 0;
    Stream copy_stream;                      // compute stream of the _host_ entry points
    Stream d2h_stream;                       // drains finished panels to the host while the factorisation continues
    Stream h2d_stream;                       // uploads the later column chunks while the first ones are being factored
    Stream cu_stream[CU_STREAMS];            // catch-up: reflectors of finished panels applied to a column chunk that arrived late (chunks alternate)
    // dhqr_qr_host_f64 -> look-ahead driver: column chunks still on their way to the device.  Chunk j = global columns [c0, c1),
    // usable once `ev` has fired, joins the trailing matrix at step `join` (after a catch-up with the reflectors of panels < join)
    struct UpChunk { int64_t c0, c1; cudaEvent_t ev; int join; };
    std::vector<UpChunk> up_chunks;
    int host_chunk = 512;                    // option: columns per upload chunk (0: one upload, no overlap)
    int host_first = 0;                      // option: columns of the first upload (0: three panels)
    int host_h2d_gbs = 50, host_tflops = 27; // option: what the join-step planner assumes about the link and the device
    int host_chain_us = 300;                 // option: ... and about the duration of a step of the schedule while the window is narrow
    std::vector<Event> panel_events;
    // set by dhqr_qr_host_f64: finished columns are copied back as soon as their panel is final
    double* mirror_host = nullptr;
    int64_t mirror_lda = 0;
    // kernel attribute state
    bool attrs_set = false;
    // per-kernel-class CUDA-event profiling (option "profile")
    int profile = 0;
    struct ProfRec { int slot; Event e0, e1; };
    struct ProfSlot { const char* name; double ms = 0.0; int64_t count = 0; double work = 0.0; };
    std::vector<ProfRec> prof_pending;
    std::vector<ProfSlot> prof_slots;
    Event prof_open;
};

static constexpr int NBMAX = 128;
static constexpr int MAXCTAS_FACTOR = 3;

// gemm tile configurations
static constexpr int G1_BN = 64, G1_NPW = 2;                // gemm_vta<128>: 128 x 64 tile, 8 MMA + 2 TMA warps
static constexpr int G1S_BN = 128, G1S_NPW = 4;             // gemm_vta<32> : 32 x 128 tile, 4 MMA + 4 TMA warps
static constexpr int G2_BM = 128, G2_BN = YT;               // gemm_cvy: 128 x 64 tile, 8 MMA + 1 TMA warps, 2 CTAs/SM
static constexpr int CVY_TILES_PER_CTA = 1;                 // gemm_cvy_p: tiles one CTA walks through (short-lived CTAs leave SMs to the panel chain)

static size_t smem_g1(int nbp, int bn) { return (size_t)2 * (nbp + bn) * LD1 * 8 + 4 * 8; }
static size_t smem_g2() { return (size_t)2 * (2 * KC * LD1 + G2_BN * LDK) * 8 + 4 * 8; }
static size_t smem_tinv(int nbp) { return ((size_t)nbp * (nbp + 1) + 4 * 32 * 33 + (nbp == 128 ? 64 * 65 : 0)) * 8; }
static size_t smem_ymake(int nbp) { return ((size_t)nbp * nbp + YCOLS * nbp) * 8; }

#define K_G1_128 k_gemm_vta<128, G1_BN, 4, 2, G1_NPW>
#define K_G1_32 k_gemm_vta<32, G1S_BN, 1, 4, G1S_NPW>

static int set_attrs(dhqr_context* c) {
    if (c->attrs_set) return 0;
    CU(cudaFuncSetAttribute(K_G1_128, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_g1(128, G1_BN)));
    CU(cudaFuncSetAttribute(K_G1_32, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_g1(32, G1S_BN)));
    CU(cudaFuncSetAttribute(k_gemm_cvy, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_g2()));
    CU(cudaFuncSetAttribute(k_gemm_cvy, cudaFuncAttributePreferredSharedMemoryCarveout, 100));
    CU(cudaFuncSetAttribute(k_gemm_cvy_p, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_g2()));
    CU(cudaFuncSetAttribute(k_gemm_cvy_p, cudaFuncAttributePreferredSharedMemoryCarveout, 100));
    CU(cudaFuncSetAttribute(k_gram_sym, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SMEM_GRAM_SYM));
    CU(cudaFuncSetAttribute(k_tinv<128>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_tinv(128)));
    CU(cudaFuncSetAttribute(k_tinv<32>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_tinv(32)));
    CU(cudaFuncSetAttribute(k_ymake<128>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_ymake(128)));
    CU(cudaFuncSetAttribute(k_ymake<32>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_ymake(32)));
    CU(cudaFuncSetAttribute(k_panel, cudaFuncAttributeMaxDynamicSharedMemorySize, 184 * 1024));
    CU(cudaFuncSetAttribute(k_chol128, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SMEM_WIDE1));
    CU(cudaFuncSetAttribute(k_hr128, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SMEM_WIDE1));
    CU(cudaFuncSetAttribute(k_vpk_rmul, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SMEM_RMUL));
    CU(cudaFuncSetAttribute(k_trimm128, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SMEM_TRIMM));
    CU(cudaFuncSetAttribute(k_trimm_z, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SMEM_TRIMM));
    CU(cudaFuncSetAttribute(k_trecon, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SMEM_TRECON));
    CU(cudaFuncSetAttribute(k_apply1_tma, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
    c->attrs_set = true;
    return 0;
}

static constexpr int64_t WPART_TILES = 2304;   // capacity of the partial buffer in 128 x 64 tiles (151 MB per set)

// npanels: outer panels of the factorisation about to run (T' slots of the look-ahead schedule); catchup: also size the fourth
// V buffer / workspace set (dhqr_qr_host_f64 only)
static int ensure_workspace(dhqr_context* c, int64_t m, int64_t n_local_max, int64_t npanels = 0, bool catchup = false) {
    TRY(set_attrs(c));
    const int64_t vrows = rup(m, 128) + 128;
    for (int b = 0; b < (catchup ? 3 + CU_STREAMS : 3); ++b) TRY(c->vpk2[b].grow((size_t)(vrows / KC1) * VPK_CHUNK));
    TRY(c->linv_all.grow((size_t)std::max<int64_t>(npanels, 4) * NBMAX * NBMAX));
    const int64_t tiles_max = (n_local_max + NBMAX + G1_BN - 1) / G1_BN + 1;
    for (int b = 0; b < (catchup ? 3 + CU_STREAMS : 3); ++b) {
        auto& w = c->ws[b];
        // set 2 only ever updates the <= 128 columns of one panel: a quarter of the split-K partial buffer is plenty
        TRY(w.wpart.grow((size_t)(b != 2 ? std::max(WPART_TILES, tiles_max) : WPART_TILES / 4) * NBMAX * G1_BN));
        TRY(w.wsum.grow((size_t)NBMAX * (rup(n_local_max + NBMAX, 128) + 128)));
        TRY(w.ypk.grow((size_t)(NBMAX / KC) * YT * LDK * ((n_local_max + YT - 1) / YT + 2)));
        TRY(w.linv.grow((size_t)NBMAX * NBMAX));
    }
    bool fresh2 = false, fresh = false;   // new exchange cells: the tags start over
    TRY(c->cells2.grow((2 * (size_t)(PANEL_MAXG + 1) * (IB * (IB + 1) / 2) + IB * IB + 2 * IB) * 2, &fresh2));
    TRY(c->fast_stats.grow(2));
    TRY(c->cells.grow((size_t)IB * (PANEL_MAXG + 2) * IB * 2, &fresh));
    if (fresh2 || fresh) c->ll_epoch = 0;
    bool fresh_ctl = false;
    TRY(c->wctl.grow(1, &fresh_ctl));
    if (fresh_ctl) {
        const WideCtl init = {W_NOFAIL, 0, {0, 0}};
        CU(cudaMemcpy(c->wctl, &init, sizeof(init), cudaMemcpyHostToDevice));
    }
    TRY(c->wbuf.grow((size_t)5 * WP * WP + 3 * XL_ELEMS));
    TRY(c->v1.grow((size_t)2 * rup(m + 4, 2)));
    TRY(c->xbuf.grow(1));
    return 0;
}

static int prof_slot(dhqr_context* c, const char* name) {
    for (size_t i = 0; i < c->prof_slots.size(); ++i)
        if (!strcmp(c->prof_slots[i].name, name)) return (int)i;
    dhqr_context::ProfSlot s;
    s.name = name;
    c->prof_slots.push_back(s);
    return (int)c->prof_slots.size() - 1;
}
// pre(): open a CUDA-event bracket on the launching stream when profiling is on
static void pre(dhqr_context* c, cudaStream_t st) {
    if (!c->profile) return;
    c->prof_open.create(cudaEventDefault);
    cudaEventRecord(c->prof_open, st);
}
static int post(dhqr_context* c, cudaStream_t st, const char* what, double work = 0.0) {
    c->launches++;
    if (c->profile && c->prof_open) {
        dhqr_context::ProfRec r;
        r.slot = prof_slot(c, what);
        r.e0 = std::move(c->prof_open);
        r.e1.create(cudaEventDefault);
        cudaEventRecord(r.e1, st);
        c->prof_slots[r.slot].work += work;
        c->prof_pending.push_back(std::move(r));
    }
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return set_err(1000 + (int)e, "launch of %s failed: %s", what, cudaGetErrorString(e));
    if (c->sync) {
        e = cudaStreamSynchronize(st);
        if (e != cudaSuccess) return set_err(1000 + (int)e, "%s failed: %s", what, cudaGetErrorString(e));
    }
    return 0;
}

// ------------------------------------------------------------------------------------------------
// block-reflector application  C <- (I - V T' V') C  on window rows >= row_lo
//   V: nbp columns of the packed V buffer starting at Vcols (window row 0), T from the Gram matrix.
// ------------------------------------------------------------------------------------------------
// splits over the row chunks: fill whole waves of SMs
static int pick_splits(int tiles, int nchunks, int sms, int64_t cap_tiles) {
    tiles = std::max(tiles, 1);
    int smax = std::max(1, std::min(nchunks / 4, (MAXCTAS_FACTOR * sms) / tiles));
    smax = std::max(smax, std::min(1 + (sms + tiles - 1) / tiles, std::max(1, nchunks / 2)));
    smax = (int)std::min<int64_t>(smax, std::max<int64_t>(1, cap_tiles / tiles));
    int best = 1;
    double beste = 0.0;
    for (int s = 1; s <= smax; ++s) {
        const int ctas = tiles * s;
        const double e = (double)ctas / ((double)sms * ((ctas + sms - 1) / sms));
        if (e > beste + 1e-9) { beste = e; best = s; }
    }
    return best;
}

// block-reflector application  C <- (I - V T' V') C  on window rows >= row_lo
//   V = packed columns [voff, voff + nbp) of `vpk` (columns beyond the live ones are zero); T from the
//   Gram matrix; `w` = the workspace set of the calling chain.
static int apply_block_reflector(dhqr_context* c, cudaStream_t st, const double* vpk, dhqr_context::WSet& w, int voff, int nbp,
                                 int64_t rows, int64_t row_lo, double* C, int64_t ldc, int ncols, bool reuse_T = false,
                                 double* linv_io = nullptr, int gate = 0, int trans = 0) {
    double* linv = linv_io ? linv_io : w.linv;   // where T' is written (or read from, with reuse_T)
    // reuse_T: w.linv already holds T' of this V (same chain, previous call) -> skip the Gram block and k_tinv
    if (ncols <= 0 || rows <= 0) return 0;
    const bool small = (nbp <= 32);
    const int NBPK = small ? 32 : 128;          // kernel instantiation
    const int bn = small ? G1S_BN : G1_BN;
    const int nv = reuse_T ? 0 : NBPK;
    const int next = nv + ncols;
    const int tiles = (next + bn - 1) / bn;
    const int nchunks = (int)((rows + KC1 - 1) / KC1);
    const int nsplit = pick_splits(tiles, nchunks, c->sms, (int64_t)(w.wpart.size() / ((size_t)bn * NBPK)));
    const int64_t pstride = (int64_t)tiles * bn * NBPK;
    if ((size_t)(pstride * nsplit) > w.wpart.size()) return set_err(4001, "internal: W partial workspace too small");
    if ((size_t)next * NBPK > w.wsum.size()) return set_err(4003, "internal: W workspace too small");
    GemmVtaArgs g1;
    g1.vpk = vpk; g1.voff = voff; g1.nv = nv;
    g1.A = C; g1.lda = ldc; g1.rows = rows; g1.na = ncols; g1.nchunks = nchunks;
    g1.a_aligned = (((uintptr_t)C & 15) == 0 && (ldc & 1) == 0) ? 1 : 0;
    g1.Wp = w.wpart; g1.pstride = pstride;
    dim3 grid1(tiles, nsplit);
    pre(c, st);
    if (small) {
        K_G1_32<<<grid1, (1 * 4 + G1S_NPW) * 32, smem_g1(32, G1S_BN), st>>>(g1);
    } else {
        K_G1_128<<<grid1, (4 * 2 + G1_NPW) * 32, smem_g1(128, G1_BN), st>>>(g1);
    }
    TRY(post(c, st, small ? "k_gemm_vta32" : "k_gemm_vta128", 2.0 * (double)rows * nbp * ((double)ncols + nv)));
    const int ygrid = (ncols + YCOLS - 1) / YCOLS;
    if (small && !reuse_T) {
        pre(c, st);
        k_mid32<<<ygrid, 512, 0, st>>>(w.wpart, pstride, nsplit, ncols, w.ypk, linv, trans);
        TRY(post(c, st, "k_mid32"));
    } else {
        pre(c, st);
        const int64_t nelem = (int64_t)next * NBPK;
        k_wreduce<<<(unsigned)std::min<int64_t>((nelem + 255) / 256, 8 * c->sms), 256, 0, st>>>(w.wpart, pstride, nsplit, nelem, w.wsum);
        TRY(post(c, st, "k_wreduce"));
        if (!reuse_T) {
            pre(c, st);
            if (small) k_tinv<32><<<1, 512, smem_tinv(32), st>>>(w.wsum, linv);
            else k_tinv<128><<<1, 512, smem_tinv(128), st>>>(w.wsum, linv);
            TRY(post(c, st, small ? "k_tinv32" : "k_tinv128"));
        }
        pre(c, st);
        if (small) k_ymake<32><<<ygrid, 256, smem_ymake(32), st>>>(w.wsum, nv, ncols, linv, w.ypk, trans);
        else k_ymake<128><<<ygrid, 256, smem_ymake(128), st>>>(w.wsum, nv, ncols, linv, w.ypk, trans);
        TRY(post(c, st, small ? "k_ymake32" : "k_ymake128"));
    }
    pre(c, st);
    GemmCvyArgs g2;
    g2.C = C; g2.ldc = ldc; g2.rows = rows; g2.row_lo = row_lo; g2.ncols = ncols;
    g2.vpk = vpk; g2.voff = voff; g2.ypk = w.ypk;
    g2.nkq = small ? 1 : (int)(rup(nbp, KC) / KC); g2.nkq_alloc = NBPK / KC;
    g2.ctl = c->wctl; g2.gate = gate;
    dim3 grid2((unsigned)((rows + G2_BM - 1) / G2_BM), (unsigned)((ncols + G2_BN - 1) / G2_BN));
    g2.tiles_m = (int)grid2.x; g2.tiles_n = (int)grid2.y;
    g2.tiles_per_cta = CVY_TILES_PER_CTA;
    if (g2.nkq == 4) k_gemm_cvy_p<<<(g2.tiles_m * g2.tiles_n + CVY_TILES_PER_CTA - 1) / CVY_TILES_PER_CTA, 9 * 32, smem_g2(), st>>>(g2);
    else k_gemm_cvy<<<grid2, 9 * 32, smem_g2(), st>>>(g2);
    TRY(post(c, st, small ? "k_gemm_cvy32" : "k_gemm_cvy128", 2.0 * (double)rows * (small ? 32 : nbp) * (double)ncols));
    return 0;
}

// ------------------------------------------------------------------------------------------------
// cooperative panel launch: factor mp x ncols (<= IB) at P, V block -> vout columns
// ------------------------------------------------------------------------------------------------
static int launch_panel(dhqr_context* c, cudaStream_t st, double* vpk, double* P, int64_t ldp, int64_t mp, int ncols,
                        double* alpha, int voff, int64_t vtop, int64_t vrows, int gate = 0) {
    // under look-ahead the panel kernel leaves most SMs to the bulk update running beside it
    int gmax = c->lookahead ? 64 : c->sms;
    gmax = std::min(std::min(gmax, c->sms), PANEL_MAXG);
    int64_t rpc = std::max<int64_t>((mp + gmax - 1) / gmax, 64);
    rpc = rup(rpc, 8);
    while ((size_t)IB * ((size_t)rpc + 4) * 8 > 184 * 1024 && gmax < std::min(c->sms, PANEL_MAXG)) {   // slab too big: use more CTAs
        gmax = std::min(gmax * 2, std::min(c->sms, PANEL_MAXG));
        rpc = rup(std::max<int64_t>((mp + gmax - 1) / gmax, 64), 8);
    }
    const int G = (int)((mp + rpc - 1) / rpc);
    const int lds = (int)rpc + 4;   // rpc is a multiple of 8 -> lds == 4 mod 8
    const size_t smem = (size_t)IB * lds * 8;
    if (smem > 184 * 1024) return set_err(-2, "m too large for the resident panel kernel (%lld rows per CTA)", (long long)rpc);
    if (c->ll_epoch > 0xF0000000u) {   // tag space nearly used up: start over with clean cells
        CU(cudaMemsetAsync(c->cells, 0, sizeof(unsigned long long) * c->cells.size(), st));
        CU(cudaMemsetAsync(c->cells2, 0, sizeof(unsigned long long) * c->cells2.size(), st));
        c->ll_epoch = 0;
    }
    PanelArgs a;
    a.P = P; a.ldp = ldp; a.mp = mp; a.ncols = ncols; a.alpha = alpha;
    a.vpk = vpk; a.voff = voff; a.vtop = vtop; a.vrows = vrows;
    a.rows_per_cta = (int)rpc; a.lds = lds;
    a.cells = c->cells; a.epoch = c->ll_epoch;
    a.cells2 = c->cells2; a.fast = c->panel_fast; a.fast_stats = c->fast_stats;
    a.ctl = c->wctl; a.gate = gate;
    void* args[] = {&a};
    pre(c, st);
    cudaError_t e = cudaLaunchCooperativeKernel((void*)k_panel, dim3(G), dim3(PANEL_THREADS), args, smem, st);
    if (e != cudaSuccess) return set_err(1000 + (int)e, "cooperative launch of k_panel failed: %s", cudaGetErrorString(e));
    c->ll_epoch += IB + 8;
    return post(c, st, "k_panel", 16.0 * (double)mp * ncols);   // work = bytes: panel read once + written once
}

// ------------------------------------------------------------------------------------------------
// partition bookkeeping: global list of panels (owner, first global column, width)
// ------------------------------------------------------------------------------------------------
struct Panel { int owner; int64_t c; int kb; };

static int gather_partition(dhqr_context* c, cudaStream_t st, int64_t col0, int64_t n_local, std::vector<int64_t>& col0s,
                            std::vector<int64_t>& nls) {
    col0s.assign(c->nranks, 0);
    nls.assign(c->nranks, 0);
    if (c->nranks == 1) { col0s[0] = col0; nls[0] = n_local; return 0; }
    int64_t mine[2] = {col0, n_local};
    CU(cudaMemcpyAsync(c->d_i64, mine, sizeof(mine), cudaMemcpyHostToDevice, st));
    NC(g_nccl.AllGather(c->d_i64, c->d_i64 + 2, 2, ncclInt64, c->comm, st));
    std::vector<int64_t> all(2 * c->nranks);
    CU(cudaMemcpyAsync(all.data(), c->d_i64 + 2, sizeof(int64_t) * 2 * c->nranks, cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    for (int r = 0; r < c->nranks; ++r) { col0s[r] = all[2 * r]; nls[r] = all[2 * r + 1]; }
    return 0;
}

static int check_partition(const std::vector<int64_t>& col0s, const std::vector<int64_t>& nls, int64_t n_global) {
    // DArray (1,P) grid: contiguous, ascending with rank (S:19, test/runtests.jl:71)
    int64_t next = 0;
    for (size_t r = 0; r < col0s.size(); ++r) {
        if (col0s[r] != next || nls[r] < 0) return set_err(-4, "column blocks must be contiguous and ascending with rank (rank %zu: col0=%lld, expected %lld)", r, (long long)col0s[r], (long long)next);
        next += nls[r];
    }
    if (next != n_global) return set_err(-3, "column blocks cover %lld columns, n_global=%lld", (long long)next, (long long)n_global);
    return 0;
}

static void build_panels(const std::vector<int64_t>& col0s, const std::vector<int64_t>& nls, int nb, std::vector<Panel>& out) {
    out.clear();
    for (size_t r = 0; r < col0s.size(); ++r)
        for (int64_t o = 0; o < nls[r]; o += nb) out.push_back({(int)r, col0s[r] + o, (int)std::min<int64_t>(nb, nls[r] - o)});
}

static int check_common(dhqr_context* c, int64_t m, int64_t n_global, int64_t col0, int64_t n_local, const void* A, int64_t lda) {
    if (!c) return set_err(-1, "null handle");
    if (m < 0) return set_err(-2, "m < 0");
    if (n_global < 0 || n_global > m) return set_err(-3, "need 0 <= n_global <= m (reference asserts full column rank shapes)");
    if (col0 < 0 || col0 > n_global) return set_err(-4, "col0 out of range");
    if (n_local < 0 || col0 + n_local > n_global) return set_err(-5, "n_local out of range");
    if (n_local > 0 && !A) return set_err(-6, "null matrix pointer");
    if (lda < std::max<int64_t>(1, m)) return set_err(-7, "lda < max(1,m)");
    return 0;
}

// right-hand sides b (m x nrhs): a bad argument is refused with minus its position in the entry point's argument list
static int check_rhs(int64_t m, int nrhs, const void* b, int64_t ldb, int idx_b, int idx_ldb, int idx_nrhs) {
    if (nrhs < 0) return set_err(-idx_nrhs, "nrhs < 0");
    if (nrhs > 0 && !b) return set_err(-idx_b, "null b");
    if (ldb < std::max<int64_t>(1, m)) return set_err(-idx_ldb, "ldb < max(1,m)");
    return 0;
}

// ------------------------------------------------------------------------------------------------
// qr!: blocked driver  (S:113-148, S:198-213)
// ------------------------------------------------------------------------------------------------
struct PanelGeom { int64_t r0, rows, vrows; int nbp; };
static PanelGeom panel_geom(const Panel& p, int64_t m) {
    PanelGeom g;
    g.r0 = p.c & ~(int64_t)31;              // window start: 32-row aligned for the TMA chunks
    g.rows = m - g.r0;                       // valid window rows
    g.vrows = rup(g.rows, 128);
    g.nbp = (int)rup(p.kb, IB);
    return g;
}

// Packs the kb columns of the panel at src (mp rows; tril: zeros above the diagonal, where a factored panel keeps R) into vpk
// with panel row 0 at window row vtop.  packed_cols (32 or 128) columns are written, those beyond kb as zeros: they must
// cover the nbp the block update then reads.
static int pack_panel(dhqr_context* c, cudaStream_t st, const double* src, int64_t lda, int64_t mp, int kb, int tril, double* vpk,
                      int64_t vtop, int64_t vrows, int packed_cols) {
    dim3 grid((unsigned)std::min<int64_t>((vrows / 4 + 255) / 256, 4 * c->sms), packed_cols);
    pre(c, st);
    k_pack<<<grid, 256, 0, st>>>(src, lda, mp, kb, tril, vpk, 0, vtop, vrows);
    return post(c, st, "k_pack");
}

// factor one outer panel on stream st: inner panels of IB columns + updates inside the outer panel; V -> vpk
// (the 32-column chain: one cooperative launch per inner panel, S:127-135 column by column in the worst case)
static int factor_outer_panel_narrow(dhqr_context* c, cudaStream_t st, double* vpk, dhqr_context::WSet& w, const Panel& p, int64_t m,
                                     int64_t col0, double* A, int64_t lda, double* alpha, int step) {
    const PanelGeom g = panel_geom(p, m);
    for (int o = 0; o < p.kb; o += IB) {
        const int ib = std::min(IB, p.kb - o);
        const int64_t cs = p.c + o;                                   // global column == pivot row
        double* P = A + (cs - col0) * lda + cs;
        TRY(launch_panel(c, st, vpk, P, lda, m - cs, ib, alpha + cs, o, cs - g.r0, g.vrows, step));
        const int rem = p.kb - (o + ib);
        if (rem > 0)   // update the rest of the outer panel with this sub-panel's reflectors
            TRY(apply_block_reflector(c, st, vpk, w, o, IB, g.rows, cs - g.r0, A + (cs + ib - col0) * lda + g.r0, lda, rem, false,
                                      nullptr, step));
    }
    if (g.nbp > IB && g.nbp < NBMAX) {   // zero the V columns the 128-wide kernels read beyond nbp
        k_vpk_zero_cols<<<2 * c->sms, 256, 0, st>>>(vpk, g.vrows / KC1, g.nbp, NBMAX);
        TRY(post(c, st, "k_vpk_zero_cols"));
    }
    return 0;
}

// Partial Gram matrices of the packed panel in `vpk` (window rows `rows`) -> w.wpart; returns the number of partials and their stride.
static int launch_panel_gram(dhqr_context* c, cudaStream_t st, const double* vpk, dhqr_context::WSet& w, int64_t rows, int* nsplit_out,
                             int64_t* pstride_out) {
    const int nchunks = (int)((rows + KC1 - 1) / KC1);
    const int64_t pstride = (int64_t)WP * WP;
    pre(c, st);
    const int cps = std::max(1, (nchunks + c->sms - 1) / c->sms);                           // chunks per CTA: whole waves of equal CTAs
    const int nsplit = (nchunks + cps - 1) / cps;
    if ((size_t)nsplit * pstride > w.wpart.size()) return set_err(4001, "internal: W partial workspace too small");
    GramSymArgs g;
    g.vpk = vpk; g.nchunks = nchunks; g.Wp = w.wpart; g.pstride = pstride;
    k_gram_sym<<<nsplit, (GS_MMA_WARPS + 1) * 32, SMEM_GRAM_SYM, st>>>(g);
    *nsplit_out = nsplit;
    *pstride_out = pstride;
    return post(c, st, "k_gram128", 2.0 * (double)rows * WP * WP);
}

// the 128-column chain (dhqr_wide.cuh): CholeskyQR2 + Householder reconstruction of a full aligned outer panel
static bool wide_eligible(const dhqr_context* c, const Panel& p, int64_t m, int nb) {
    return c->wide_panel && nb == WP && p.kb == WP && (p.c & 31) == 0 && m - p.c >= WP;
}
static int factor_outer_panel_wide(dhqr_context* c, cudaStream_t st, double* vpk, dhqr_context::WSet& w, const Panel& p, int64_t m,
                                   int64_t col0, double* A, int64_t lda, double* alpha, int step, double* linv_out) {
    const PanelGeom g = panel_geom(p, m);       // r0 == p.c: the window starts at the pivot row
    double* P = A + (p.c - col0) * lda + p.c;
    double* R1 = c->wbuf, *R2 = R1 + WP * WP, *Rt = R2 + WP * WP, *Rr = Rt + WP * WP, *MT = Rr + WP * WP;
    double* Z1 = MT + WP * WP, *Z2 = Z1 + XL_ELEMS, *Z23 = Z2 + XL_ELEMS;
    double* vflag = vpk + KC1;                  // padding row 64 of packed column 0: travels with the V buffer
    const int nq = (int)(g.vrows / KC1);
    RmulArgs r;
    r.vpk = vpk; r.ctl = c->wctl; r.step = step; r.P = nullptr; r.ldp = lda; r.mp = g.rows;
    auto rmul = [&](int q0, int n, const double* Z, double* Pout) -> int {
        if (n <= 0) return 0;
        r.q0 = q0; r.nq = n; r.ZL = Z; r.P = Pout;
        pre(c, st);
        k_vpk_rmul<<<std::min(n, c->sms), 256, SMEM_RMUL, st>>>(r);
        return post(c, st, "k_vpk_rmul", 2.0 * 64.0 * n * WP * 80.0);
    };
    // Gram matrix of the packed panel: partials of vpk' vpk over the window rows
    int nsplit = 0;
    int64_t pstride = 0;
    auto gram = [&]() -> int { return launch_panel_gram(c, st, vpk, w, g.rows, &nsplit, &pstride); };
    TRY(pack_panel(c, st, P, lda, g.rows, WP, 0, vpk, 0, g.vrows, WP));
    TRY(gram());
    pre(c, st);
    k_wreduce4<<<(WP * WP * 4) / 256, 256, 0, st>>>(w.wpart, pstride, nsplit, (int64_t)WP * WP, w.wsum);
    TRY(post(c, st, "k_wreduce"));
    pre(c, st);
    k_chol128<<<1, 512, SMEM_WIDE1, st>>>(w.wsum, R1, Z1, c->wctl, step, vflag, c->wide_kappa);
    TRY(post(c, st, "k_chol128"));
    TRY(rmul(0, nq, Z1, nullptr));
    TRY(gram());
    pre(c, st);
    k_gram2_finish<<<256, 256, 0, st>>>(w.wpart, pstride, nsplit, w.wsum, R2, Z2, c->wctl, step, vflag);
    TRY(post(c, st, "k_gram2_finish"));
    // Two small kernels sit beside the chain, not in it (their own high-priority stream, unless the per-launch profile or the
    // debug sync asks for plain stream order): Rt = R2 R1 overlaps the solve of the top chunks, k_trecon the last pass
    cudaStream_t sx = (!c->profile && !c->sync) ? c->aux_stream : st;
    if (sx != st) { CU(cudaEventRecord(c->ev_aux[0], st)); CU(cudaStreamWaitEvent(sx, c->ev_aux[0], 0)); }
    pre(c, sx);
    k_trimm128<<<10, 256, SMEM_TRIMM, sx>>>(R2, R1, Rt, c->wctl, step);
    TRY(post(c, sx, "k_trimm128"));
    if (sx != st) CU(cudaEventRecord(c->ev_aux[1], sx));
    TRY(rmul(0, 2, Z2, nullptr));
    if (sx != st) CU(cudaStreamWaitEvent(st, c->ev_aux[1], 0));
    pre(c, st);
    k_hr128<<<1, 512, SMEM_WIDE1, st>>>(vpk, Rt, P, lda, alpha + p.c, Rr, MT, c->wctl, step);
    TRY(post(c, st, "k_hr128"));
    if (linv_out) {     // T' of the panel from the reconstruction: the owner's next block update needs neither V'V nor k_tinv
        if (sx != st) { CU(cudaEventRecord(c->ev_aux[2], st)); CU(cudaStreamWaitEvent(sx, c->ev_aux[2], 0)); }
        pre(c, sx);
        k_trecon<<<4, 256, SMEM_TRECON, sx>>>(vpk, MT, linv_out, c->wctl, step);
        TRY(post(c, sx, "k_trecon"));
        if (sx != st) CU(cudaEventRecord(c->ev_aux[3], sx));
    }
    pre(c, st);
    k_trimm_z<<<10, 256, SMEM_TRIMM, st>>>(Rr, R2, Z23, c->wctl, step);
    TRY(post(c, st, "k_trimm_z"));
    TRY(rmul(2, nq - 2, Z23, P));
    if (linv_out && sx != st) CU(cudaStreamWaitEvent(st, c->ev_aux[3], 0));   // T' is part of the panel's result
    c->wide_panels++;
    return 0;
}

static int factor_outer_panel(dhqr_context* c, cudaStream_t st, double* vpk, dhqr_context::WSet& w, const Panel& p, int64_t m,
                              int64_t col0, double* A, int64_t lda, double* alpha, int step, bool wide, double* linv_out = nullptr) {
    if (c->wctl) {   // clear the guards of the previous panel and the verdict that travels with this V buffer
        k_wide_begin<<<1, 32, 0, st>>>(c->wctl, vpk + KC1);
        TRY(post(c, st, "k_wide_begin"));
    }
    if (wide) return factor_outer_panel_wide(c, st, vpk, w, p, m, col0, A, lda, alpha, step, linv_out);
    return factor_outer_panel_narrow(c, st, vpk, w, p, m, col0, A, lda, alpha, step);
}

static int mirror_panel_to_host(dhqr_context* c, cudaStream_t st, const Panel& p, int64_t m, int64_t col0, const double* A,
                                int64_t lda) {
    if (!c->mirror_host) return 0;   // host entry point only: this panel's columns are final -> start their D2H now
    Event& ev = c->panel_events.emplace_back();
    CU(ev.create(cudaEventDisableTiming));
    CU(cudaEventRecord(ev, st));
    CU(cudaStreamWaitEvent(c->d2h_stream, ev, 0));
    CU(cudaMemcpy2DAsync(c->mirror_host + p.c * c->mirror_lda, (size_t)c->mirror_lda * 8, A + (p.c - col0) * lda, (size_t)lda * 8,
                         (size_t)m * 8, (size_t)p.kb, cudaMemcpyDeviceToHost, c->d2h_stream));
    return 0;
}

// Which panels go through the 128-column chain: those at or beyond `wide_from` that are full and aligned.
struct Plan { int kstart; int wide_from; int nb; };
static bool plan_wide(const dhqr_context* c, const Plan& pl, const std::vector<Panel>& panels, int k, int64_t m) {
    return k >= pl.wide_from && wide_eligible(c, panels[k], m, pl.nb);
}

// single stream, one panel after the other (options lookahead = 0, sync, profile; any number of ranks)
static int qr_blocked_serial(dhqr_context* c, cudaStream_t st, int64_t m, int64_t col0, int64_t nl, double* A, int64_t lda,
                             double* alpha, const std::vector<Panel>& panels, const Plan& pl) {
    const int64_t lend = col0 + nl;
    double* vpk = c->vpk2[0];
    auto& w = c->ws[0];
    for (int k = pl.kstart; k < (int)panels.size(); ++k) {
        const Panel& p = panels[k];
        const PanelGeom g = panel_geom(p, m);
        bool haveT = false;
        if (c->rank == p.owner) {
            const bool wide = plan_wide(c, pl, panels, k, m);
            TRY(factor_outer_panel(c, st, vpk, w, p, m, col0, A, lda, alpha, k, wide, w.linv));
            TRY(mirror_panel_to_host(c, st, p, m, col0, A, lda));
            haveT = wide;
        }
        if (c->nranks > 1) {
            // C2 (S:141-143): the owner's reflectors go to every rank, once per panel instead of once per column
            NC(g_nccl.Broadcast(vpk, vpk, (size_t)(g.vrows / KC1) * VPK_CHUNK, ncclFloat64, p.owner, c->comm, st));
            NC(g_nccl.Broadcast(alpha + p.c, alpha + p.c, (size_t)p.kb, ncclFloat64, p.owner, c->comm, st));
            k_wide_note<<<1, 32, 0, st>>>(c->wctl, vpk + KC1, k);
            TRY(post(c, st, "k_wide_note"));
        }
        // trailing update of the local columns right of the panel (S:198-213 for nb columns at once)
        const int64_t t0 = std::max(p.c + p.kb, col0);
        if (t0 < lend)
            TRY(apply_block_reflector(c, st, vpk, w, 0, g.nbp, g.rows, p.c - g.r0, A + (t0 - col0) * lda + g.r0, lda, (int)(lend - t0),
                                      haveT, nullptr, k + 1));
    }
    return 0;
}

// look-ahead: the panel chain (latency bound) runs on a high-priority stream ahead of the bulk trailing update, which stays on
// the caller's stream.  SPMD over ranks: the owner of a panel factors it, the packed V block is broadcast on the high-priority
// stream (the only stream that issues collectives), every rank updates its own columns.
//   hp step k: wait next[k-1];  owner(k+1): apply V_k -> columns of panel k+1, factor panel k+1 (V -> vpk[(k+1)%3]);
//              broadcast vpk[(k+1)%3] + alpha slice;  signal panel[k+1]                                    set 1
//   st step k: wait panel[k];   (a) apply V_k -> local columns of panel k+2, signal next[k];
//                               (b) apply V_k -> local columns right of panel k+2 (T reused)                set 0
// Every column block receives every V exactly once and in order; the panel chain only depends on the small
// (a) parts, i.e. it has two bulk updates of slack.  Three V buffers: V_{k+2} replaces V_{k-1}, whose last
// reader (b)_{k-1} precedes (a)_k on st (hence the wait on next[k-1] on every rank before the broadcast).
static int qr_blocked_lookahead(dhqr_context* c, cudaStream_t st, int64_t m, int64_t col0, int64_t nl, double* A, int64_t lda,
                                double* alpha, const std::vector<Panel>& panels, const Plan& pl) {
    const int64_t lend = col0 + nl;
    const int K = (int)panels.size(), K0 = pl.kstart;
    cudaStream_t hp = c->hp_stream;
    // the events of this call: destroyed on return, when the work they order is enqueued
    std::vector<Event> evPanel(K), evNext(K), evBulk(K), evA2(K), evHp(K), evCatch;
    std::vector<char> haveA2(K, 0);
    // stage timeline of the pipelined host entry (option host_trace; dhqr_qr_host_f64 is the only caller that mirrors to the host)
    const bool trace = c->host_trace && c->mirror_host;
    const unsigned evflags = trace ? cudaEventDefault : cudaEventDisableTiming;
    for (int k = K0; k < K; ++k) {
        CU(evA2[k].create(cudaEventDisableTiming));
        CU(evPanel[k].create(evflags));
        CU(evNext[k].create(evflags));
        CU(evBulk[k].create(evflags));
    }
    // local intersection of the global column range [a, b) -> pointer + count
    auto clip = [&](int64_t a, int64_t b, int64_t& lo, int64_t& hi) { lo = std::max(a, col0); hi = std::min(b, lend); return hi > lo; };
    // publish panel k (already factored on its owner into vpk[k%3]) to every rank.  The collectives run on their own stream:
    // the owner's chain goes on with panel k+1 (it has V_k already) while V_k travels; the other ranks pick it up through
    // evPanel[k].  The comm stream first waits for everything queued on hp so far: on the owner that is the factorisation of
    // panel k, on every rank the last reads of the ring slot's previous occupant V_{k-3}.
    cudaStream_t cs = c->comm_stream;
    auto publish = [&](int k) -> int {
        if (c->nranks > 1) {
            const PanelGeom g = panel_geom(panels[k], m);
            double* v = c->vpk2[k % 3];
            CU(evHp[k].create(cudaEventDisableTiming));
            CU(cudaEventRecord(evHp[k], hp));
            CU(cudaStreamWaitEvent(cs, evHp[k], 0));
            NC(g_nccl.Broadcast(v, v, (size_t)(g.vrows / KC1) * VPK_CHUNK, ncclFloat64, panels[k].owner, c->comm, cs));
            NC(g_nccl.Broadcast(alpha + panels[k].c, alpha + panels[k].c, (size_t)panels[k].kb, ncclFloat64, panels[k].owner, c->comm, cs));
            k_wide_note<<<1, 32, 0, cs>>>(c->wctl, v + KC1, k);   // the owner's verdict on the panel arrived with the buffer
            TRY(post(c, cs, "k_wide_note"));
            CU(cudaEventRecord(evPanel[k], cs));
        } else {
            CU(cudaEventRecord(evPanel[k], hp));
        }
        return 0;
    };
    // V_k is usable on stream s: the owner has it once its own chain got there (hp order / evHp), the others once it arrived
    auto wait_panel = [&](cudaStream_t s, int k) {
        if (c->nranks > 1 && c->rank == panels[k].owner) {
            if (s != hp) cudaStreamWaitEvent(s, evHp[k], 0);
        } else {
            cudaStreamWaitEvent(s, evPanel[k], 0);
        }
    };
    // Host entry (dhqr_qr_host_f64, one rank, first pass): columns [wend, lend) are still on their way to the device in chunks
    // (c->up_chunks).  The schedule runs on the window [col0, wend); a chunk joins at the step its plan names - at the latest
    // while it still lies right of panel k+2 - after a CATCH-UP on its own stream: the reflectors of panels < k, re-packed from
    // the factored columns, applied to the chunk with the T' kept in the per-panel slots.  Same reflectors in the same order on
    // every column, only the time at which a column receives them changes.
    const bool windowed = !c->up_chunks.empty() && c->nranks == 1 && K0 == 0;
    int64_t wend = windowed ? std::min(lend, c->up_chunks.front().c0) : lend;
    size_t upnext = 0;
    std::vector<char> haveTslot(K, 0);
    auto catch_up = [&](const dhqr_context::UpChunk& u, int lane, int k, cudaEvent_t done) -> int {
        cudaStream_t cu = c->cu_stream[lane];
        double* vpk_cu = c->vpk2[3 + lane];
        auto& ws_cu = c->ws[3 + lane];
        cudaStreamWaitEvent(cu, u.ev, 0);
        for (int q = K0; q < k; ++q) {
            const Panel& pq = panels[q];
            const PanelGeom gq = panel_geom(pq, m);
            cudaStreamWaitEvent(cu, evPanel[q], 0);                   // V_q is final in A ...
            cudaStreamWaitEvent(cu, evNext[q], 0);                    // ... and T'_q sits in its slot
            TRY(pack_panel(c, cu, A + (pq.c - col0) * lda + pq.c, lda, m - pq.c, pq.kb, 1, vpk_cu, pq.c - gq.r0, gq.vrows,
                           gq.nbp <= IB ? IB : NBMAX));
            TRY(apply_block_reflector(c, cu, vpk_cu, ws_cu, 0, gq.nbp, gq.rows, pq.c - gq.r0, A + (u.c0 - col0) * lda + gq.r0, lda,
                                      (int)(u.c1 - u.c0), haveTslot[q] != 0, c->tslot(q), q + 1));
        }
        cudaEventRecord(done, cu);
        return 0;
    };
    std::vector<int> joinedAt;
    const int rc = [&]() -> int {
        Event fork;
        CU(fork.create(evflags));
        cudaEventRecord(fork, st);
        cudaStreamWaitEvent(hp, fork, 0);                          // hp starts after everything already queued on st
        std::vector<char> ownT(K, 0);       // T'_k already sits in the ring slot on this rank (wide panel factored here, k_trecon)
        if (c->rank == panels[K0].owner) {
            const bool wide = plan_wide(c, pl, panels, K0, m);
            TRY(factor_outer_panel(c, hp, c->vpk2[K0 % 3], c->ws[1], panels[K0], m, col0, A, lda, alpha, K0, wide, c->tslot(K0)));
            TRY(mirror_panel_to_host(c, hp, panels[K0], m, col0, A, lda));
            if (wide) { ownT[K0] = 1; cudaEventRecord(evNext[K0], hp); }
        }
        TRY(publish(K0));
        for (int k = K0; k < K; ++k) {
            const Panel& p = panels[k];
            const PanelGeom g = panel_geom(p, m);
            const double* vk = c->vpk2[k % 3];
            const int64_t t0 = p.c + p.kb;                                               // first trailing column
            const int64_t t1 = k + 1 < K ? panels[k + 1].c + panels[k + 1].kb : t0;      // end of panel k+1
            const int64_t t2 = k + 2 < K ? panels[k + 2].c + panels[k + 2].kb : t1;      // end of panel k+2
            int64_t lo, hi;
            // chunks that join the window at this step: planned, or forced because step k+1 would reach into them
            const int64_t wold = wend;
            const size_t up0 = upnext;
            if (windowed) {
                const int64_t t3 = k + 3 < K ? panels[k + 3].c + panels[k + 3].kb : lend;   // end of panel k+3
                while (upnext < c->up_chunks.size() && (c->up_chunks[upnext].join <= k || c->up_chunks[upnext].c0 < t3)) {
                    const auto& u = c->up_chunks[upnext];
                    if (u.c0 < t2 || u.c0 != wend) return set_err(4005, "internal: upload chunk %d joins too late (step %d)", (int)upnext, k);
                    Event& done = evCatch.emplace_back();
                    CU(done.create(evflags));
                    joinedAt.push_back(k);
                    TRY(catch_up(u, (int)(upnext % CU_STREAMS), k, done));
                    wend = u.c1;
                    ++upnext;
                }
                if (wend < t2) return set_err(4005, "internal: window ends at %lld before panel %d", (long long)wend, k + 2);
            }
            double* lk = c->tslot(k);
            bool haveT = ownT[k];                                        // T'_k in lk (this rank)
            if (k + 1 < K) {
                // vpk[(k+1)%3] was last read by the bulk update k-2 (and, on the owner of panel k-2, by its broadcast)
                if (k - 2 >= K0) {
                    cudaStreamWaitEvent(hp, evBulk[k - 2], 0);
                    if (haveA2[k - 2]) cudaStreamWaitEvent(hp, evA2[k - 2], 0);
                    if (c->nranks > 1) cudaStreamWaitEvent(hp, evPanel[k - 2], 0);
                }
                if (c->rank == panels[k + 1].owner) {
                    wait_panel(hp, k);
                    if (k - 1 >= K0 && haveA2[k - 1]) cudaStreamWaitEvent(hp, evA2[k - 1], 0);   // V_{k-1} reached these columns
                    if (clip(t0, t1, lo, hi)) {
                        const bool hadT = haveT;
                        TRY(apply_block_reflector(c, hp, vk, c->ws[1], 0, g.nbp, g.rows, p.c - g.r0, A + (lo - col0) * lda + g.r0, lda,
                                                  (int)(hi - lo), haveT, lk, k + 1));
                        haveT = true;
                        if (!hadT) cudaEventRecord(evNext[k], hp);       // T'_k is in the ring: the bulk update may start
                    }
                    const bool widen = plan_wide(c, pl, panels, k + 1, m);
                    TRY(factor_outer_panel(c, hp, c->vpk2[(k + 1) % 3], c->ws[1], panels[k + 1], m, col0, A, lda, alpha, k + 1, widen,
                                           c->tslot(k + 1)));
                    if (widen) { ownT[k + 1] = 1; cudaEventRecord(evNext[k + 1], hp); }
                    TRY(mirror_panel_to_host(c, hp, panels[k + 1], m, col0, A, lda));
                }
                TRY(publish(k + 1));
            }
            // columns of panel k+2: their V_0..V_{k-1} come from the bulk updates up to k-1.  This apply is off the chain's
            // stream (it overlaps the factorisation of panel k+1); the chain picks it up through evA2[k] before it applies
            // V_{k+1} to the same columns.
            if (clip(t1, t2, lo, hi)) {
                cudaStream_t s2 = c->hp2_stream;
                cudaEventRecord(evA2[k], hp);                            // (used as a scratch event first: order s2 behind hp so far,
                cudaStreamWaitEvent(s2, evA2[k], 0);                     //  i.e. behind T'_k and behind the last reader of workspace set 2)
                if (k - 1 >= K0) cudaStreamWaitEvent(s2, evBulk[k - 1], 0);
                wait_panel(s2, k);
                const bool hadT = haveT;
                TRY(apply_block_reflector(c, s2, vk, c->ws[2], 0, g.nbp, g.rows, p.c - g.r0, A + (lo - col0) * lda + g.r0, lda,
                                          (int)(hi - lo), haveT, lk, k + 1));
                haveT = true;
                if (!hadT) cudaEventRecord(evNext[k], s2);               // T'_k came from this apply
                cudaEventRecord(evA2[k], s2);
                haveA2[k] = true;
            }
            if (!haveT) cudaEventRecord(evNext[k], hp);                  // keep the event defined (timeline tracing)
            wait_panel(st, k);
            if (clip(t2, std::min(lend, wold), lo, hi)) {
                if (haveT) cudaStreamWaitEvent(st, evNext[k], 0);
                TRY(apply_block_reflector(c, st, vk, c->ws[0], 0, g.nbp, g.rows, p.c - g.r0, A + (lo - col0) * lda + g.r0, lda,
                                          (int)(hi - lo), haveT, haveT ? lk : nullptr, k + 1));
            }
            for (size_t j = up0; j < upnext; ++j) {                      // the chunks that joined at this step, each behind its catch-up
                const auto& u = c->up_chunks[j];
                cudaStreamWaitEvent(st, evCatch[j], 0);
                if (haveT) cudaStreamWaitEvent(st, evNext[k], 0);
                TRY(apply_block_reflector(c, st, vk, c->ws[0], 0, g.nbp, g.rows, p.c - g.r0, A + (u.c0 - col0) * lda + g.r0, lda,
                                          (int)(u.c1 - u.c0), haveT, haveT ? lk : nullptr, k + 1));
            }
            haveTslot[k] = haveT;
            cudaEventRecord(evBulk[k], st);
        }
        cudaStreamWaitEvent(st, evPanel[K - 1], 0);                // join: alpha and the last panel come from hp / the comm stream
        if (c->nranks > 1) {
            cudaEventRecord(evHp[K - 1], hp);                      // (re-recorded: everything queued on hp)
            cudaStreamWaitEvent(st, evHp[K - 1], 0);
        }
        if (trace) {   // ms since the first chunk was on the device
            cudaStreamSynchronize(st);
            cudaStreamSynchronize(hp);
            for (size_t j = 0; j < evCatch.size(); ++j) {
                float tu = -1.f, tc = -1.f;
                cudaEventSynchronize(evCatch[j]);
                cudaEventElapsedTime(&tu, fork, c->up_chunks[j].ev);
                cudaEventElapsedTime(&tc, fork, evCatch[j]);
                fprintf(stderr, "[dhqr host] chunk at column %5lld: uploaded %7.2f ms, joins at step %2d (planned %2d), caught up %7.2f ms\n",
                        (long long)c->up_chunks[j].c0, tu, joinedAt[j], c->up_chunks[j].join, tc);
            }
            for (int k = K0; k < K; ++k) {
                float tp = 0.f, tt = 0.f, tb = 0.f;
                cudaEventElapsedTime(&tp, fork, evPanel[k]);
                cudaEventElapsedTime(&tt, fork, evNext[k]);
                cudaEventElapsedTime(&tb, fork, evBulk[k]);
                fprintf(stderr, "[dhqr host] step %2d: panel %7.2f  T' %7.2f  bulk %7.2f ms\n", k, tp, tt, tb);
            }
        }
        return 0;
    }();
    // error path: the caller's stream must not run ahead of (or return before) work already queued on the internal stream
    Event hpdone;
    if (rc && hpdone.create(cudaEventDisableTiming) == cudaSuccess) {
        cudaEventRecord(hpdone, hp);
        cudaStreamWaitEvent(st, hpdone, 0);
        cudaEventRecord(hpdone, cs);
        cudaStreamWaitEvent(st, hpdone, 0);
        cudaEventRecord(hpdone, c->hp2_stream);
        cudaStreamWaitEvent(st, hpdone, 0);
        for (int i = 0; i < CU_STREAMS; ++i) {
            cudaEventRecord(hpdone, c->cu_stream[i]);
            cudaStreamWaitEvent(st, hpdone, 0);
        }
    }
    if (rc) return rc;
    const cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return set_err(1000 + (int)e, "look-ahead enqueue failed: %s", cudaGetErrorString(e));
    return 0;
}

// largest row count the resident 32-column panel kernel can take on this device (slab of rows in shared memory)
static int64_t narrow_panel_max_rows(const dhqr_context* c) {
    const int gmax = std::min(c->sms, PANEL_MAXG);
    const int64_t rpc = ((184 * 1024) / (IB * 8) - 4) & ~(int64_t)7;
    return rpc * gmax;
}

static int qr_blocked(dhqr_context* c, cudaStream_t st, int64_t m, int64_t n, int64_t col0, int64_t nl, double* A,
                      int64_t lda, double* alpha, int nb) {
    std::vector<int64_t> col0s, nls;
    TRY(gather_partition(c, st, col0, nl, col0s, nls));
    TRY(check_partition(col0s, nls, n));
    int64_t nlmax = 0;
    for (auto v : nls) nlmax = std::max(nlmax, v);
    std::vector<Panel> panels;
    build_panels(col0s, nls, nb, panels);
    TRY(ensure_workspace(c, m, nlmax, (int64_t)panels.size(), !c->up_chunks.empty()));
    if (panels.empty()) return 0;
    // rank-uniform precondition, checked on every rank BEFORE the first collective: a panel that neither chain can take
    // would otherwise fail on its owner only and leave the other ranks inside ncclBroadcast
    Plan pl = {0, 0, nb};
    for (int k = 0; k < (int)panels.size(); ++k)
        if (m - panels[k].c > narrow_panel_max_rows(c))
            return set_err(-2, "m too large for the resident panel kernel (%lld rows; limit %lld)", (long long)(m - panels[k].c),
                           (long long)narrow_panel_max_rows(c));
    const bool la = c->lookahead && panels.size() > 1 && !c->sync && !c->profile;
    for (;;) {
        bool any_wide = false;
        for (int k = pl.kstart; k < (int)panels.size(); ++k) any_wide |= plan_wide(c, pl, panels, k, m);
        k_wide_reset<<<1, 32, 0, st>>>(c->wctl);
        TRY(post(c, st, "k_wide_reset"));
        const bool use_la = la && (int)panels.size() - pl.kstart > 1;
        if (!use_la && !c->up_chunks.empty()) {   // the serial schedule knows nothing about columns still in flight: wait for them
            for (const auto& u : c->up_chunks) CU(cudaStreamWaitEvent(st, u.ev, 0));
            c->up_chunks.clear();
        }
        const int rc = use_la ? qr_blocked_lookahead(c, st, m, col0, nl, A, lda, alpha, panels, pl)
                              : qr_blocked_serial(c, st, m, col0, nl, A, lda, alpha, panels, pl);
        c->up_chunks.clear();                     // every chunk has joined (or the pass failed): a restart sees the whole matrix
        if (rc || !any_wide) return rc;
        // The wide chain is speculative: its guards are evaluated on the device.  One synchronisation per factorisation to
        // learn whether a panel was refused; if so, everything from that panel on was skipped on the device and is redone
        // here, that panel with the 32-column chain (same result on every rank: the verdict travels with the V buffer).
        int fail = W_NOFAIL;
        CU(cudaMemcpyAsync(&fail, &((WideCtl*)c->wctl)->fail_step, sizeof(int), cudaMemcpyDeviceToHost, st));
        CU(cudaStreamSynchronize(st));
        if (fail == W_NOFAIL) return 0;
        if (fail < pl.kstart || fail >= (int)panels.size()) return set_err(4004, "internal: bad restart index %d", fail);
        c->wide_redone++;
        pl.kstart = fail;
        pl.wide_from = fail + 1;
    }
}

// qr!: unblocked driver (nb == 1): one reflector per step, as the reference does it (S:127-144)
static int qr_unblocked(dhqr_context* c, cudaStream_t st, int64_t m, int64_t n, int64_t col0, int64_t nl, double* A,
                        int64_t lda, double* alpha) {
    std::vector<int64_t> col0s, nls;
    TRY(gather_partition(c, st, col0, nl, col0s, nls));
    TRY(check_partition(col0s, nls, n));
    TRY(ensure_workspace(c, m, nl));
    const int64_t lend = col0 + nl;
    if (c->nranks == 1 && n > 0 && m <= (int64_t)UW_MAXI * UW_THREADS && !c->profile && !c->sync) {
        // single GPU, short columns: the whole column loop as one persistent cooperative launch (k_unblocked_wave)
        bool fresh = false;   // new flags (64 spare): the tags start over
        if (c->uw_flags.size() < (size_t)n) TRY(c->uw_flags.grow((size_t)n + 64, &fresh));
        if (fresh) c->uw_epoch = 0;
        if (c->uw_epoch > 0xFFFFFFF0u) { CU(cudaMemsetAsync(c->uw_flags, 0, sizeof(unsigned int) * c->uw_flags.size(), st)); c->uw_epoch = 0; }
        const unsigned int tag = ++c->uw_epoch;
        int nn = (int)n;
        unsigned int* flags = c->uw_flags;
        void* args[] = {&A, &lda, &m, &nn, &alpha, &flags, (void*)&tag};
        const int G = (int)std::min<int64_t>(c->sms, n);
        pre(c, st);
        cudaError_t e = cudaLaunchCooperativeKernel((void*)k_unblocked_wave, dim3(G), dim3(UW_THREADS), args, 0, st);
        if (e != cudaSuccess) return set_err(1000 + (int)e, "cooperative launch of k_unblocked_wave failed: %s", cudaGetErrorString(e));
        return post(c, st, "k_unblocked_wave", 16.0 * (double)m * n * n / 2);
    }
    if (c->nranks == 1 && n > 0 && (size_t)((m + 2) & ~(int64_t)1) * 8 * (A1_CW + 1) <= 200 * 1024) {
        // single GPU, the column tile fits in shared memory: one launch per column step (the next reflector is formed by the
        // CTA that has just updated its column, k_apply1_tma), two v buffers alternating between steps
        const int64_t voff = rup(m + 4, 2);
        k_house1<<<1, 1024, 0, st>>>(A, m, alpha, c->v1);
        TRY(post(c, st, "k_house1"));
        for (int64_t j = 0; j + 1 < n; ++j) {
            const int lead = (int)(j & 1);
            const int64_t lenw = m - j + lead, lenp = (lenw + 1) & ~(int64_t)1;
            const int nc = (int)(n - j - 1);
            double* C = A + (j + 1) * lda + (j - lead);
            const int aligned = (((uintptr_t)C & 15) == 0 && (lda & 1) == 0) ? 1 : 0;
            double* vcur = c->v1 + (j & 1) * voff, *vnext = c->v1 + ((j + 1) & 1) * voff;
            pre(c, st);
            cudaLaunchConfig_t cfg = {};
            cfg.gridDim = dim3((nc + A1_CW - 1) / A1_CW);
            cfg.blockDim = dim3(A1_THREADS);
            cfg.dynamicSmemBytes = (size_t)lenp * 8 * (A1_CW + 1);
            cfg.stream = st;
            cudaLaunchAttribute at[1];
            at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
            at[0].val.programmaticStreamSerializationAllowed = c->profile ? 0 : 1;   // event brackets want plain stream order
            cfg.attrs = at;
            cfg.numAttrs = 1;
            const double* vc = vcur;
            const int64_t ldc = lda;
            CU(cudaLaunchKernelEx(&cfg, k_apply1_tma, vc, lenw, C, ldc, nc, aligned, vnext, alpha + j + 1, lead));
            TRY(post(c, st, "k_apply1_tma", 16.0 * (double)(m - j) * nc));
        }
        return 0;
    }
    for (int owner = 0; owner < c->nranks; ++owner) {
        for (int64_t j = col0s[owner]; j < col0s[owner] + nls[owner]; ++j) {
            const int lead = (int)(j & 1);          // window starts on an even row so TMA sources stay 16B aligned
            const int64_t len = m - j;
            if (c->rank == owner) {
                if (lead) CU(cudaMemsetAsync(c->v1, 0, sizeof(double), st));
                k_house1<<<1, 1024, 0, st>>>(A + (j - col0) * lda + j, len, alpha + j, c->v1 + lead);
                TRY(post(c, st, "k_house1"));
            }
            if (c->nranks > 1) {
                NC(g_nccl.Broadcast(c->v1, c->v1, (size_t)(len + lead + 1), ncclFloat64, owner, c->comm, st));
                NC(g_nccl.Broadcast(alpha + j, alpha + j, 1, ncclFloat64, owner, c->comm, st));
            }
            const int64_t t0 = std::max(j + 1, col0);
            if (t0 >= lend) continue;
            const int nc = (int)(lend - t0);
            double* C = A + (t0 - col0) * lda + (j - lead);
            const int64_t lenw = len + lead;
            const int64_t lenp = (lenw + 1) & ~(int64_t)1;
            const size_t smem = (size_t)lenp * 8 * (A1_CW + 1);
            if (smem <= 200 * 1024) {
                const int aligned = (((uintptr_t)C & 15) == 0 && (lda & 1) == 0) ? 1 : 0;
                k_apply1_tma<<<(nc + A1_CW - 1) / A1_CW, A1_THREADS, smem, st>>>(c->v1, lenw, C, lda, nc, aligned, nullptr, nullptr, lead);
                TRY(post(c, st, "k_apply1_tma"));
            } else {
                k_apply1_direct<<<std::min(nc, 8 * c->sms), A1_THREADS, 0, st>>>(c->v1, lenw, C, lda, nc);
                TRY(post(c, st, "k_apply1_direct"));
            }
        }
    }
    return 0;
}

// ------------------------------------------------------------------------------------------------
// solve phases
// ------------------------------------------------------------------------------------------------
// Q'b on the local reflectors: panels of <= 128 reflectors, each applied as a block reflector
// built from V alone (T recomputed from V'V), so only (A, alpha) are needed, like the reference.
static int apply_qt_local(dhqr_context* c, cudaStream_t st, int64_t m, int64_t col0, int64_t nl, const double* A,
                          int64_t lda, double* b, int64_t ldb, int nrhs, int notrans = 0) {
    // notrans: b <- Q b = H_1 (H_2 (... H_n b)): the panels in reverse order, each as I - V T V' (T instead of T')
    if (nl <= 0) return 0;
    const int64_t ofirst = notrans ? ((nl - 1) / NBMAX) * NBMAX : 0, ostep = notrans ? -(int64_t)NBMAX : NBMAX;
    for (int64_t o = ofirst; o >= 0 && o < nl; o += ostep) {
        const int kb = (int)std::min<int64_t>(NBMAX, nl - o);
        const int64_t cs = col0 + o;
        const PanelGeom g = panel_geom({0, cs, kb}, m);
        const int nbp = kb <= IB ? IB : NBMAX;
        TRY(pack_panel(c, st, A + o * lda + cs, lda, m - cs, kb, 1, c->vpk2[0], cs - g.r0, g.vrows, nbp));
        TRY(apply_block_reflector(c, st, c->vpk2[0], c->ws[0], 0, nbp, g.rows, cs - g.r0, b + g.r0, ldb, nrhs, false, nullptr, 0, notrans));
    }
    return 0;
}

// One right-hand side: T' of every local panel first (independent of b, so with several ranks every rank does this while b is
// still with its predecessors), then the sweep with two GEMV-shaped launches per panel (k_qt_dot, k_qt_axpy).
static constexpr int QT_MAXG = 1024;
static int qt_prepare(dhqr_context* c, cudaStream_t st, int64_t m, int64_t col0, int64_t nl, const double* A, int64_t lda) {
    const int npl = (int)((nl + NBMAX - 1) / NBMAX);
    if (npl <= 0) return 0;
    TRY(c->qt_T.grow((size_t)npl * NBMAX * NBMAX));
    TRY(c->qt_part.grow((size_t)(QT_MAXG + 1) * WP));     // last row: y
    TRY(c->qt_ticket.grow(1));
    auto& w = c->ws[0];
    if ((size_t)npl * NBMAX * NBMAX > w.wsum.size()) return set_err(4006, "internal: Gram workspace too small");
    for (int p = 0; p < npl; ++p) {
        const int64_t o = (int64_t)p * NBMAX, cs = col0 + o;
        const int kb = (int)std::min<int64_t>(NBMAX, nl - o);
        const PanelGeom g = panel_geom({0, cs, kb}, m);
        TRY(pack_panel(c, st, A + o * lda + cs, lda, m - cs, kb, 1, c->vpk2[0], cs - g.r0, g.vrows, NBMAX));
        int nsplit = 0;
        int64_t pstride = 0;
        TRY(launch_panel_gram(c, st, c->vpk2[0], w, g.rows, &nsplit, &pstride));
        pre(c, st);
        k_wreduce4<<<(WP * WP * 4) / 256, 256, 0, st>>>(w.wpart, pstride, nsplit, (int64_t)WP * WP, w.wsum + (size_t)p * WP * WP);
        TRY(post(c, st, "k_wreduce4"));
    }
    pre(c, st);
    k_tinv<128><<<npl, 512, smem_tinv(128), st>>>(w.wsum, c->qt_T, (int64_t)WP * WP);
    TRY(post(c, st, "k_tinv128"));
    return 0;
}

static int apply_qt_local_vec(dhqr_context* c, cudaStream_t st, int64_t m, int64_t col0, int64_t nl, const double* A, int64_t lda,
                              double* b, int notrans) {
    const int npl = (int)((nl + NBMAX - 1) / NBMAX);
    for (int q = 0; q < npl; ++q) {
        const int p = notrans ? npl - 1 - q : q;
        const int64_t o = (int64_t)p * NBMAX, cs = col0 + o;
        QtArgs a;
        a.V = A + o * lda + cs; a.lda = lda; a.mp = m - cs; a.kb = (int)std::min<int64_t>(NBMAX, nl - o);
        a.b = b + cs; a.Linv = c->qt_T + (size_t)p * NBMAX * NBMAX;
        a.part = c->qt_part; a.y = c->qt_part + (size_t)QT_MAXG * WP; a.ticket = c->qt_ticket; a.trans = notrans;
        int64_t rpc = rup(std::max<int64_t>((a.mp + c->sms - 1) / c->sms, 64), 32);                // one CTA per SM
        rpc = std::min<int64_t>(rpc, QT_MAXROWS);
        const int64_t G = (a.mp + rpc - 1) / rpc;
        if (G > QT_MAXG) return set_err(4007, "internal: too many k_qt_dot CTAs");                  // callers check m first
        a.rows_per_cta = (int)rpc;
        pre(c, st);
        k_qt_dot<<<(unsigned)G, QT_THREADS, 0, st>>>(a);
        TRY(post(c, st, "k_qt_dot", 8.0 * (double)a.mp * a.kb));
        pre(c, st);
        k_qt_axpy<<<(unsigned)((a.mp + QT_AROWS - 1) / QT_AROWS), QT_ATHREADS, 0, st>>>(a);
        TRY(post(c, st, "k_qt_axpy", 8.0 * (double)a.mp * a.kb));
    }
    return 0;
}
static bool qt_vec_ok(const dhqr_context* c, int64_t m, int nrhs) { return c->qt_vec && nrhs == 1 && m <= (int64_t)QT_MAXG * QT_MAXROWS; }

static constexpr size_t BS_BLOCK_WORDS = 32 * 2;   // k_backsolve_wave cells of one 32-row block: 32 cells of 2 words

static int backsolve_local(dhqr_context* c, cudaStream_t st, int64_t col0, int64_t nl, const double* A, int64_t lda,
                           const double* alpha, double* y, int64_t ldy, int nrhs, double* x, int64_t ldx) {
    if (nl <= 0) return 0;
    // one launch per right-hand side: a wavefront over 32-row strips (k_backsolve_wave); needs every CTA resident at once
    const int64_t nbk = (nl + 31) / 32, nlow = (col0 + 31) / 32;
    if (nbk + nlow <= c->bs_wave_max_ctas && nbk <= (int64_t)(c->bs_cells.size() / BS_BLOCK_WORDS)) {
        for (int rhs = 0; rhs < nrhs; ++rhs) {
            if (c->bs_epoch > 0xFFFFFFF0u) {
                CU(cudaMemsetAsync(c->bs_cells, 0, sizeof(unsigned long long) * c->bs_cells.size(), st));
                c->bs_epoch = 0;
            }
            k_backsolve_wave<<<(unsigned)(nbk + nlow), BW_THREADS, 0, st>>>(A, lda, alpha, y + (int64_t)rhs * ldy, x + (int64_t)rhs * ldx, col0, nl,
                                                                          (int)nlow, c->bs_cells, ++c->bs_epoch);
            TRY(post(c, st, "k_backsolve_wave"));
        }
        return 0;
    }
    // fallback: blocks of BS_BLK columns, last to first (S:260: i = n:-1:1), one launch per block
    for (int64_t o = ((nl - 1) / BS_BLK) * BS_BLK; o >= 0; o -= BS_BLK) {
        const int bs = (int)std::min<int64_t>(BS_BLK, nl - o);
        const int64_t c0 = col0 + o;
        const int grid = (int)std::max<int64_t>(1, std::min<int64_t>((c0 + 255) / 256, 2 * c->sms));
        k_backsolve_step<<<grid, 256, 0, st>>>(A + o * lda, lda, alpha, y, ldy, nrhs, x, ldx, c0, bs);
        TRY(post(c, st, "k_backsolve_step"));
    }
    return 0;
}

// The options of dhqr_set_option / dhqr_get_option (documented in include/dhqr.h).  A flag stores any nonzero value as 1;
// a bounded option refuses, with range_err, a value outside [lo, hi] or not a multiple of mult; wide_kappa is a double
// read back truncated; a read-only option has a getter instead of a member.
struct OptionDef {
    const char* key;
    enum Kind { FLAG, INT, REAL, READ_ONLY } kind;
    int dhqr_context::*ival;                   // FLAG, INT
    double dhqr_context::*dval;                // REAL
    int64_t lo, hi, mult;                      // INT, REAL
    const char* range_err;                     // INT, REAL
    int (*get)(dhqr_context*, int64_t*);       // READ_ONLY
};
static int get_fast_stat(dhqr_context* c, int which, int64_t* value) {
    int st2[2] = {0, 0};
    if (c->fast_stats) CU(cudaMemcpy(st2, c->fast_stats, sizeof(st2), cudaMemcpyDeviceToHost));
    *value = st2[which];
    return 0;
}
static const OptionDef OPTIONS[] = {
    {"nb", OptionDef::INT, &dhqr_context::nb, nullptr, 32, 128, 32, "nb must be a multiple of 32 in [32,128]"},
    {"sync", OptionDef::FLAG, &dhqr_context::sync},
    {"profile", OptionDef::FLAG, &dhqr_context::profile},
    {"lookahead", OptionDef::FLAG, &dhqr_context::lookahead},
    {"host_trace", OptionDef::FLAG, &dhqr_context::host_trace},
    {"host_chunk", OptionDef::INT, &dhqr_context::host_chunk, nullptr, 0, INT64_MAX, 128, "host_chunk must be a non-negative multiple of 128"},
    {"host_first", OptionDef::INT, &dhqr_context::host_first, nullptr, 0, INT64_MAX, 1, "host_first < 0"},
    {"host_h2d_gbs", OptionDef::INT, &dhqr_context::host_h2d_gbs, nullptr, 1, INT64_MAX, 1, "host_h2d_gbs < 1"},
    {"host_chain_us", OptionDef::INT, &dhqr_context::host_chain_us, nullptr, 1, INT64_MAX, 1, "host_chain_us < 1"},
    {"host_tflops", OptionDef::INT, &dhqr_context::host_tflops, nullptr, 1, INT64_MAX, 1, "host_tflops < 1"},
    {"qt_vec", OptionDef::FLAG, &dhqr_context::qt_vec},
    {"panel_fast", OptionDef::FLAG, &dhqr_context::panel_fast},
    {"wide_panel", OptionDef::FLAG, &dhqr_context::wide_panel},
    {"wide_kappa", OptionDef::REAL, nullptr, &dhqr_context::wide_kappa, 1, INT64_MAX, 1, "wide_kappa < 1"},
    {"wide_panels", OptionDef::READ_ONLY, nullptr, nullptr, 0, 0, 0, nullptr, [](dhqr_context* c, int64_t* v) { *v = c->wide_panels; return 0; }},
    {"wide_redone", OptionDef::READ_ONLY, nullptr, nullptr, 0, 0, 0, nullptr, [](dhqr_context* c, int64_t* v) { *v = c->wide_redone; return 0; }},
    {"panels_fast", OptionDef::READ_ONLY, nullptr, nullptr, 0, 0, 0, nullptr, [](dhqr_context* c, int64_t* v) { return get_fast_stat(c, 0, v); }},
    {"panels_fallback", OptionDef::READ_ONLY, nullptr, nullptr, 0, 0, 0, nullptr, [](dhqr_context* c, int64_t* v) { return get_fast_stat(c, 1, v); }},
    {"sms", OptionDef::READ_ONLY, nullptr, nullptr, 0, 0, 0, nullptr, [](dhqr_context* c, int64_t* v) { *v = c->sms; return 0; }},
    {"rank", OptionDef::READ_ONLY, nullptr, nullptr, 0, 0, 0, nullptr, [](dhqr_context* c, int64_t* v) { *v = c->rank; return 0; }},
    {"nranks", OptionDef::READ_ONLY, nullptr, nullptr, 0, 0, 0, nullptr, [](dhqr_context* c, int64_t* v) { *v = c->nranks; return 0; }},
};
static const OptionDef* find_option(const char* key) {
    for (const OptionDef& o : OPTIONS)
        if (!strcmp(o.key, key)) return &o;
    return nullptr;
}

// ------------------------------------------------------------------------------------------------
// C-ABI
// ------------------------------------------------------------------------------------------------
extern "C" {

int dhqr_version(void) { return DHQR_VERSION; }
const char* dhqr_last_error(void) { return g_err; }

static int create_common(dhqr_handle* h, int device) {
    if (!h) return set_err(-1, "null handle pointer");
    int ndev = 0;
    CU(cudaGetDeviceCount(&ndev));
    if (device < 0 || device >= ndev) return set_err(-2, "device %d out of range (%d devices)", device, ndev);
    CU(cudaSetDevice(device));
    cudaDeviceProp prop;
    CU(cudaGetDeviceProperties(&prop, device));
    if (prop.major < 10) return set_err(5001, "libdhqr is built for sm_100a only; device %d is sm_%d%d", device, prop.major, prop.minor);
    std::unique_ptr<dhqr_context> c(new dhqr_context());   // a failure below releases what was made so far
    c->device = device;
    c->sms = prop.multiProcessorCount;
    TRY(c->d_i64.grow(2 * 1025));
    CU(c->copy_stream.create());
    CU(c->d2h_stream.create());
    CU(c->h2d_stream.create());
    for (int i = 0; i < CU_STREAMS; ++i) CU(c->cu_stream[i].create());
    {
        int lo = 0, hi = 0;
        CU(cudaDeviceGetStreamPriorityRange(&lo, &hi));
        CU(c->hp_stream.create(hi));
        CU(c->comm_stream.create(hi));
        CU(c->hp2_stream.create(hi));
        CU(c->aux_stream.create(hi));
        for (int i = 0; i < 4; ++i) CU(c->ev_aux[i].create(cudaEventDisableTiming));
    }
    *h = c.release();
    return 0;
}

int dhqr_create(dhqr_handle* h, int device) { return create_common(h, device); }

int dhqr_nccl_unique_id(void* out) {
    if (!out) return set_err(-1, "null output");
    TRY(load_nccl());
    ncclUniqueId id;
    NC(g_nccl.GetUniqueId(&id));
    memcpy(out, &id, sizeof(id));
    return 0;
}

int dhqr_create_dist(dhqr_handle* h, int device, const void* unique_id, int rank, int nranks) {
    if (nranks < 1 || nranks > 1024) return set_err(-5, "nranks out of range");
    if (rank < 0 || rank >= nranks) return set_err(-4, "rank out of range");
    if (nranks > 1 && !unique_id) return set_err(-3, "null unique id");
    TRY(create_common(h, device));
    dhqr_context* c = *h;
    c->rank = rank;
    c->nranks = nranks;
    if (nranks > 1) {
        TRY(load_nccl());
        ncclUniqueId id;
        memcpy(&id, unique_id, sizeof(id));
        NC(g_nccl.CommInitRank(&c->comm, nranks, id, rank));
    }
    return 0;
}

int dhqr_destroy(dhqr_handle c) {
    if (!c) return 0;
    cudaSetDevice(c->device);
    cudaDeviceSynchronize();
    if (c->comm) g_nccl.CommDestroy(c->comm);
    delete c;   // the owners release every buffer, stream and event
    return 0;
}

int dhqr_set_option(dhqr_handle c, const char* key, int64_t value) {
    if (!c) return set_err(-1, "null handle");
    if (!key) return set_err(-2, "null key");
    const OptionDef* o = find_option(key);
    if (!o || o->kind == OptionDef::READ_ONLY) return set_err(-2, "unknown option '%s'", key);
    if (o->kind == OptionDef::FLAG) {
        c->*o->ival = value ? 1 : 0;
        return 0;
    }
    if (value < o->lo || value > o->hi || value % o->mult) return set_err(-3, "%s", o->range_err);
    if (o->kind == OptionDef::REAL) c->*o->dval = (double)value;
    else c->*o->ival = (int)value;
    return 0;
}

int dhqr_get_option(dhqr_handle c, const char* key, int64_t* value) {
    if (!c) return set_err(-1, "null handle");
    if (!key) return set_err(-2, "null key");
    if (!value) return set_err(-3, "null value");
    const OptionDef* o = find_option(key);
    if (!o) return set_err(-2, "unknown option '%s'", key);
    if (o->kind == OptionDef::READ_ONLY) return o->get(c, value);
    *value = o->kind == OptionDef::REAL ? (int64_t)(c->*o->dval) : c->*o->ival;
    return 0;
}

int dhqr_launch_count(dhqr_handle c, int64_t* count) {
    if (!c) return set_err(-1, "null handle");
    if (!count) return set_err(-2, "null count");
    *count = c->launches;
    return 0;
}

static int prof_drain(dhqr_context* c) {
    for (auto& r : c->prof_pending) {
        float ms = 0.f;
        CU(cudaEventSynchronize(r.e1));
        CU(cudaEventElapsedTime(&ms, r.e0, r.e1));
        c->prof_slots[r.slot].ms += ms;
        c->prof_slots[r.slot].count += 1;
    }
    c->prof_pending.clear();
    return 0;
}

int dhqr_profile_reset(dhqr_handle c) {
    if (!c) return set_err(-1, "null handle");
    TRY(prof_drain(c));
    for (auto& s : c->prof_slots) { s.ms = 0.0; s.count = 0; s.work = 0.0; }
    return 0;
}

int dhqr_profile_get(dhqr_handle c, int index, char* name, int name_len, double* ms, int64_t* count, double* work) {
    if (!c) return set_err(-1, "null handle");
    TRY(prof_drain(c));
    if (index < 0 || index >= (int)c->prof_slots.size()) return set_err(-2, "index out of range");
    const auto& s = c->prof_slots[index];
    if (name && name_len > 0) { strncpy(name, s.name, name_len - 1); name[name_len - 1] = 0; }
    if (ms) *ms = s.ms;
    if (count) *count = s.count;
    if (work) *work = s.work;
    return 0;
}

int dhqr_qr_f64(dhqr_handle c, int64_t m, int64_t n_global, int64_t col0, int64_t n_local, double* dA, int64_t lda,
                double* d_alpha, int nb, void* stream) {
    TRY(check_common(c, m, n_global, col0, n_local, dA, lda));
    if (n_global > 0 && !d_alpha) return set_err(-8, "null alpha");
    if (nb == 0) nb = c->nb;
    if (nb != 1 && (nb < 32 || nb > 128 || nb % 32)) return set_err(-9, "nb must be 0, 1 or a multiple of 32 in [32,128]");
    if (n_global == 0) return 0;
    CU(cudaSetDevice(c->device));
    cudaStream_t st = (cudaStream_t)stream;
    if (nb == 1) return qr_unblocked(c, st, m, n_global, col0, n_local, dA, lda, d_alpha);
    return qr_blocked(c, st, m, n_global, col0, n_local, dA, lda, d_alpha, nb);
}

// b <- Q'b (notrans = 0; C3, S:227-229: the owners act on b one after the other, b travels rank -> rank + 1) or
// b <- Qb = H_1 ... H_n b (notrans = 1: the owners act in reverse rank order, b travels rank -> rank - 1)
static int apply_q_sweep(dhqr_context* c, int64_t m, int64_t n_global, int64_t col0, int64_t n_local, const double* dA, int64_t lda,
                         double* d_b, int64_t ldb, int nrhs, void* stream, int notrans) {
    TRY(check_common(c, m, n_global, col0, n_local, dA, lda));
    TRY(check_rhs(m, nrhs, d_b, ldb, 8, 9, 10));
    if (n_global == 0 || nrhs == 0) return 0;
    CU(cudaSetDevice(c->device));
    cudaStream_t st = (cudaStream_t)stream;
    std::vector<int64_t> col0s, nls;
    TRY(gather_partition(c, st, col0, n_local, col0s, nls));
    TRY(check_partition(col0s, nls, n_global));
    TRY(ensure_workspace(c, m, std::max<int64_t>(n_local, nrhs)));
    const int from = notrans ? c->rank + 1 : c->rank - 1, to = notrans ? c->rank - 1 : c->rank + 1;
    const int last = notrans ? 0 : c->nranks - 1;   // the rank that finishes b
    const size_t cnt = (size_t)ldb * (nrhs - 1) + m;
    const bool vec = qt_vec_ok(c, m, nrhs);
    if (vec) TRY(qt_prepare(c, st, m, col0, n_local, dA, lda));
    if (c->nranks > 1 && from >= 0 && from < c->nranks) NC(g_nccl.Recv(d_b, cnt, ncclFloat64, from, c->comm, st));
    if (vec) TRY(apply_qt_local_vec(c, st, m, col0, n_local, dA, lda, d_b, notrans));
    else TRY(apply_qt_local(c, st, m, col0, n_local, dA, lda, d_b, ldb, nrhs, notrans));
    if (c->nranks > 1) {
        if (to >= 0 && to < c->nranks) NC(g_nccl.Send(d_b, cnt, ncclFloat64, to, c->comm, st));
        NC(g_nccl.Broadcast(d_b, d_b, cnt, ncclFloat64, last, c->comm, st));
    }
    return 0;
}

int dhqr_apply_qt_f64(dhqr_handle c, int64_t m, int64_t n_global, int64_t col0, int64_t n_local, const double* dA,
                      int64_t lda, double* d_b, int64_t ldb, int nrhs, void* stream) {
    return apply_q_sweep(c, m, n_global, col0, n_local, dA, lda, d_b, ldb, nrhs, stream, 0);
}

int dhqr_apply_q_f64(dhqr_handle c, int64_t m, int64_t n_global, int64_t col0, int64_t n_local, const double* dA,
                     int64_t lda, double* d_b, int64_t ldb, int nrhs, void* stream) {
    return apply_q_sweep(c, m, n_global, col0, n_local, dA, lda, d_b, ldb, nrhs, stream, 1);
}

int dhqr_backsolve_f64(dhqr_handle c, int64_t m, int64_t n_global, int64_t col0, int64_t n_local, const double* dA,
                       int64_t lda, const double* d_alpha, double* d_b, int64_t ldb, int nrhs, void* stream) {
    TRY(check_common(c, m, n_global, col0, n_local, dA, lda));
    if (n_global > 0 && !d_alpha) return set_err(-8, "null alpha");
    TRY(check_rhs(m, nrhs, d_b, ldb, 9, 10, 11));
    if (n_global == 0 || nrhs == 0) return 0;
    CU(cudaSetDevice(c->device));
    cudaStream_t st = (cudaStream_t)stream;
    std::vector<int64_t> col0s, nls;
    TRY(gather_partition(c, st, col0, n_local, col0s, nls));
    TRY(check_partition(col0s, nls, n_global));
    TRY(c->xbuf.grow((size_t)n_global * nrhs));
    const size_t blocks = (size_t)(n_local + 31) / 32;
    bool fresh = false;   // new cells (64 blocks spare): the tags start over
    if (c->bs_cells.size() < (blocks + 1) * BS_BLOCK_WORDS) TRY(c->bs_cells.grow((blocks + 64) * BS_BLOCK_WORDS, &fresh));
    if (fresh) c->bs_epoch = 0;
    if (!c->bs_wave_max_ctas) {
        int per_sm = 0;
        CU(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_backsolve_wave, BW_THREADS, 0));
        c->bs_wave_max_ctas = std::max(1, per_sm * c->sms);
    }
    // C4 (S:260-267), column oriented: the last owner solves its block of unknowns and removes their
    // contribution from the rows above; the partially reduced right-hand side then moves one rank down.
    const size_t cnt = (size_t)ldb * (nrhs - 1) + n_global;
    if (c->nranks > 1 && c->rank + 1 < c->nranks) {
        NC(g_nccl.Recv(d_b, cnt, ncclFloat64, c->rank + 1, c->comm, st));
        NC(g_nccl.Recv(c->xbuf, (size_t)n_global * nrhs, ncclFloat64, c->rank + 1, c->comm, st));
    }
    TRY(backsolve_local(c, st, col0, n_local, dA, lda, d_alpha, d_b, ldb, nrhs, c->xbuf, n_global));
    if (c->nranks > 1) {
        if (c->rank > 0) {
            NC(g_nccl.Send(d_b, cnt, ncclFloat64, c->rank - 1, c->comm, st));
            NC(g_nccl.Send(c->xbuf, (size_t)n_global * nrhs, ncclFloat64, c->rank - 1, c->comm, st));
        }
        NC(g_nccl.Broadcast(c->xbuf, c->xbuf, (size_t)n_global * nrhs, ncclFloat64, 0, c->comm, st));
    }
    CU(cudaMemcpy2DAsync(d_b, (size_t)ldb * 8, c->xbuf, (size_t)n_global * 8, (size_t)n_global * 8, nrhs,
                         cudaMemcpyDeviceToDevice, st));
    return 0;
}

int dhqr_solve_f64(dhqr_handle c, int64_t m, int64_t n_global, int64_t col0, int64_t n_local, const double* dA,
                   int64_t lda, const double* d_alpha, double* d_b, int64_t ldb, int nrhs, void* stream) {
    TRY(dhqr_apply_qt_f64(c, m, n_global, col0, n_local, dA, lda, d_b, ldb, nrhs, stream));   // S:288
    return dhqr_backsolve_f64(c, m, n_global, col0, n_local, dA, lda, d_alpha, d_b, ldb, nrhs, stream);   // S:291
}

// ---- ComplexF64 (S:9, S:51-59, S:162-196; test/runtests.jl:43) -------------------------------------------------------
// Panels of 64 complex columns: complex column-by-column panel, then the trailing update as the REAL block reflector of the
// 128 vectors [v_r, v_i] on the real view of the matrix (dhqr_complex.cuh).  Single GPU.
static int check_complex(dhqr_context* c, int64_t m, int64_t n_global, int64_t col0, int64_t n_local, const void* A, int64_t lda) {
    TRY(check_common(c, m, n_global, col0, n_local, A, lda));
    if (c->nranks != 1 || col0 != 0 || n_local != n_global) return set_err(-1, "the ComplexF64 path is single-GPU (col0 = 0, n_local = n_global)");
    return 0;
}

static int pack_complex_panel(dhqr_context* c, cudaStream_t st, const double2* P, int64_t lda, int64_t mpc, int kb, int64_t vrows) {
    dim3 grid((unsigned)std::min<int64_t>((vrows + 255) / 256, 4 * c->sms), NBMAX);
    k_pack_c<<<grid, 256, 0, st>>>(P, lda, mpc, kb, c->vpk2[0], 0, vrows);
    return post(c, st, "k_pack_c");
}

int dhqr_qr_c64(dhqr_handle c, int64_t m, int64_t n_global, int64_t col0, int64_t n_local, void* dA, int64_t lda, void* d_alpha,
                void* stream) {
    TRY(check_complex(c, m, n_global, col0, n_local, dA, lda));
    if (n_global > 0 && !d_alpha) return set_err(-8, "null alpha");
    if (n_global == 0) return 0;
    CU(cudaSetDevice(c->device));
    cudaStream_t st = (cudaStream_t)stream;
    const int64_t n = n_global;
    TRY(ensure_workspace(c, 2 * m, n));
    double2* A = (double2*)dA;
    double2* alpha = (double2*)d_alpha;
    for (int64_t c0 = 0; c0 < n; c0 += CPW) {
        const int kb = (int)std::min<int64_t>(CPW, n - c0);
        double2* P = A + c0 * lda + c0;
        const int64_t mpc = m - c0;
        for (int j = 0; j < kb; ++j) {                       // S:127-144 restricted to the panel
            double2* col = P + (int64_t)j * lda + j;
            k_house1_c<<<1, 1024, 0, st>>>(col, mpc - j, alpha + c0 + j);
            TRY(post(c, st, "k_house1_c"));
            if (j + 1 < kb) {
                k_apply1_c<<<kb - j - 1, 256, 0, st>>>(col, mpc - j, col + lda, lda, kb - j - 1);
                TRY(post(c, st, "k_apply1_c"));
            }
        }
        const int64_t t0 = c0 + kb;
        if (t0 < n) {                                        // S:198-213 for the columns right of the panel, blocked
            const int64_t rows = 2 * mpc, vrows = rup(rows, 128);
            TRY(pack_complex_panel(c, st, P, lda, mpc, kb, vrows));
            TRY(apply_block_reflector(c, st, c->vpk2[0], c->ws[0], 0, NBMAX, rows, 0, (double*)(A + t0 * lda + c0), 2 * lda, (int)(n - t0)));
        }
    }
    return 0;
}

int dhqr_apply_qt_c64(dhqr_handle c, int64_t m, int64_t n_global, int64_t col0, int64_t n_local, const void* dA, int64_t lda,
                      void* d_b, int64_t ldb, int nrhs, void* stream) {
    TRY(check_complex(c, m, n_global, col0, n_local, dA, lda));
    TRY(check_rhs(m, nrhs, d_b, ldb, 8, 9, 10));
    if (n_global == 0 || nrhs == 0) return 0;
    CU(cudaSetDevice(c->device));
    cudaStream_t st = (cudaStream_t)stream;
    TRY(ensure_workspace(c, 2 * m, std::max<int64_t>(n_global, nrhs)));
    const double2* A = (const double2*)dA;
    double2* b = (double2*)d_b;
    for (int64_t c0 = 0; c0 < n_global; c0 += CPW) {         // S:232-242, panel by panel
        const int kb = (int)std::min<int64_t>(CPW, n_global - c0);
        const int64_t mpc = m - c0, rows = 2 * mpc, vrows = rup(rows, 128);
        TRY(pack_complex_panel(c, st, A + c0 * lda + c0, lda, mpc, kb, vrows));
        TRY(apply_block_reflector(c, st, c->vpk2[0], c->ws[0], 0, NBMAX, rows, 0, (double*)(b + c0), 2 * ldb, nrhs));
    }
    return 0;
}

int dhqr_backsolve_c64(dhqr_handle c, int64_t m, int64_t n_global, int64_t col0, int64_t n_local, const void* dA, int64_t lda,
                       const void* d_alpha, void* d_b, int64_t ldb, int nrhs, void* stream) {
    TRY(check_complex(c, m, n_global, col0, n_local, dA, lda));
    if (n_global > 0 && !d_alpha) return set_err(-8, "null alpha");
    TRY(check_rhs(m, nrhs, d_b, ldb, 9, 10, 11));
    if (n_global == 0 || nrhs == 0) return 0;
    CU(cudaSetDevice(c->device));
    cudaStream_t st = (cudaStream_t)stream;
    const int64_t n = n_global;
    TRY(c->xbuf.grow((size_t)2 * n * nrhs));
    const double2* A = (const double2*)dA;
    double2* x = (double2*)(double*)c->xbuf;
    for (int64_t o = ((n - 1) / BS_BLK) * BS_BLK; o >= 0; o -= BS_BLK) {     // S:260: i = n:-1:1, by blocks
        const int bs = (int)std::min<int64_t>(BS_BLK, n - o);
        const int grid = (int)std::max<int64_t>(1, std::min<int64_t>((o + 255) / 256, 2 * c->sms));
        k_backsolve_step_c<<<grid, 256, 0, st>>>(A + o * lda, lda, (const double2*)d_alpha, (double2*)d_b, ldb, nrhs, x, n, o, bs);
        TRY(post(c, st, "k_backsolve_step_c"));
    }
    CU(cudaMemcpy2DAsync(d_b, (size_t)ldb * 16, x, (size_t)n * 16, (size_t)n * 16, nrhs, cudaMemcpyDeviceToDevice, st));
    return 0;
}

int dhqr_solve_c64(dhqr_handle c, int64_t m, int64_t n_global, int64_t col0, int64_t n_local, const void* dA, int64_t lda,
                   const void* d_alpha, void* d_b, int64_t ldb, int nrhs, void* stream) {
    TRY(dhqr_apply_qt_c64(c, m, n_global, col0, n_local, dA, lda, d_b, ldb, nrhs, stream));                   // S:288
    return dhqr_backsolve_c64(c, m, n_global, col0, n_local, dA, lda, d_alpha, d_b, ldb, nrhs, stream);       // S:291
}

int dhqr_partialdot_c64(dhqr_handle c, const void* d_a, const void* d_b, int64_t i0, int64_t i1, void* d_out, void* stream) {
    if (!c) return set_err(-1, "null handle");
    if (!d_a) return set_err(-2, "null a");
    if (!d_b) return set_err(-3, "null b");
    if (i0 < 0) return set_err(-4, "i0 < 0");
    if (i1 < i0) return set_err(-5, "i1 < i0");
    if (!d_out) return set_err(-6, "null out");
    CU(cudaSetDevice(c->device));
    cudaStream_t st = (cudaStream_t)stream;
    k_partialdot_c<<<1, 1024, 0, st>>>((const double2*)d_a, (const double2*)d_b, i0, i1, (double2*)d_out);
    return post(c, st, "k_partialdot_c");
}

// ---- host-buffer entry points --------------------------------------------------------------------
// Plan of the chunked upload of dhqr_qr_host_f64: chunk boundaries B (multiples of nb; B[0] = 0, B.back() = n) and, for every
// chunk after the first, the step of the look-ahead schedule at which it joins the trailing matrix.  A chunk joins as soon as
// the model says it has arrived (earlier = less catch-up work), at the latest one step before the panel chain reaches into it.
// The model has two parameters (options host_h2d_gbs, host_tflops); a wrong guess costs idle time, never correctness: the
// driver orders every use of a chunk behind its upload event and forces a join that the plan names too late.
struct UploadModel { int chunk, first, h2d_gbs, tflops, chain_us; };
static void plan_upload(const UploadModel* c, int64_t m, int64_t n, int nb, std::vector<int64_t>& B, std::vector<int>& join) {
    B.assign(1, 0);
    join.assign(1, 0);
    // the schedule starts on panels 0..2: the first (exposed) upload is those three panels unless option host_first asks for more;
    // the second chunk ends where a first chunk of 1.5 chunks would have, so that the later boundaries do not move
    const int64_t chunk = rup(c->chunk, nb), second = std::max(rup(chunk + chunk / 2, nb), 3 * (int64_t)nb);
    const int64_t first = c->first > 0 ? std::min(std::max(rup(c->first, nb), 3 * (int64_t)nb), second) : 3 * (int64_t)nb;
    if (c->chunk <= 0 || m < n || n < second + chunk) { B.push_back(n); return; }
    B.push_back(first);
    if (second > first) B.push_back(second);
    while (B.back() < n) B.push_back(std::min(n, B.back() + chunk));
    if (n - B[B.size() - 2] < chunk / 2) B.erase(B.end() - 2);           // no sliver at the end
    const int nch = (int)B.size() - 1, K = (int)((n + nb - 1) / nb);
    const double U = 1e9 * c->h2d_gbs, R = 1e12 * c->tflops, chain = 1e-6 * c->chain_us;
    auto tup = [&](int j) { return (double)B[j + 1] * (double)m * 8.0 / U; };
    join.assign(nch, 0);
    double T = tup(0);
    int64_t wend = B[1];
    int nxt = 1;
    for (int k = 0; k < K; ++k) {
        while (nxt < nch && (B[nxt] < std::min<int64_t>(n, (int64_t)nb * (k + 4)) || tup(nxt) <= T)) {
            T = std::max(T, tup(nxt));                        // (the catch-up runs beside the schedule on its own stream)
            join[nxt] = k;
            wend = B[nxt + 1];
            ++nxt;
        }
        T += std::max(chain, 4.0 * (double)(m - (int64_t)nb * k) * nb * (double)std::max<int64_t>(0, wend - (int64_t)nb * (k + 1)) / R);
    }
}

int dhqr_plan_host_upload(int64_t m, int64_t n, int nb, int chunk, int first, int h2d_gbs, int tflops, int chain_us, int cap,
                          int64_t* bounds, int* join, int* nchunks) {
    if (m < 0) return set_err(-1, "m < 0");
    if (n < 0 || n > m) return set_err(-2, "need 0 <= n <= m");
    if (nb < 32 || nb > 128 || nb % 32) return set_err(-3, "nb must be a multiple of 32 in [32,128]");
    if (chunk < 0 || first < 0) return set_err(chunk < 0 ? -4 : -5, "negative width");
    if (h2d_gbs < 1 || tflops < 1 || chain_us < 1) return set_err(h2d_gbs < 1 ? -6 : (tflops < 1 ? -7 : -8), "model parameters must be positive");
    if (!bounds || !join || !nchunks) return set_err(!bounds ? -10 : (!join ? -11 : -12), "null output");
    const UploadModel um = {chunk, first, h2d_gbs, tflops, chain_us};
    std::vector<int64_t> B;
    std::vector<int> J;
    plan_upload(&um, m, n, nb, B, J);
    const int nch = (int)B.size() - 1;
    if (cap < nch + 1) return set_err(-9, "cap too small: %d chunks", nch);
    for (int j = 0; j <= nch; ++j) bounds[j] = B[j];
    for (int j = 0; j < nch; ++j) join[j] = J[j];
    *nchunks = nch;
    return 0;
}

int dhqr_qr_host_f64(dhqr_handle c, int64_t m, int64_t n, double* hA, int64_t lda, double* h_alpha, int nb) {
    TRY(check_common(c, m, n, 0, n, hA, lda));
    if (n > 0 && !h_alpha) return set_err(-6, "null alpha");
    if (c->nranks != 1) return set_err(-1, "host entry points are single-GPU");
    if (nb != 0 && nb != 1 && (nb < 32 || nb > 128 || nb % 32)) return set_err(-9, "nb must be 0, 1 or a multiple of 32 in [32,128]");
    if (n == 0) return 0;
    CU(cudaSetDevice(c->device));
    const int64_t ldd = rup(m, 32);                       // padded device leading dimension (aligned TMA sources)
    const bool blocked = (nb != 1);
    const int nbe = nb == 0 ? c->nb : nb;
    // The matrix goes up in column chunks.  Only the first upload is exposed: the factorisation starts on it, every later chunk
    // travels while the device works and joins the trailing matrix through a catch-up (qr_blocked_lookahead); finished panels
    // stream back while later panels are factored.  One factorisation, the same reflectors as with the matrix resident.
    std::vector<int64_t> B;
    std::vector<int> join;
    const UploadModel um = {c->host_chunk, c->host_first, c->host_h2d_gbs, c->host_tflops, c->host_chain_us};
    if (blocked) plan_upload(&um, m, n, nbe, B, join);
    else { B = {0, n}; join = {0}; }
    const int nch = (int)B.size() - 1;
    TRY(c->hostA.grow((size_t)ldd * n + (size_t)n));
    // everything sized once, before the pipeline starts: growing a buffer later would synchronise the device
    TRY(ensure_workspace(c, m, n, blocked ? (n + nbe - 1) / nbe + 1 : 0, nch > 1));
    double* dA = c->hostA;
    double* dal = c->hostA + (size_t)ldd * n;
    cudaStream_t st = c->copy_stream;
    std::vector<Event> evUp;
    struct timespec ts0;
    clock_gettime(CLOCK_MONOTONIC, &ts0);
    auto stamp = [&](const char* what, bool sync_all) {
        if (!c->host_trace) return;
        if (sync_all) { cudaStreamSynchronize(st); }
        struct timespec ts;
        clock_gettime(CLOCK_MONOTONIC, &ts);
        fprintf(stderr, "[dhqr host] %-34s %8.2f ms\n", what, (ts.tv_sec - ts0.tv_sec) * 1e3 + (ts.tv_nsec - ts0.tv_nsec) * 1e-6);
    };
    if (c->host_trace) {
        fprintf(stderr, "[dhqr host] upload chunks (first column : join step):");
        for (int j = 0; j < nch; ++j) fprintf(stderr, " %lld:%d", (long long)B[j], join[j]);
        fprintf(stderr, "\n");
    }
    c->up_chunks.clear();
    const int rc = [&]() -> int {
        CU(cudaMemcpy2DAsync(dA, (size_t)ldd * 8, hA, (size_t)lda * 8, (size_t)m * 8, (size_t)B[1], cudaMemcpyHostToDevice, st));
        if (nch > 1) {
            // the later chunks go up one after the other BEHIND the first (concurrent uploads would share the link and delay the
            // start of the factorisation), on their own stream
            Event& e0 = evUp.emplace_back();
            CU(e0.create(cudaEventDisableTiming));
            CU(cudaEventRecord(e0, st));
            CU(cudaStreamWaitEvent(c->h2d_stream, e0, 0));
            for (int j = 1; j < nch; ++j) {
                Event& e = evUp.emplace_back();
                CU(e.create(c->host_trace ? cudaEventDefault : cudaEventDisableTiming));
                CU(cudaMemcpy2DAsync(dA + B[j] * ldd, (size_t)ldd * 8, hA + B[j] * lda, (size_t)lda * 8, (size_t)m * 8, (size_t)(B[j + 1] - B[j]),
                                     cudaMemcpyHostToDevice, c->h2d_stream));
                CU(cudaEventRecord(e, c->h2d_stream));
                c->up_chunks.push_back({B[j], B[j + 1], e, join[j]});
            }
        }
        stamp("first chunk uploaded", true);
        if (blocked) { c->mirror_host = hA; c->mirror_lda = lda; }   // finished panels stream back while later panels are factored
        TRY(dhqr_qr_f64(c, m, n, 0, n, dA, ldd, dal, nb, st));
        stamp("factored", true);
        if (!blocked) CU(cudaMemcpy2DAsync(hA, (size_t)lda * 8, dA, (size_t)ldd * 8, (size_t)m * 8, (size_t)n, cudaMemcpyDeviceToHost, st));
        CU(cudaMemcpyAsync(h_alpha, dal, (size_t)n * 8, cudaMemcpyDeviceToHost, st));
        return 0;
    }();
    // on every exit of the pipeline: nothing of it may still run (or still write to hA) when the call returns
    c->mirror_host = nullptr;
    c->up_chunks.clear();
    cudaError_t e0 = cudaStreamSynchronize(c->h2d_stream), e1 = cudaStreamSynchronize(st), e2 = cudaStreamSynchronize(c->d2h_stream);
    cudaError_t e3 = cudaSuccess;
    for (int i = 0; i < CU_STREAMS; ++i) { const cudaError_t e4 = cudaStreamSynchronize(c->cu_stream[i]); if (e3 == cudaSuccess) e3 = e4; }
    stamp("everything back on the host", false);
    c->panel_events.clear();
    if (rc) return rc;
    if (e0 != cudaSuccess) return set_err(1000 + (int)e0, "qr_host H2D: %s", cudaGetErrorString(e0));
    if (e1 != cudaSuccess) return set_err(1000 + (int)e1, "qr_host: %s", cudaGetErrorString(e1));
    if (e2 != cudaSuccess) return set_err(1000 + (int)e2, "qr_host D2H: %s", cudaGetErrorString(e2));
    if (e3 != cudaSuccess) return set_err(1000 + (int)e3, "qr_host catch-up: %s", cudaGetErrorString(e3));
    return 0;
}

int dhqr_ldiv_host_f64(dhqr_handle c, int64_t m, int64_t n, const double* hA, int64_t lda, const double* h_alpha,
                       const double* h_b, double* h_x) {
    TRY(check_common(c, m, n, 0, n, hA, lda));
    if (n > 0 && !h_alpha) return set_err(-6, "null alpha");
    if (m > 0 && !h_b) return set_err(-7, "null b");
    if (n > 0 && !h_x) return set_err(-8, "null x");
    if (c->nranks != 1) return set_err(-1, "host entry points are single-GPU");
    if (n == 0) return 0;
    CU(cudaSetDevice(c->device));
    const int64_t ldd = rup(m, 32);
    TRY(c->hostA.grow((size_t)ldd * n + (size_t)n));
    TRY(c->hostB.grow((size_t)ldd));
    double* dA = c->hostA;
    double* dal = c->hostA + (size_t)ldd * n;
    cudaStream_t st = c->copy_stream;
    CU(cudaMemcpy2DAsync(dA, (size_t)ldd * 8, hA, (size_t)lda * 8, (size_t)m * 8, (size_t)n, cudaMemcpyHostToDevice, st));
    CU(cudaMemcpyAsync(dal, h_alpha, (size_t)n * 8, cudaMemcpyHostToDevice, st));
    CU(cudaMemcpyAsync(c->hostB, h_b, (size_t)m * 8, cudaMemcpyHostToDevice, st));   // S:318: b itself is never touched
    TRY(dhqr_solve_f64(c, m, n, 0, n, dA, ldd, dal, c->hostB, ldd, 1, st));
    CU(cudaMemcpyAsync(h_x, c->hostB, (size_t)n * 8, cudaMemcpyDeviceToHost, st));     // S:320
    CU(cudaStreamSynchronize(st));
    return 0;
}

// ---- primitives ---------------------------------------------------------------------------------
int dhqr_partialdot_f64(dhqr_handle c, const double* d_a, const double* d_b, int64_t i0, int64_t i1, double* d_out,
                        void* stream) {
    if (!c) return set_err(-1, "null handle");
    if (!d_a) return set_err(-2, "null a");
    if (!d_b) return set_err(-3, "null b");
    if (i0 < 0) return set_err(-4, "i0 < 0");
    if (i1 < i0) return set_err(-5, "i1 < i0");
    if (!d_out) return set_err(-6, "null out");
    CU(cudaSetDevice(c->device));
    cudaStream_t st = (cudaStream_t)stream;
    k_partialdot<<<1, 1024, 0, st>>>(d_a, d_b, i0, i1, d_out);
    return post(c, st, "k_partialdot");
}

int dhqr_fill_uniform_f64(dhqr_handle c, uint64_t seed, int64_t i0, int64_t j0, int64_t m, int64_t n, double* dA,
                          int64_t lda, void* stream) {
    if (!c) return set_err(-1, "null handle");
    if (m < 0) return set_err(-5, "m < 0");
    if (n < 0) return set_err(-6, "n < 0");
    if (m == 0 || n == 0) return 0;
    if (!dA) return set_err(-7, "null matrix");
    if (lda < m) return set_err(-8, "lda < m");
    CU(cudaSetDevice(c->device));
    cudaStream_t st = (cudaStream_t)stream;
    dim3 grid((unsigned)std::min<int64_t>((m + 255) / 256, 1024), (unsigned)std::min<int64_t>(n, 4096));
    k_fill_uniform<<<grid, 256, 0, st>>>(seed, i0, j0, m, n, dA, lda);
    return post(c, st, "k_fill_uniform");
}

// ---- kernel-level hooks ---------------------------------------------------------------------------
int dhqr_k_block_reflector_f64(dhqr_handle c, int64_t rows, int nbp, const double* dV, int64_t ldv, int64_t row_lo,
                               int ncols, double* dC, int64_t ldc, double* d_linv_out, void* stream) {
    if (!c) return set_err(-1, "null handle");
    if (rows <= 0) return set_err(-2, "rows <= 0");
    if (nbp < 1 || nbp > 128) return set_err(-3, "nbp out of range");
    if (!dV) return set_err(-4, "null V");
    if (ldv < rows) return set_err(-5, "ldv < rows");
    if (!dC) return set_err(-8, "null C");
    CU(cudaSetDevice(c->device));
    cudaStream_t st = (cudaStream_t)stream;
    TRY(ensure_workspace(c, rows, ncols));
    const int nbk = nbp <= IB ? IB : NBMAX;
    TRY(pack_panel(c, st, dV, ldv, rows, nbp, 0, c->vpk2[0], 0, panel_geom({0, 0, nbp}, rows).vrows, nbk));
    TRY(apply_block_reflector(c, st, c->vpk2[0], c->ws[0], 0, nbk, rows, row_lo, dC, ldc, ncols));
    if (d_linv_out) CU(cudaMemcpyAsync(d_linv_out, c->ws[0].linv, sizeof(double) * (size_t)nbk * nbk, cudaMemcpyDeviceToDevice, st));
    return 0;
}

int dhqr_debug_copy_f64(dhqr_handle c, const char* which, double* d_dst, int64_t nelems, void* stream) {
    if (!c) return set_err(-1, "null handle");
    if (!which) return set_err(-2, "null name");
    if (!d_dst) return set_err(-3, "null destination");
    const double* src = nullptr;
    size_t have = 0;
    if (!strcmp(which, "wpart")) { src = c->ws[0].wpart; have = c->ws[0].wpart.size(); }
    else if (!strcmp(which, "wsum")) { src = c->ws[0].wsum; have = c->ws[0].wsum.size(); }
    else if (!strcmp(which, "ypk")) { src = c->ws[0].ypk; have = c->ws[0].ypk.size(); }
    else if (!strcmp(which, "linv")) { src = c->ws[0].linv; have = (size_t)NBMAX * NBMAX; }
    else if (!strcmp(which, "vpk")) { src = c->vpk2[0]; have = c->vpk2[0].size(); }
    else if (!strcmp(which, "wide")) { src = c->wbuf; have = c->wbuf.size(); }
    else return set_err(-2, "unknown buffer '%s'", which);
    if (nelems < 0 || (size_t)nelems > have) return set_err(-4, "nelems out of range (have %zu)", have);
    CU(cudaMemcpyAsync(d_dst, src, sizeof(double) * (size_t)nelems, cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
    return 0;
}

int dhqr_k_panel_f64(dhqr_handle c, int64_t rows, int ncols, double* dP, int64_t ldp, double* d_alpha, void* stream) {
    if (!c) return set_err(-1, "null handle");
    if (rows <= 0) return set_err(-2, "rows <= 0");
    if (ncols < 1 || ncols > IB || ncols > rows) return set_err(-3, "ncols out of range");
    if (!dP) return set_err(-4, "null panel");
    if (ldp < rows) return set_err(-5, "ldp < rows");
    if (!d_alpha) return set_err(-6, "null alpha");
    CU(cudaSetDevice(c->device));
    cudaStream_t st = (cudaStream_t)stream;
    TRY(ensure_workspace(c, rows, ncols));
    return launch_panel(c, st, c->vpk2[0], dP, ldp, rows, ncols, d_alpha, 0, 0, rup(rows, 128));
}

int dhqr_k_wide_panel_f64(dhqr_handle c, int64_t rows, double* dP, int64_t ldp, double* d_alpha, int* refused, void* stream) {
    if (!c) return set_err(-1, "null handle");
    if (rows < WP) return set_err(-2, "rows < 128");
    if (!dP) return set_err(-3, "null panel");
    if (ldp < rows) return set_err(-4, "ldp < rows");
    if (!d_alpha) return set_err(-5, "null alpha");
    if (!refused) return set_err(-6, "null result");
    CU(cudaSetDevice(c->device));
    cudaStream_t st = (cudaStream_t)stream;
    TRY(ensure_workspace(c, rows, WP));
    k_wide_reset<<<1, 32, 0, st>>>(c->wctl);
    TRY(post(c, st, "k_wide_reset"));
    const Panel p = {0, 0, WP};
    TRY(factor_outer_panel(c, st, c->vpk2[0], c->ws[0], p, rows, 0, dP, ldp, d_alpha, 0, true, c->ws[0].linv));
    WideCtl host;
    CU(cudaMemcpyAsync(&host, c->wctl, sizeof(host), cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    *refused = host.status != 0 || host.fail_step != W_NOFAIL;
    return 0;
}

}  // extern "C"
