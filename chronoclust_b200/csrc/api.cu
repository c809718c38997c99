// api.cu -- host side of the C ABI declared in include/chronoclust_b200.h: device-resident
// structure-of-arrays microcluster stores, chunk orchestration of the ordered kernels, the offline
// pipeline, import/export.  One handle = one device + one stream.  No CPU fallback anywhere: every
// numeric result is produced by the kernels in nearest.cuh / online.cuh / offline.cuh.
#include "../../include/chronoclust_b200.h"
#ifdef CCB_DEBUG
#include "debug.h"
#endif

#include <cfloat>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <functional>
#include <memory>
#include <string>
#include <utility>
#include <vector>

#include "nearest.cuh"
#include "offline.cuh"
#include "online.cuh"
#include "engine.cuh"
#include "stats.cuh"

using namespace ccb;

namespace {

thread_local std::string g_err;

const int kDPs[] = {4, 8, 12, 16, 24, 32, 40, 48, 64};
int round_dp(int D) {
    for (int v : kDPs)
        if (D <= v) return v;
    return -1;
}
#define CCB_DISPATCH_DP(dp, ...)                    \
    switch (dp) {                                   \
    case 4: { constexpr int kDP = 4; __VA_ARGS__ } break;  \
    case 8: { constexpr int kDP = 8; __VA_ARGS__ } break;  \
    case 12: { constexpr int kDP = 12; __VA_ARGS__ } break; \
    case 16: { constexpr int kDP = 16; __VA_ARGS__ } break; \
    case 24: { constexpr int kDP = 24; __VA_ARGS__ } break; \
    case 32: { constexpr int kDP = 32; __VA_ARGS__ } break; \
    case 40: { constexpr int kDP = 40; __VA_ARGS__ } break; \
    case 48: { constexpr int kDP = 48; __VA_ARGS__ } break; \
    case 64: { constexpr int kDP = 64; __VA_ARGS__ } break; \
    default: break;                                 \
    }

bool is_pow2(double k) {
    if (!(k > 0.0) || std::isinf(k)) return false;
    int e;
    return std::frexp(k, &e) == 0.5;
}

constexpr int MAX_SLABS = 148;

// ---- owners of device memory, page-locked host memory, streams, events and graphs -----------------------------------
// Move-only; the destructor releases what the owner holds.  An owner takes what a call made only when the call succeeded
// (the runtime does not promise what a failed call leaves in its output argument).  An owner converts to the raw pointer
// or handle, which is what the kernels and the runtime take.
template <typename T, auto Release>
struct Own {
    T p{};
    Own() = default;
    explicit Own(T q) : p(q) {}
    Own(Own &&o) noexcept : p(o.p) { o.p = T{}; }
    Own &operator=(Own &&o) noexcept { // (what this held goes to o and is released with it)
        std::swap(p, o.p);
        return *this;
    }
    ~Own() {
        if (p) Release(p);
    }
    operator T() const { return p; }
    T operator->() const { return p; }
};
template <typename T> using Dev = Own<T *, cudaFree>;
template <typename T> using Pinned = Own<T *, cudaFreeHost>;
using Stream = Own<cudaStream_t, cudaStreamDestroy>;
using Event = Own<cudaEvent_t, cudaEventDestroy>;

template <typename O, typename F>
cudaError_t make(O &o, F create) {
    decltype(o.p) q{};
    const cudaError_t e = create(&q);
    if (e == cudaSuccess) o = O(q);
    return e;
}
template <typename T> cudaError_t alloc(Dev<T> &o, size_t bytes) { return make(o, [=](T **q) { return cudaMalloc(q, bytes); }); }
template <typename T> cudaError_t alloc(Pinned<T> &o, size_t bytes) { return make(o, [=](T **q) { return cudaMallocHost(q, bytes); }); }
cudaError_t create(Stream &o, int prio) {
    return make(o, [=](cudaStream_t *q) { return cudaStreamCreateWithPriority(q, cudaStreamNonBlocking, prio); });
}
cudaError_t create(Event &o, unsigned flags) { return make(o, [=](cudaEvent_t *q) { return cudaEventCreateWithFlags(q, flags); }); }

// Grow-only buffer.  ensure(bytes) does nothing when the capacity suffices; a growth allocates the new memory before it
// releases the old, and a failed one keeps the old memory and capacity.  Contents are not preserved.
template <typename O>
struct Grow : O {
    size_t cap = 0;
    cudaError_t ensure(size_t bytes) {
        if (bytes <= cap) return cudaSuccess;
        O n;
        const cudaError_t e = alloc(n, bytes);
        if (e != cudaSuccess) return e;
        O::operator=(std::move(n));
        cap = bytes;
        return cudaSuccess;
    }
};

// Stream-ordered pool memory for the length of a scope: cudaMallocAsync on s, cudaFreeAsync on s when the scope ends.
struct Scratch {
    const cudaStream_t s;
    void *p = nullptr;
    explicit Scratch(cudaStream_t st) : s(st) {}
    Scratch(const Scratch &) = delete;
    ~Scratch() {
        if (p) cudaFreeAsync(p, s);
    }
    cudaError_t alloc(size_t bytes) {
        void *q;
        const cudaError_t e = cudaMallocAsync(&q, bytes, s);
        if (e == cudaSuccess) p = q;
        return e;
    }
    template <typename T> T *as() const { return static_cast<T *>(p); }
};

// the arrays of one microcluster list; Store is their view for the kernels
struct StoreMem {
    Dev<double> cf1, cf2, cen, w;
    Dev<uint64_t> mask;
    Dev<int64_t> id;
    Dev<int32_t> uid;
    Dev<double2> cw;
    int cap = 0;
    Store view() const {
        Store s;
        memset(&s, 0, sizeof s); // (Eng holds Stores and is compared with memcmp)
        s.cf1 = cf1, s.cf2 = cf2, s.cen = cen, s.w = w, s.mask = mask, s.id = id, s.uid = uid, s.cw = cw;
        s.cap = cap;
        return s;
    }
};

// what the block-speculative engine allocates once per handle: control blocks, the arrays of BsWs, kernel 1's slab lists
struct BsMem {
    Dev<BsCtl> bc;
    Pinned<BsCtl> h_bc;
    Dev<EngIo> io;
    Pinned<EngIo> h_io;
    std::vector<Dev<void>> arrays;
    double *tk_dist_slab = nullptr;
    int32_t *tk_idx_slab = nullptr;
};

struct GraphSlot { // a graph of the engine, its executable and the Eng it was captured with
    Own<cudaGraph_t, cudaGraphDestroy> graph;
    Own<cudaGraphExec_t, cudaGraphExecDestroy> exec;
    Eng eng{};
};

} // namespace

struct ccb_handle {
    ccb_params prm{};
    int D = 0, DP = 0, div_mode = 0, cnt_gt1 = 0;
    double wsel = 1.0;
    Stream stream; // first member: destroyed last, after everything that was enqueued on it
    StoreMem Pm[2], Om[2];
    Store P[2]{}, O[2]{}; // their views
    int pcur = 0, ocur = 0;
    Dev<Ctl> d_ctl;
    Pinned<Ctl> h_ctl;
    double mu = 0, omicron = 0;
    int64_t pi = 0;
    bool have_params = false;
    // ingest buffers
    Grow<Dev<double>> d_X;
    // host rows as copied (float32 ones, and the full-width rows of a column-subset ingest), before k_stage_rows gathers /
    // widens them into d_X
    Grow<Dev<unsigned char>> d_stg;
    Grow<Dev<int32_t>> d_cols; // [CCB_MAX_D] column map of a column-subset ingest
    Grow<Dev<double>> d_cof;   // [CCB_MAX_D] arcsinh cofactors of the last ingest by source column (0: linear)
    Grow<Dev<int32_t>> d_assign;
    Grow<Dev<uint8_t>> d_stage;
    Grow<Dev<int32_t>> d_pnew, d_pfin, d_onew; // kernel 3 plan codes
    // block-speculative engine (engine.cuh)
    int bs_bmax = 32768, bs_bmin = 1024, bs_iters = 3;
    BsMem bs;
    BsWs ws{}; // view of bs, ws_tiles, ws_dbg and ws_first
    Dev<void> ws_tiles[7];
    Dev<int64_t> ws_dbg;
    Dev<int32_t> ws_first;
    int ws_first_cap = 0;
    BsCtl bc_base{}; // counters folded in by ccb_reset
    bool bs_use_graph = true;   // CUDA graph with device-driven WHILE nodes (stream launches when per-kernel timing is on)
    // Two cached graphs: the double-buffered stores flip at every ccb_begin_timepoint with decay, so consecutive timepoints
    // alternate between two sets of (baked-in) pointers -- with one slot the graph was re-captured and re-instantiated at
    // every timepoint (~1 ms each).  [0] is the current slot.
    GraphSlot graphs[2];
    Stream cap[3]; // capture streams: block loop, round loop, side branch
    Event ev_fork, ev_join;
    Stream copy_stream; // host -> device segments of ccb_ingest, ahead of the engine
    Stream res_stream;  // device -> host copies of the per-cell results of a finished segment, behind the engine
    Grow<Pinned<unsigned char>> h_res; // page-locked bounce buffer of those results ([n] int32 assignments, then [n] stages)
    // [4][CCB_MAX_D] scale_ / min_ of the scaled ingest; after a column-subset ingest also scale_ / min_ by source column
    Grow<Dev<double>> d_scale;
    // where the rows and per-cell results of the last ingest live (ccb_cluster_stats): the double rows the engine read
    // (d_X or the caller's device rows) and the assignments (d_assign or the caller's device buffer) -- recorded, not copied.
    // After a column-subset ingest, the full-width rows instead (d_stg or the caller's device rows), in their own dtype.
    struct {
        const void *X = nullptr;
        int64_t ld = 0, N = 0;
        const int32_t *assign = nullptr;
        int32_t dtype = CCB_DTYPE_F64, W = 0;
        uint64_t colmask = 0; // the clustering columns of a column-subset ingest (0: none)
        bool scaled = false, valid = false;
        bool raw_tx = false; // X holds raw values of an ingest with cofactors (d_cof): ccb_cluster_stats transforms them
    } last;
    Event ev_seg[8];
    // offline results (host copies)
    int64_t off_M = 0;
    std::vector<int64_t> cl_off, cl_members;
    std::vector<double> cl_w, cl_cf1, cl_cf2, cl_cen, cl_pref;
    std::vector<int32_t> cl_label;
    // offline workspace: grow-only device buffers, kept between calls (the white-box export reads them lazily)
    enum { OB_CORE, OB_CLS, OB_NBR, OB_WNBR, OB_CNT, OB_QUEUE, OB_LABEL, OB_ORDER, OB_CLOFF, OB_NCL, OB_SUBMASK, OB_OMASK,
           OB_D1, OB_D2, OB_DC, OB_DW, OB_COUNT };
    Grow<Dev<void>> ob[OB_COUNT];
    int off_csr_min_m = 0;
    ccb_stats st{};
    ccb_stats st_base{}; // device-side counters folded in by ccb_reset
    std::string err;
    void *dnrm2 = nullptr;
    // optional per-category GPU timing (CUDA events on the handle's stream)
    bool timing = false;
    struct Ev { Event a, b; int cat; };
    std::vector<Ev> ev_pending;
    std::vector<Event> ev_pool;
    double cat_ms[CCB_NCAT] = {0};
    int64_t cat_n[CCB_NCAT] = {0};
};

namespace {

int fail(ccb_handle *h, int code, const char *fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    if (h) h->err = buf;
    g_err = buf;
    return code;
}
// A failed call stays the runtime's last error until someone reads it: CK clears it, so that the next launch check
// does not report it again.
#define CK(h, call)                                                                                        \
    do {                                                                                                   \
        cudaError_t e_ = (call);                                                                           \
        if (e_ != cudaSuccess) {                                                                           \
            cudaGetLastError();                                                                            \
            return fail(h, e_ == cudaErrorMemoryAllocation ? CCB_ENOMEM : CCB_ECUDA, "%s:%d %s: %s", __FILE__, \
                        __LINE__, #call, cudaGetErrorString(e_));                                          \
        }                                                                                                  \
    } while (0)
#define CKL(h) CK(h, cudaGetLastError())

// first call of every entry point that takes a handle
int enter(ccb_handle *h) {
    if (!h) return fail(nullptr, CCB_EINVAL, "null handle");
    CK(h, cudaSetDevice(h->prm.device));
    return CCB_OK;
}

// RAII bracket: records CUDA events around the launches of one category when timing is enabled
struct Timed {
    ccb_handle *h;
    ccb_handle::Ev e{};
    bool on;
    Timed(ccb_handle *h_, int cat) : h(h_), on(h_ && h_->timing) {
        if (!on) return;
        auto get = [&](Event &x) {
            if (h->ev_pool.empty()) {
                create(x, cudaEventDefault);
                return;
            }
            x = std::move(h->ev_pool.back());
            h->ev_pool.pop_back();
        };
        get(e.a);
        get(e.b);
        e.cat = cat;
        cudaEventRecord(e.a, h->stream);
    }
    void stop() {
        if (!on) return;
        cudaEventRecord(e.b, h->stream);
        h->ev_pending.push_back(std::move(e));
        on = false;
    }
    ~Timed() { stop(); }
};
void drain_timing(ccb_handle *h) { // call after a stream synchronize
    for (auto &e : h->ev_pending) {
        float ms = 0.f;
        if (cudaEventElapsedTime(&ms, e.a, e.b) == cudaSuccess) {
            h->cat_ms[e.cat] += ms;
            h->cat_n[e.cat] += 1;
        }
        h->ev_pool.push_back(std::move(e.a));
        h->ev_pool.push_back(std::move(e.b));
    }
    h->ev_pending.clear();
}

int alloc_store(ccb_handle *h, StoreMem &S, int cap) {
    const size_t nd = (size_t)cap * h->D + 2; // + slack for 16-byte rounded bulk copies
    CK(h, alloc(S.cf1, nd * 8));
    CK(h, alloc(S.cf2, nd * 8));
    CK(h, alloc(S.cen, nd * 8));
    CK(h, alloc(S.w, (size_t)cap * 8));
    CK(h, alloc(S.mask, (size_t)cap * 8));
    CK(h, alloc(S.id, (size_t)cap * 8));
    CK(h, alloc(S.uid, (size_t)cap * 4));
    CK(h, alloc(S.cw, (size_t)cap * h->DP * sizeof(double2)));
    S.cap = cap;
    return CCB_OK;
}
// Grows both ping-pong buffers of a list to >= want entries, preserving the first n of the current one.  Both new
// buffers are allocated and filled before the list takes them: after a failure the list keeps its old pair.
int grow_store(ccb_handle *h, bool outliers, int n, int64_t want) {
    StoreMem *S = outliers ? h->Om : h->Pm;
    const int cur = outliers ? h->ocur : h->pcur;
    if (want <= S[cur].cap) return CCB_OK;
    int64_t cap = S[cur].cap;
    while (cap < want) cap *= 2;
    if (cap > (int64_t)1 << 30) return fail(h, CCB_ELIMIT, "microcluster list would exceed 2^30 entries");
    const int D = h->D, DP = h->DP;
    StoreMem nw[2];
    int rc;
    if ((rc = alloc_store(h, nw[cur], (int)cap)) || (rc = alloc_store(h, nw[1 - cur], (int)cap))) return rc;
    const StoreMem &o = S[cur];
    StoreMem &c = nw[cur];
    cudaStream_t s = h->stream;
    CK(h, cudaMemcpyAsync(c.cf1, o.cf1, (size_t)n * D * 8, cudaMemcpyDeviceToDevice, s));
    CK(h, cudaMemcpyAsync(c.cf2, o.cf2, (size_t)n * D * 8, cudaMemcpyDeviceToDevice, s));
    CK(h, cudaMemcpyAsync(c.cen, o.cen, (size_t)n * D * 8, cudaMemcpyDeviceToDevice, s));
    CK(h, cudaMemcpyAsync(c.w, o.w, (size_t)n * 8, cudaMemcpyDeviceToDevice, s));
    CK(h, cudaMemcpyAsync(c.mask, o.mask, (size_t)n * 8, cudaMemcpyDeviceToDevice, s));
    CK(h, cudaMemcpyAsync(c.id, o.id, (size_t)n * 8, cudaMemcpyDeviceToDevice, s));
    CK(h, cudaMemcpyAsync(c.uid, o.uid, (size_t)n * 4, cudaMemcpyDeviceToDevice, s));
    CK(h, cudaMemcpyAsync(c.cw, o.cw, (size_t)n * DP * sizeof(double2), cudaMemcpyDeviceToDevice, s));
    CK(h, cudaStreamSynchronize(s));
    Store *V = outliers ? h->O : h->P;
    for (int i = 0; i < 2; ++i) {
        S[i] = std::move(nw[i]);
        V[i] = S[i].view();
    }
    return CCB_OK;
}

int sync_ctl(ccb_handle *h) { // device control block -> pinned host mirror
    CK(h, cudaMemcpyAsync(h->h_ctl, h->d_ctl, sizeof(Ctl), cudaMemcpyDeviceToHost, h->stream));
    CK(h, cudaStreamSynchronize(h->stream));
    if (h->timing) drain_timing(h);
    return CCB_OK;
}
int push_ctl(ccb_handle *h) {
    CK(h, cudaMemcpyAsync(h->d_ctl, h->h_ctl, sizeof(Ctl), cudaMemcpyHostToDevice, h->stream));
    return CCB_OK;
}

Num make_num(const ccb_handle *h) {
    Num nm{};
    nm.delta2 = h->prm.delta2;
    nm.k = h->prm.k;
    nm.wsel = h->wsel;
    nm.eps2 = h->prm.eps2;
    nm.beta_mu = h->prm.beta * h->mu; // beta * mu, hddstream.py:413, 524
    nm.pi = h->pi;
    nm.D = h->D;
    nm.DP = h->DP;
    nm.div_mode = h->div_mode;
    nm.cnt_gt1 = h->cnt_gt1;
    // the gate compares count(pref' != 1) with pi; for k == 1 that count is 0 and the gate is vacuous,
    // as it is whenever pi >= D (hddstream.py:315-321)
    nm.pi_active = (h->prm.k != 1.0) && (h->pi < (int64_t)h->D);
    return nm;
}

// Static split of kernel 1: (row groups) x (slabs of the MC axis).  Few cells: enough slabs to fill the GPU twice.
// Many cells: the slab count that balances the waves -- gx CTAs in ceil(gx / resident) waves waste the tail of the last
// one (13 % for the dense 1e6 x 4096 benchmark at one slab); a few slabs make the waves finer.
template <int kDP, int K>
void nearest_static_split(int div_mode, int64_t nrows_max, int M, int max_slabs, int &gx, int &slab_mcs, int &nslab) {
    using Cfg = NearestCfg<kDP, K>;
    gx = (int)((nrows_max + Cfg::CELLS - 1) / Cfg::CELLS);
    int want = gx > 0 ? (2 * 148 + gx - 1) / gx : 1;
    if (want > max_slabs) want = max_slabs;
    const int tiles = (M + Cfg::TM - 1) / Cfg::TM;
    if (want > tiles) want = tiles;
    if (want < 1) want = 1;
    if (gx > 148) {
        int occ = 1;
        if (div_mode) cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, k_nearest<kDP, K, true>, NEAREST_THREADS, 0);
        else cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, k_nearest<kDP, K, false>, NEAREST_THREADS, 0);
        const double resident = 148.0 * std::max(occ, 1);
        auto loss = [&](int sl) {
            const double w = (double)gx * sl / resident;
            return w <= 1.0 ? 0.0 : std::ceil(w) / w - 1.0;
        };
        int best = want;
        for (int sl = want + 1; sl <= std::min(std::min(max_slabs, tiles), want + 7) && loss(best) > 0.03; ++sl)
            if (loss(sl) < loss(best)) best = sl;
        want = best;
    }
    slab_mcs = ((tiles + want - 1) / want) * Cfg::TM;
    nslab = (M + slab_mcs - 1) / slab_mcs;
}

// kernel 1 launch over an explicit cw array
template <int K>
int launch_nearest(ccb_handle *h, cudaStream_t s, int DP, int div_mode, const double *X, const int32_t *rows,
                   const int32_t *nrows_dev, int64_t row_off, int64_t nrows_max, int64_t ld, int D, const double2 *cw,
                   int M, double *slab_dist, int32_t *slab_idx, double *out_dist, int32_t *out_idx, int max_slabs,
                   int *nslab_out, const int32_t *range_dev = nullptr, const int32_t *M_dev = nullptr) {
    int launched = 0;
    CCB_DISPATCH_DP(DP, {
        int gx, slab_mcs, nslab;
        nearest_static_split<kDP, K>(div_mode, nrows_max, M, max_slabs, gx, slab_mcs, nslab);
        dim3 grid(gx, nslab);
        double *od = nslab == 1 ? out_dist : slab_dist;
        int32_t *oi = nslab == 1 ? out_idx : slab_idx;
        if (div_mode)
            k_nearest<kDP, K, true><<<grid, NEAREST_THREADS, 0, s>>>(X, rows, nrows_dev, row_off, nrows_max, ld, D, cw,
                                                                     M, slab_mcs, od, oi, range_dev, M_dev, 0, nullptr);
        else
            k_nearest<kDP, K, false><<<grid, NEAREST_THREADS, 0, s>>>(X, rows, nrows_dev, row_off, nrows_max, ld, D, cw,
                                                                      M, slab_mcs, od, oi, range_dev, M_dev, 0, nullptr);
        launched = 1;
        if (nslab > 1) {
            k_topk_merge<K><<<(unsigned)((nrows_max + 255) / 256), 256, 0, s>>>(slab_dist, slab_idx, nrows_dev, row_off,
                                                                                nrows_max, nslab, out_dist, out_idx, range_dev);
            launched = 2;
        }
        if (nslab_out) *nslab_out = nslab;
    })
    if (!launched) return fail(h, CCB_ELIMIT, "unsupported padded dimensionality %d", DP);
    if (h) h->st.kernel_launches += launched;
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return fail(h, CCB_ECUDA, "k_nearest launch: %s", cudaGetErrorString(e));
    return CCB_OK;
}

// kernel 1 with the device-side work split (block-speculative engine): rows[range_dev[0] .. range_dev[1]) of the
// row list against the first min(M_bound, *M_dev) entries of cw; slab lists at [list position][max_slabs][K]
constexpr int NEAREST_DYN_GRID = 148 * 4;
template <int K>
int launch_nearest_dyn(ccb_handle *h, cudaStream_t s, int DP, int div_mode, const double *X, const int32_t *rows, int64_t ld,
                       int D, const double2 *cw, int M_bound, double *slab_dist, int32_t *slab_idx, double *out_dist,
                       int32_t *out_idx, int max_slabs, int rows_max, const int32_t *range_dev, const int32_t *M_dev,
                       const XRef *xref) {
    int launched = 0;
    CCB_DISPATCH_DP(DP, {
        using Cfg = NearestCfg<kDP, K>;
        if (div_mode)
            k_nearest<kDP, K, true><<<NEAREST_DYN_GRID, NEAREST_THREADS, 0, s>>>(X, rows, nullptr, 0, 0, ld, D, cw, M_bound, 0,
                                                                                 slab_dist, slab_idx, range_dev, M_dev, max_slabs, xref);
        else
            k_nearest<kDP, K, false><<<NEAREST_DYN_GRID, NEAREST_THREADS, 0, s>>>(X, rows, nullptr, 0, 0, ld, D, cw, M_bound, 0,
                                                                                  slab_dist, slab_idx, range_dev, M_dev, max_slabs, xref);
        k_topk_merge_dyn<K><<<std::min(NEAREST_DYN_GRID, (rows_max + 3) / 4), 128, 0, s>>>(
            slab_dist, slab_idx, range_dev, M_dev, M_bound, NEAREST_DYN_GRID, max_slabs, Cfg::TM, Cfg::CELLS,
            Cfg::CAN_SPLIT ? Cfg::TMS : 0, out_dist, out_idx);
        launched = 2;
    })
    if (!launched) return fail(h, CCB_ELIMIT, "unsupported padded dimensionality %d", DP);
    if (h) h->st.kernel_launches += launched;
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return fail(h, CCB_ECUDA, "k_nearest launch: %s", cudaGetErrorString(e));
    return CCB_OK;
}

// ---- block-speculative engine: workspace and block enqueue ------------------------------------------
constexpr int BS_MAX_SLABS = 256; // (k_topk_merge_dyn: a lane walks up to 8 slab lists)

// The workspace of the engine.  Each part is built aside and taken by the handle (and its view ws) only once every
// allocation of the part has succeeded.
int ensure_bs_ws(ccb_handle *h) {
    const int B = h->bs_bmax, D = h->D;
    if (!h->bs.bc) {
        CCB_DISPATCH_DP(h->DP, {
            CK(h, cudaFuncSetAttribute(k_bs_chain_p<kDP>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                       (int)ChainPCfg<kDP>::SMEM));
        })
        BsMem m;
        CK(h, alloc(m.bc, sizeof(BsCtl)));
        CK(h, cudaMemset(m.bc, 0, sizeof(BsCtl)));
        CK(h, alloc(m.h_bc, sizeof(BsCtl)));
        memset(m.h_bc, 0, sizeof(BsCtl));
        CK(h, alloc(m.io, sizeof(EngIo)));
        CK(h, alloc(m.h_io, sizeof(EngIo)));
        BsWs w = h->ws;
        w.bmax = B;
        auto arr = [&](auto *&p, size_t n) {
            Dev<void> d;
            const cudaError_t e = alloc(d, std::max<size_t>(n, 1) * sizeof(*p));
            p = static_cast<std::remove_reference_t<decltype(p)>>(d.p);
            m.arrays.push_back(std::move(d));
            return e;
        };
#define WSA(field, n) CK(h, arr(w.field, (n)))
        WSA(pcand, B); WSA(ospec, B); WSA(tkpos, B); WSA(dec, B); WSA(eff, B); WSA(newrank, B); WSA(pend, B); WSA(vpos, B); WSA(pbest, B);
        WSA(pflag, B); WSA(prej, B); WSA(upf, B);
        w.dp = h->DP;
        w.lsp = 2 * h->DP + 2;
        WSA(ver, (size_t)B * w.lsp); WSA(vcen, (size_t)B * D + 2);
        WSA(vr2, B); WSA(vmask, B);
        WSA(nrows, BS_RMAX); WSA(ncell, BS_RMAX);
        WSA(tk_dist, (size_t)BS_RMAX * BS_TOPK); WSA(tk_idx, (size_t)BS_RMAX * BS_TOPK);
        WSA(hkey, BS_RMAX + 1); WSA(hoff, BS_RMAX + 2); WSA(omem, BS_RMAX + 1); WSA(hrank, BS_RMAX + 2);
        WSA(hfirst, BS_RMAX + 1); WSA(okeys, BS_RMAX);
#undef WSA
        CK(h, arr(m.tk_dist_slab, (size_t)BS_RMAX * BS_MAX_SLABS * BS_TOPK));
        CK(h, arr(m.tk_idx_slab, (size_t)BS_RMAX * BS_MAX_SLABS * BS_TOPK));
        h->bs = std::move(m);
        h->ws = w;
    }
    // per-(tile, pcore key) tables follow the pcore capacity; the modified-flags follow the outlier capacity
    const int stride = h->P[h->pcur].cap;
    if (stride != h->ws.mp_stride) {
        const size_t n = ((size_t)B / 32 + 2) * stride;
        const size_t npl = (size_t)B + 4 * (size_t)stride + 8; // every key's segment is padded to a multiple of 4
        const size_t ds = (size_t)h->ws.lsp;
        const size_t bytes[7] = {n * 4, n * 4, ((size_t)stride + 2) * 4, ((size_t)stride + 2) * 4, npl * 4, npl * ds * 8,
                                 npl * ds * 8};
        Dev<void> t[7];
        for (int i = 0; i < 7; ++i) CK(h, alloc(t[i], bytes[i]));
        Dev<int64_t> dbg;
        if (h->ws_dbg) {
            CK(h, alloc(dbg, (size_t)stride * 8 * sizeof(int64_t)));
            CK(h, cudaMemset(dbg, 0, (size_t)stride * 8 * sizeof(int64_t)));
        }
        std::swap(h->ws_tiles, t);
        h->ws_dbg = std::move(dbg);
        h->ws.tilecnt = (int32_t *)h->ws_tiles[0].p;
        h->ws.tbase = (int32_t *)h->ws_tiles[1].p;
        h->ws.poff = (int32_t *)h->ws_tiles[2].p;
        h->ws.pcnt = (int32_t *)h->ws_tiles[3].p;
        h->ws.plist = (int32_t *)h->ws_tiles[4].p;
        h->ws.xg = (double *)h->ws_tiles[5].p;
        h->ws.verp = (double *)h->ws_tiles[6].p;
        h->ws.dbg = h->ws_dbg;
        h->ws.mp_stride = stride;
    }
    const int ocap = h->O[h->ocur].cap;
    if (ocap != h->ws_first_cap) {
        Dev<int32_t> f;
        CK(h, alloc(f, (size_t)ocap * 4));
        CK(h, cudaMemsetAsync(f, 0x7f, (size_t)ocap * 4, h->stream)); // 0x7f7f7f7f: "not modified"
        h->ws_first = std::move(f);
        h->ws_first_cap = ocap;
        h->ws.firstmember = h->ws_first;
    }
    return CCB_OK;
}

int sync_bc(ccb_handle *h) { // both control blocks -> pinned host mirrors
    CK(h, cudaMemcpyAsync(h->h_ctl, h->d_ctl, sizeof(Ctl), cudaMemcpyDeviceToHost, h->stream));
    CK(h, cudaMemcpyAsync(h->bs.h_bc, h->bs.bc, sizeof(BsCtl), cudaMemcpyDeviceToHost, h->stream));
    CK(h, cudaStreamSynchronize(h->stream));
    if (h->timing) drain_timing(h);
    return CCB_OK;
}

// One block = prologue + refinement rounds + commit.  Every kernel reads its work description from the device-side
// control block, so a converged (or finished) block turns the remaining launches into no-ops.  The three pieces are
// launched either on the handle's stream (bs_iters rounds enqueued per block; used when per-kernel timing is on) or
// captured once into a CUDA graph whose block loop and round loop are WHILE conditional nodes driven from the
// device (k_bs_begin / k_bs_decide / k_bs_commit call cudaGraphSetConditional): no idle launches, no host round trip.
// Kernel launch without attributes.  The kernels start with CCB_PDL() (common.cuh), but the host no longer sets the
// programmatic-stream-serialization attribute: programmatic dependent launch was measured neutral on the B200 (DESIGN.md
// §6: the gaps between the kernels of a round are not launch latency), so both of its instructions are no-ops.
template <typename... KA, typename... A>
cudaError_t launch_k(void (*k)(KA...), dim3 g, dim3 b, size_t smem, cudaStream_t s, A &&...a) {
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = g;
    cfg.blockDim = b;
    cfg.dynamicSmemBytes = smem;
    cfg.stream = s;
    return cudaLaunchKernelEx(&cfg, k, KA(std::forward<A>(a))...);
}

int launch_prologue(ccb_handle *h, const Eng &e, cudaStream_t s) {
    const int g_cells = (h->bs_bmax + BS_THREADS - 1) / BS_THREADS;
    Timed tm(h, CCB_CAT_SPEC);
    k_bs_begin<<<1, 1, 0, s>>>(e);
    CCB_DISPATCH_DP(h->DP, { launch_k(k_bs_spec<kDP>, g_cells * BS_SPLIT, BS_THREADS, 0, s, e); })
    CKL(h);
    return CCB_OK;
}

// side != nullptr (graph capture): kernel 1 + the speculated outlier decisions run on a side branch next to the
// candidate lists + pcore replay (they touch disjoint data; see the dependency notes in DESIGN.md) and join before
// k_bs_olist.
int launch_round(ccb_handle *h, const Eng &e, cudaStream_t s, int mp_grid, int mo_bound, cudaStream_t side = nullptr) {
    const int B = h->bs_bmax;
    const int g_cells = (B + BS_THREADS - 1) / BS_THREADS;
    const int g_tiles = (B / 32 + 1 + 3) / 4;
    int rc;
    cudaStream_t sa = side ? side : s;
    if (side) {
        CK(h, cudaEventRecord(h->ev_fork, s));
        CK(h, cudaStreamWaitEvent(side, h->ev_fork, 0));
    }
    {
        Timed tm(h, CCB_CAT_NEAREST);
        if ((rc = launch_nearest_dyn<BS_TOPK>(nullptr, sa, h->DP, h->div_mode, e.X, e.ws.nrows, e.ld, h->D, e.O.cw, mo_bound,
                                              h->bs.tk_dist_slab, h->bs.tk_idx_slab, e.ws.tk_dist, e.ws.tk_idx,
                                              BS_MAX_SLABS, BS_RMAX, &e.bc->tk_lo, &e.bc->Mo0,
                                              reinterpret_cast<const XRef *>(e.io))))
            return fail(h, rc, "%s", ccb_last_error(nullptr));
    }
    {
        Timed tm(h, CCB_CAT_SPEC);
        launch_k(k_bs_spec_o, BS_RMAX / BS_THREADS, BS_THREADS, 0, sa, e);
    }
    {
        Timed tm(h, CCB_CAT_LISTS);
        launch_k(k_bs_tilecnt, g_tiles, BS_THREADS, 0, s, e);
        launch_k(k_bs_pscan, std::max(mp_grid, 1), BS_CTA1, 0, s, e);
        launch_k(k_bs_pscatter, B / 32 + 1, BS_THREADS, 0, s, e);
    }
    {
        Timed tm(h, CCB_CAT_PCORE);
        CCB_DISPATCH_DP(h->DP, { launch_k(k_bs_chain_p<kDP>, std::max(mp_grid, 1), BS_CHAINP_THREADS, ChainPCfg<kDP>::SMEM, s, e); })
    }
    if (side) { // join: k_bs_olist needs the speculated outlier decisions, everything below the pcore replay
        CK(h, cudaEventRecord(h->ev_join, side));
        CK(h, cudaStreamWaitEvent(s, h->ev_join, 0));
        // second fork: pcore side of derive + verify next to the outlier-side lists / replay / derive (disjoint cells)
        CK(h, cudaEventRecord(h->ev_fork, s));
        CK(h, cudaStreamWaitEvent(side, h->ev_fork, 0));
    }
    {
        Timed tm(h, CCB_CAT_DERIVE);
        launch_k(k_bs_derive_p, g_cells, BS_THREADS, 0, sa, e);
    }
    {
        Timed tm(h, CCB_CAT_RESOLVE);
        CCB_DISPATCH_DP(h->DP, { launch_k(k_bs_verify_p<kDP>, B / 32 + 1, BS_VP_THREADS, 0, sa, e); })
    }
    {
        Timed tm(h, CCB_CAT_OLIST);
        launch_k(k_bs_olist, BS_OL_CTAS, BS_OL_THREADS, 0, s, e);
    }
    {
        Timed tm(h, CCB_CAT_CHAIN_O);
        CCB_DISPATCH_DP(h->DP, { launch_k(k_bs_chain_o<kDP>, 148 * 4, BS_THREADS, 0, s, e); }) // CTAs loop over the keys
    }
    {
        Timed tm(h, CCB_CAT_DERIVE);
        launch_k(k_bs_derive_o, BS_RMAX / BS_THREADS, BS_THREADS, 0, s, e);
    }
    if (side) {
        CK(h, cudaEventRecord(h->ev_join, side));
        CK(h, cudaStreamWaitEvent(s, h->ev_join, 0));
    }
    {
        Timed tm(h, CCB_CAT_RESOLVE);
        CCB_DISPATCH_DP(h->DP, { launch_k(k_bs_verify_o<kDP>, 148 * 4, BS_THREADS, 0, s, e); })
    }
    {
        Timed tm(h, CCB_CAT_DECIDE);
        launch_k(k_bs_decide, 1, BS_CTA1, 0, s, e);
    }
    CKL(h);
    return CCB_OK;
}
constexpr int BS_LAUNCHES_PROLOGUE = 2, BS_LAUNCHES_ROUND = 14, BS_LAUNCHES_COMMIT = 1;

int launch_commit(ccb_handle *h, const Eng &e, cudaStream_t s, int mp_grid) {
    const int g_cells = (h->bs_bmax + BS_THREADS - 1) / BS_THREADS;
    const int rows_ctas = (mp_grid + BS_RMAX + 3) / 4;
    Timed tm(h, CCB_CAT_COMMIT);
    launch_k(k_bs_commit, rows_ctas + g_cells, BS_THREADS, 0, s, e, rows_ctas); // rows | cells | (last CTA) finish
    CKL(h);
    return CCB_OK;
}

Eng make_eng(ccb_handle *h) {
    Eng e{};
    e.P = h->P[h->pcur];
    e.O = h->O[h->ocur];
    e.ctl = h->d_ctl;
    e.bc = h->bs.bc;
    e.ws = h->ws;
    return e;
}

// ---- CUDA graph of the whole ordered loop: WHILE(block) { prologue; WHILE(round) { round }; commit } ----------
// Builds into the current slot, which changes only when the build succeeds.  A failed build ends the captures it opened.
int build_graph(ccb_handle *h, const Eng &base) {
    if (!h->cap[0]) {
        // the main line of a round (lists, replay, outlier-side lists ...) is the critical path: its kernels are captured
        // from high-priority streams, the side branches (kernel 1, pcore-side derive / verify) from a low-priority one, so
        // that a small critical kernel is not queued behind the thousand CTAs of a side kernel running next to it
        int prio_lo = 0, prio_hi = 0;
        CK(h, cudaDeviceGetStreamPriorityRange(&prio_lo, &prio_hi));
        Stream c[3];
        Event fork, join;
        CK(h, create(c[0], prio_hi));
        CK(h, create(c[1], prio_hi));
        CK(h, create(c[2], prio_lo));
        CK(h, create(fork, cudaEventDisableTiming));
        CK(h, create(join, cudaEventDisableTiming));
        std::swap(h->cap, c);
        h->ev_fork = std::move(fork);
        h->ev_join = std::move(join);
    }
    GraphSlot g;
    struct Capture { // ends the capture of s if the build leaves it open
        cudaStream_t s = nullptr;
        ~Capture() {
            cudaGraph_t body;
            if (s && cudaStreamEndCapture(s, &body) != cudaSuccess) cudaGetLastError();
        }
    } c1, c2;
    Eng e = base;
    e.io = h->bs.io;
    CK(h, make(g.graph, [](cudaGraph_t *q) { return cudaGraphCreate(q, 0); }));
    cudaGraphConditionalHandle ho, hi;
    CK(h, cudaGraphConditionalHandleCreate(&ho, g.graph, 1, cudaGraphCondAssignDefault));
    CK(h, cudaGraphConditionalHandleCreate(&hi, g.graph, 0, cudaGraphCondAssignDefault));
    e.h_outer = ho;
    e.h_inner = hi;
    cudaGraphNodeParams po = {};
    po.type = cudaGraphNodeTypeConditional;
    po.conditional.handle = ho;
    po.conditional.type = cudaGraphCondTypeWhile;
    po.conditional.size = 1;
    cudaGraphNode_t outer;
    CK(h, cudaGraphAddNode(&outer, g.graph, nullptr, 0, &po));
    cudaGraph_t body_o = po.conditional.phGraph_out[0];
    const int mp_grid = e.P.cap, mo_bound = e.O.cap;
    int rc;
    CK(h, cudaStreamBeginCaptureToGraph(h->cap[0], body_o, nullptr, nullptr, 0, cudaStreamCaptureModeRelaxed));
    c1.s = h->cap[0];
    if ((rc = launch_prologue(h, e, h->cap[0]))) return rc;
    {
        cudaStreamCaptureStatus st;
        cudaGraph_t cg = nullptr;
        const cudaGraphNode_t *deps = nullptr;
        size_t ndeps = 0;
        CK(h, cudaStreamGetCaptureInfo(h->cap[0], &st, nullptr, &cg, &deps, &ndeps));
        cudaGraphNodeParams pi = {};
        pi.type = cudaGraphNodeTypeConditional;
        pi.conditional.handle = hi;
        pi.conditional.type = cudaGraphCondTypeWhile;
        pi.conditional.size = 1;
        cudaGraphNode_t inner;
        CK(h, cudaGraphAddNode(&inner, cg, deps, ndeps, &pi));
        CK(h, cudaStreamUpdateCaptureDependencies(h->cap[0], &inner, 1, cudaStreamSetCaptureDependencies));
        cudaGraph_t body_i = pi.conditional.phGraph_out[0];
        CK(h, cudaStreamBeginCaptureToGraph(h->cap[1], body_i, nullptr, nullptr, 0, cudaStreamCaptureModeRelaxed));
        c2.s = h->cap[1];
        if ((rc = launch_round(h, e, h->cap[1], mp_grid, mo_bound, h->cap[2]))) return rc;
        c2.s = nullptr;
        CK(h, cudaStreamEndCapture(h->cap[1], nullptr));
    }
    if ((rc = launch_commit(h, e, h->cap[0], mp_grid))) return rc;
    c1.s = nullptr;
    CK(h, cudaStreamEndCapture(h->cap[0], nullptr));
    CK(h, make(g.exec, [&](cudaGraphExec_t *q) { return cudaGraphInstantiate(q, g.graph, 0); }));
    g.eng = base;
    h->graphs[0] = std::move(g);
    return CCB_OK;
}

int ensure_bsv_capacity(ccb_handle *h, int blocks_ahead) {
    int rc;
    const Ctl &c = *h->h_ctl;
    const int64_t need_o = (int64_t)c.n_outlier + (int64_t)(blocks_ahead + 1) * BS_RMAX + 1;
    if ((rc = grow_store(h, true, c.n_outlier, need_o)) ||
        (rc = grow_store(h, false, c.n_pcore, c.n_pcore + blocks_ahead + 1)))
        return rc;
    return ensure_bs_ws(h);
}

// the ordered loop over cells [0, N) of a device-resident X, block-speculative engine
int ingest_core_bsv(ccb_handle *h, const double *dX, int64_t N, int64_t ld, int32_t *d_assign, uint8_t *d_stage,
                    const std::function<int()> *after_first_launch = nullptr) {
    if (!h->have_params) return fail(h, CCB_ESTATE, "ccb_begin_timepoint must precede ccb_ingest");
    if (N >= ((int64_t)1 << 31)) return fail(h, CCB_ELIMIT, "more than 2^31 - 1 cells in one call");
    cudaStream_t s = h->stream;
    int rc;
    if ((rc = ensure_bs_ws(h))) return rc;
    const bool graph = h->bs_use_graph && !h->timing;
    const int bmax = h->bs_bmax, bmin = std::min(h->bs_bmin, h->bs_bmax);
    const int itmax = graph ? (h->prm.bsv_iters > 0 ? h->bs_iters : 8) : h->bs_iters;
    k_bs_init<<<1, 1, 0, s>>>(h->bs.bc, N, itmax, bmin, bmax);
    CKL(h);
    h->st.kernel_launches++;
    if ((rc = sync_bc(h))) return rc;
    EngIo io{};
    io.X = dX;
    io.ld = ld;
    io.assign = d_assign;
    io.stage = d_stage;
    // SAFE / CONTESTED split of the speculation -- a heuristic that never affects results, only how much of the replay
    // takes the exact in-chain radius test and how often verification sends a block into another round.  SAFE = the
    // snapshot says "absorbed" (radius^2 of the tentative MC <= eps^2) and the cell is not far out (snapshot distance
    // <= 4 eps^2).  Established MCs sit right at their radius limit, so a margin below eps^2 marks almost every cell
    // CONTESTED (profiles/r1p_safe_rule_experiment.md: 10x slower); the distance bound singles out the ~1 % background
    // cells, which are exactly the ones whose radius test is open.  Speculative rejection of far cells did not pay
    // either (profiles/r1t_speculative_reject_experiment.md), nor did calling every cell SAFE whose tentative MC keeps a
    // margin below eps^2 whatever its distance (profiles/r2h_slack_rule_experiment.md): every CONTESTED cell takes the
    // exact in-chain test.  The distance bound is flat between 2 and 8 eps^2 (profiles/r2l_theta_experiment.md).
    io.theta = 4.0 * h->prm.eps2;
    io.r2safe = h->prm.eps2;
    io.r2rej = HUGE_VAL;
    io.nm = make_num(h);
    if (graph) {
        *h->bs.h_io = io;
        CK(h, cudaMemcpyAsync(h->bs.io, h->bs.h_io, sizeof(EngIo), cudaMemcpyHostToDevice, s));
    }
    int guard = 0;
    while (!h->bs.h_bc->done) {
        const BsCtl &b = *h->bs.h_bc;
        const int64_t left = N - b.pos;
        // blocks to enqueue before the next look at the control block (stream launches); the graph runs until the
        // input is consumed or a store is full, so give it room for a good stretch of blocks
        int G = (int)std::min<int64_t>(16, (left + std::max(b.next_B, 1) - 1) / std::max(b.next_B, 1) + 1);
        if (G < 1) G = 1;
        if ((rc = ensure_bsv_capacity(h, graph ? 32 : G))) return rc;
        if (b.need_grow) {
            h->bs.h_bc->need_grow = 0;
            CK(h, cudaMemcpyAsync(&h->bs.bc->need_grow, &h->bs.h_bc->need_grow, sizeof(int32_t), cudaMemcpyHostToDevice, s));
        }
        Eng e = make_eng(h);
        const int64_t pos0 = b.pos;
        const int64_t blocks0 = b.blocks, iters0 = b.iters;
        if (graph) {
            GraphSlot *g = h->graphs;
            if (!g[0].exec || memcmp(&g[0].eng, &e, sizeof(Eng)) != 0) {
                // not the current slot: the other one? (swap); otherwise rebuild the older slot
                std::swap(g[0], g[1]);
                if ((!g[0].exec || memcmp(&g[0].eng, &e, sizeof(Eng)) != 0) && (rc = build_graph(h, e))) return rc;
            }
            CK(h, cudaGraphLaunch(g[0].exec, s));
        } else {
            const Ctl &c = *h->h_ctl;
            e.X = io.X, e.ld = io.ld, e.assign = io.assign, e.stage = io.stage, e.theta = io.theta, e.r2safe = io.r2safe, e.r2rej = io.r2rej, e.nm = io.nm;
            for (int g = 0; g < G; ++g) {
                const int mp_grid = c.n_pcore + g + 1;
                const int mo_bound = (int)std::min<int64_t>(c.n_outlier + (int64_t)(g + 1) * BS_RMAX, h->O[h->ocur].cap);
                if ((rc = launch_prologue(h, e, s))) return rc;
                for (int it = 0; it < h->bs_iters; ++it)
                    if ((rc = launch_round(h, e, s, mp_grid, mo_bound))) return rc;
                if ((rc = launch_commit(h, e, s, mp_grid))) return rc;
                h->st.kernel_launches += BS_LAUNCHES_PROLOGUE + h->bs_iters * BS_LAUNCHES_ROUND + BS_LAUNCHES_COMMIT;
            }
        }
        if (after_first_launch) { // the engine is running: the caller queues the next input segment behind it
            const std::function<int()> *f = after_first_launch;
            after_first_launch = nullptr;
            if ((rc = (*f)())) return rc;
        }
        if ((rc = sync_bc(h))) return rc;
        if (graph) // kernels the graph executed: per block prologue + commit, per round the round's kernels
            h->st.kernel_launches += (h->bs.h_bc->blocks - blocks0) * (BS_LAUNCHES_PROLOGUE + BS_LAUNCHES_COMMIT) +
                                     (h->bs.h_bc->iters - iters0) * BS_LAUNCHES_ROUND + BS_LAUNCHES_PROLOGUE;
        if (h->bs.h_bc->pos == pos0 && !h->bs.h_bc->need_grow && !h->bs.h_bc->done && ++guard > 4)
            return fail(h, CCB_ESTATE, "internal: block-speculative engine made no progress at row %lld", (long long)pos0);
        if (h->bs.h_bc->pos != pos0) guard = 0;
    }
    if (after_first_launch && (rc = (*after_first_launch)())) return rc;
    h->st.points += N;
    return CCB_OK;
}

double builtin_nrm2(const double *x, int n) {
    // restatement of OpenBLAS' x86-64 dnrm2: squares, sum and square root in x87 extended precision
    long double s = 0.0L;
    for (int i = 0; i < n; ++i) s += (long double)x[i] * (long double)x[i];
    return (double)sqrtl(s);
}

// grow-only buffer of the handle's offline workspace (contents are NOT preserved across a growth)
int off_buf(ccb_handle *h, int which, size_t bytes) {
    Grow<Dev<void>> &b = h->ob[which];
    bytes = std::max<size_t>(bytes, 16);
    if (bytes <= b.cap) return CCB_OK;
    CK(h, cudaStreamSynchronize(h->stream));
    size_t cap = 256;
    while (cap < bytes) cap *= 2;
    CK(h, b.ensure(cap));
    return CCB_OK;
}

// status of the launches just made (h may be NULL: the stateless entry points)
int launched(ccb_handle *h, const char *what) {
    const cudaError_t e = cudaGetLastError();
    return e == cudaSuccess ? CCB_OK : fail(h, CCB_ECUDA, "%s: %s", what, cudaGetErrorString(e));
}

// ---- the launchers of the offline stages, shared by ccb_offline and the stateless ccb_off_* entry points -------------
// Rows [r0, r1) of M; the row-indexed outputs (nbr, cnt, submask, wnbr, iso, nnz) hold the rows from r0 on.

int launch_off_neighbours(ccb_handle *h, cudaStream_t s, const double *cen, int M, int D, int r0, int r1, double E2,
                          uint32_t *nbr, int32_t *cnt, int32_t *border, int border_cap, int32_t *n_border) {
    const int DP = round_dp(D);
    int ok = 0;
    if (r1 > r0) CK(h, cudaMemsetAsync(cnt, 0, (size_t)(r1 - r0) * sizeof(int32_t), s));
    CCB_DISPATCH_DP(DP, {
        // rows x column slabs: at least ~4 waves of CTAs on 148 SMs so that the tail does not dominate
        const int gx = (r1 - r0 + OffCfg<kDP>::ROWS - 1) / OffCfg<kDP>::ROWS;
        const int ntiles = (M + OffCfg<kDP>::TM - 1) / OffCfg<kDP>::TM;
        int gy = gx > 0 ? std::max(1, std::min(ntiles, (148 * 2 * 4 + gx - 1) / gx)) : 1;
        if (gx > 0) { // ... and a slab count whose last wave is full (391 x 4 CTAs on 296 slots were 5.28 waves)
            int occ = 1;
            cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, k_off_neighbours<kDP>, OFFN_THREADS, 0);
            const double resident = 148.0 * std::max(occ, 1);
            auto loss = [&](int sl) {
                const double w = (double)gx * sl / resident;
                return w <= 1.0 ? 0.0 : std::ceil(w) / w - 1.0;
            };
            int best = gy;
            for (int sl = gy + 1; sl <= std::min(ntiles, gy + 7) && loss(best) > 0.03; ++sl)
                if (loss(sl) < loss(best)) best = sl;
            gy = best;
        }
        if (gx > 0)
            k_off_neighbours<kDP><<<dim3(gx, gy), OFFN_THREADS, 0, s>>>(cen, M, D, r0, r1, E2, nbr, cnt, border, border_cap,
                                                                          n_border);
        ok = 1;
    })
    if (!ok) return fail(h, CCB_ELIMIT, "unsupported dimensionality %d", D);
    return launched(h, "k_off_neighbours launch");
}

// Kernel 4b with its borderline pairs settled: the pairs whose squared distance lies inside the guard band are decided on
// the host with the BLAS dnrm2 the reference itself calls (NULL: builtin_nrm2), `<= E` inclusive, and patched into nbr /
// cnt.  The pair list is scratch from the stream-ordered pool and grows to whatever the data needs (e.g. many coincident
// centroids with upsilon = 0).  Synchronises s once, and once more when pairs exist.  *n_border = the number of pairs.
int off_neighbours_settled(ccb_handle *h, cudaStream_t s, const double *cen, int M, int D, int r0, int r1, double E,
                           double E2, void *dnrm2, uint32_t *nbr, int32_t *cnt, int64_t *n_border) {
    int32_t nb = 0;
    int rc;
    for (int cap = 1 << 16;; cap = nb) {
        Scratch sc(s); // [0] pair count | [1, 1 + 2 cap) pairs (row, col) | cap bytes of decisions
        CK(h, sc.alloc(4 + (size_t)cap * 9));
        int32_t *buf = sc.as<int32_t>();
        CK(h, cudaMemsetAsync(buf, 0, 4, s));
        if ((rc = launch_off_neighbours(h, s, cen, M, D, r0, r1, E2, nbr, cnt, buf + 1, cap, buf))) return rc;
        if (h) h->st.kernel_launches++;
        CK(h, cudaMemcpyAsync(&nb, buf, 4, cudaMemcpyDeviceToHost, s));
        CK(h, cudaStreamSynchronize(s));
        if (nb > cap) continue; // again with a list that holds every pair
        *n_border = nb;
        if (nb == 0) return CCB_OK;
        std::vector<int32_t> pairs(2 * (size_t)nb);
        std::vector<double> hc((size_t)M * D), x(D);
        std::vector<uint8_t> dec(nb);
        CK(h, cudaMemcpy(pairs.data(), buf + 1, pairs.size() * 4, cudaMemcpyDeviceToHost));
        CK(h, cudaMemcpy(hc.data(), cen, hc.size() * 8, cudaMemcpyDeviceToHost));
        typedef double (*nrm2_fn)(int *, double *, int *);
        for (int i = 0; i < nb; ++i) {
            const int p_ = pairs[2 * i], q_ = pairs[2 * i + 1];
            for (int d = 0; d < D; ++d) x[d] = hc[(size_t)q_ * D + d] - hc[(size_t)p_ * D + d];
            int n = D, inc = 1;
            const double r = dnrm2 ? ((nrm2_fn)dnrm2)(&n, x.data(), &inc) : builtin_nrm2(x.data(), D);
            dec[i] = r <= E;
        }
        uint8_t *ddec = reinterpret_cast<uint8_t *>(buf + 1 + 2 * (size_t)nb);
        CK(h, cudaMemcpyAsync(ddec, dec.data(), nb, cudaMemcpyHostToDevice, s));
        k_off_patch<<<(nb + 127) / 128, 128, 0, s>>>(nbr, cnt, buf + 1, ddec, nb, r0, (M + 31) / 32);
        if ((rc = launched(h, "k_off_patch"))) return rc;
        if (h) h->st.kernel_launches++;
        CK(h, cudaStreamSynchronize(s)); // dec (host) is read by the copy above
        return CCB_OK;
    }
}

int launch_off_subspace(ccb_handle *h, cudaStream_t s, const double *cen, int M, int D, int r0, int r1, const uint32_t *nbr,
                        const int32_t *cnt, double delta, uint64_t *submask) {
    if (r1 == r0) return CCB_OK;
    CK(h, cudaMemsetAsync(submask, 0, (size_t)(r1 - r0) * 8, s));
    const int64_t t = (int64_t)(r1 - r0) * D;
    k_off_subspace<<<(unsigned)((t + 127) / 128), 128, 0, s>>>(cen, M, D, r0, r1, nbr, cnt, delta, submask);
    return launched(h, "k_off_subspace");
}

int launch_off_weighted(ccb_handle *h, cudaStream_t s, const double *cen, int M, int D, int r0, int r1, const uint32_t *nbr,
                        const uint64_t *submask_all, double k, double E2, uint32_t *wnbr) {
    if (r1 == r0) return CCB_OK;
    k_off_weighted<<<(unsigned)((r1 - r0 + 3) / 4), OFFW_THREADS, 0, s>>>(cen, M, D, r0, r1, nbr, submask_all, k, E2, wnbr);
    return launched(h, "k_off_weighted");
}

int launch_offc_rowinfo(ccb_handle *h, cudaStream_t s, const uint32_t *wnbr, int M, int r0, int r1, uint8_t *iso,
                        int32_t *nnz) {
    if (r1 > r0) k_offc_rowinfo<<<(unsigned)((r1 - r0 + 3) / 4), 128, 0, s>>>(wnbr, r0, r1, (M + 31) / 32, iso, nnz);
    return launched(h, "k_offc_rowinfo");
}

// iso / off: of all M rows (global CSR)
int launch_offc_fill(ccb_handle *h, cudaStream_t s, const uint32_t *wnbr, int M, int r0, int r1, const uint8_t *iso,
                     const int64_t *off, int32_t *col) {
    if (r1 > r0) k_offc_fill<<<(unsigned)((r1 - r0 + 3) / 4), 128, 0, s>>>(wnbr, r0, r1, (M + 31) / 32, iso, off, col);
    return launched(h, "k_offc_fill");
}

// The stateless entry points take their scratch from the device's stream-ordered pool; raise its release threshold once
// so that it keeps what it has instead of handing the memory back to the driver at every synchronisation.
void tune_pool(int device) {
    static bool done[64] = {false};
    if (device < 0 || device >= 64 || done[device]) return;
    cudaMemPool_t pool;
    if (cudaDeviceGetDefaultMemPool(&pool, device) == cudaSuccess) {
        uint64_t keep = UINT64_MAX;
        cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &keep);
    }
    done[device] = true;
}

// first call of every stateless entry point
int enter_device(int device) {
    CK(nullptr, cudaSetDevice(device));
    tune_pool(device);
    return CCB_OK;
}

// kernel 4e: ordered cluster growth.  Small M (the online hot path: tens of pcore MCs): the single-launch bit-row
// kernel.  Large M (config C4): isolated MCs in parallel, CSR lists for the rest, clusters merged by seed rank
// (offline.cuh).  Both produce identical label / order / cl_off / n_cl.  cls [M] and queue [2M + 2] are scratch.
constexpr int OFF_CSR_MIN_M = 2048; // default switch-over; ccb_params.off_csr_min_m / the csr_min_m argument move it

// The ordered growth over a CSR of the weighted neighbourhoods and the merge with the isolated microclusters' clusters by
// seed rank (offline.cuh).  i32: scratch of 7 M + 16 int32; cls [M] zeroed; queue [2 M + 2].
void offc_grow_and_merge(cudaStream_t s, int M, const int64_t *off, const int32_t *col, const uint8_t *core, const uint8_t *iso,
                         const uint64_t *submask, int cnt_gt1, int64_t pi, uint8_t *cls, int32_t *queue, int32_t *i32,
                         int32_t *label, int32_t *order, int32_t *cl_off, int32_t *n_cl, int64_t total_nnz) {
    const size_t m = (size_t)M;
    int32_t *order_s = i32, *cl_off_s = order_s + m, *seed_of = cl_off_s + m + 1, *n_cl_s = seed_of + m + 1,
            *seedflag = n_cl_s + 1, *size_by_node = seedflag + m, *rank = size_by_node + m, *size_by_cluster = rank + m + 1;
    const int tgrid = (M + 255) / 256;
    // short lists (a sparse graph): one warp over the compacted non-isolated microclusters, no block barriers; long lists:
    // the 1024-thread walk.  total_nnz < 0 = unknown.  (cand / its flags / ranks live in buffers the later kernels rewrite.)
    if (total_nnz >= 0 && total_nnz <= (int64_t)M * 16) {
        int32_t *candflag = seedflag, *candrank = rank, *cand = size_by_node;
        k_offc_candflag<<<tgrid, 256, 0, s>>>(M, iso, candflag);
        k_offc_scan<int32_t><<<1, OFFG_THREADS, 0, s>>>(candflag, M, candrank);
        k_offc_candscatter<<<tgrid, 256, 0, s>>>(M, candflag, candrank, cand);
        // (a non-isolated microcluster owns >= 1 CSR entry, so total_nnz bounds the number of candidates, too)
        const size_t smem = (size_t)total_nnz * 22 + 64;
        if (smem <= 200 * 1024) { // the whole non-isolated graph fits one CTA's shared memory: walk it there
            cudaFuncSetAttribute(k_offc_grow_smem, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
            k_offc_grow_smem<<<1, 1024, smem, s>>>(cand, candrank, M, off, col, core, submask, cnt_gt1, pi, order_s, cl_off_s,
                                                   seed_of, n_cl_s, (int)total_nnz + 1, (int)total_nnz + 1);
        } else {
            k_offc_grow_warp<<<1, 32, 0, s>>>(cand, candrank + M, off, col, core, submask, cnt_gt1, pi, cls, queue, order_s,
                                              cl_off_s, seed_of, n_cl_s);
        }
    } else {
        k_offc_grow<<<1, OFFG_THREADS, 0, s>>>(M, off, col, core, iso, submask, cnt_gt1, pi, cls, queue, order_s, cl_off_s,
                                               seed_of, n_cl_s);
    }
    k_offc_seeds<<<tgrid, 256, 0, s>>>(M, iso, core, submask, cnt_gt1, pi, seed_of, cl_off_s, n_cl_s, seedflag, size_by_node,
                                       label);
    k_offc_seeds_serial<<<tgrid, 256, 0, s>>>(seed_of, cl_off_s, n_cl_s, seedflag, size_by_node);
    k_offc_scan<int32_t><<<1, OFFG_THREADS, 0, s>>>(seedflag, M, rank);
    cudaMemsetAsync(size_by_cluster, 0, m * 4, s);
    k_offc_sizes<<<tgrid, 256, 0, s>>>(M, seedflag, rank, size_by_node, size_by_cluster, n_cl);
    k_offc_scan<int32_t><<<1, OFFG_THREADS, 0, s>>>(size_by_cluster, M, cl_off);
    k_offc_scatter_iso<<<tgrid, 256, 0, s>>>(M, iso, seedflag, rank, size_by_node, cl_off, order, label);
    k_offc_scatter_serial<<<148, 256, 0, s>>>(seed_of, cl_off_s, n_cl_s, order_s, rank, cl_off, order, label);
}

// off[M] -- the CSR size, the last entry of the exclusive prefix of the row lengths -- read back to the host
int csr_total(ccb_handle *h, cudaStream_t s, const int64_t *off, int M, int64_t *total) {
    CK(h, cudaMemcpyAsync(total, off + M, 8, cudaMemcpyDeviceToHost, s));
    CK(h, cudaStreamSynchronize(s));
    return CCB_OK;
}

// offc_grow_and_merge over a CSR of `total` entries (iso / off / col of all M rows), its scratch from the stream-ordered pool
int off_clusters_csr(ccb_handle *h, cudaStream_t s, int M, const int64_t *off, const int32_t *col, int64_t total,
                     const uint8_t *iso, const uint8_t *core, const uint64_t *submask, int cnt_gt1, int64_t pi,
                     int32_t *label, int32_t *order, int32_t *cl_off, int32_t *n_cl) {
    // int32 scratch of offc_grow_and_merge (7 M + 16) | queue (2 M + 2) | cls (M bytes)
    const size_t m = (size_t)M;
    Scratch sc(s);
    CK(h, sc.alloc((9 * m + 18) * 4 + m));
    int32_t *i32 = sc.as<int32_t>(), *queue = i32 + 7 * m + 16;
    uint8_t *cls = reinterpret_cast<uint8_t *>(queue + 2 * m + 2);
    cudaMemsetAsync(cls, 0, m, s);
    offc_grow_and_merge(s, M, off, col, core, iso, submask, cnt_gt1, pi, cls, queue, i32, label, order, cl_off, n_cl, total);
    return launched(h, "offline cluster growth");
}

// cls [M] and queue [2 M + 2]: scratch of the bit-row scan
int launch_off_clusters(ccb_handle *h, cudaStream_t s, int M, const uint32_t *wnbr, const uint8_t *core,
                        const uint64_t *submask, int cnt_gt1, int64_t pi, uint8_t *cls, int32_t *queue, int32_t *label,
                        int32_t *order, int32_t *cl_off, int32_t *n_cl, int *launches, int csr_min_m) {
    *launches = 0;
    auto bit_rows = [&]() {
        cudaMemsetAsync(cls, 0, (size_t)std::max(M, 1), s);
        k_off_clusters<<<1, OFFC_THREADS, 0, s>>>(M, wnbr, core, submask, cnt_gt1, pi, cls, queue, label, order, cl_off, n_cl);
        *launches += 1;
        return launched(h, "k_off_clusters");
    };
    if (M < (csr_min_m > 0 ? csr_min_m : OFF_CSR_MIN_M) || M == 0) return bit_rows();
    // off (M + 1) | nnz (M int32) | iso (M bytes)
    const size_t m = (size_t)M;
    Scratch sc(s), sc_col(s);
    CK(h, sc.alloc((m + 1) * 8 + m * 5));
    int64_t *off = sc.as<int64_t>();
    int32_t *nnz = reinterpret_cast<int32_t *>(off + m + 1);
    uint8_t *iso = reinterpret_cast<uint8_t *>(nnz + m);
    int rc;
    int64_t total = 0;
    if ((rc = launch_offc_rowinfo(h, s, wnbr, M, 0, M, iso, nnz))) return rc;
    k_offc_scan<int64_t><<<1, OFFG_THREADS, 0, s>>>(nnz, M, off);
    *launches += 2;
    if ((rc = csr_total(h, s, off, M, &total))) return rc;
    if (total > (int64_t)INT32_MAX - 1) // a CSR that large buys nothing over the bit rows
        return bit_rows();
    CK(h, sc_col.alloc((size_t)std::max<int64_t>(total, 1) * 4));
    int32_t *col = sc_col.as<int32_t>();
    if ((rc = launch_offc_fill(h, s, wnbr, M, 0, M, iso, off, col))) return rc;
    *launches += 1;
    rc = off_clusters_csr(h, s, M, off, col, total, iso, core, submask, cnt_gt1, pi, label, order, cl_off, n_cl);
    *launches += 8;
    return rc;
}

// Probes of the pcore replay pattern (mode 3 of ccb_fp64_peak): one warp runs the CLEAN-stage schedule of k_bs_chain_p over
// a ring of records in shared memory -- per cell one dependent DADD, the store of the previous version, the load of an
// addend one batch ahead -- under different conditions; sink[8 + v] = cycles per cell of variant v:
//   0 DADD chain only (addends in registers)      1 + addends from LDS      2 + STS of every version
//   3 as 2, while two other warps spin on mbarrier try_wait (the producer / store threads of the kernel)
//   4 as 2 with 64-bit accesses replaced by lane-strided 8-byte accesses of a 26-element record (the real layout)
template <int VAR>
__device__ __forceinline__ double chain_probe_run(double *sm, int lane, long long &cyc) {
    constexpr int LSP = 26, NB = 64, GS = 8, NG = NB / GS, REP = 32;
    double v = 1.0 + lane * 1e-9;
    uint32_t xa = smem_u32(sm) + (lane < LSP ? lane : 0) * 8;
    asm volatile("" : "+r"(xa));
    const bool st_ok = lane < LSP;
    const long long t0 = clock64();
    for (int rep = 0; rep < REP; ++rep) {
        double R[2][GS];
#pragma unroll
        for (int q = 0; q < GS; ++q) R[0][q] = VAR >= 1 ? lds_f64(xa + (q * LSP) * 8) : 1e-12 * q;
#pragma unroll
        for (int k = 0; k < NG; ++k) {
#pragma unroll
            for (int q = 0; q < GS; ++q) {
                const double nv = ccb::dadd(v, R[k & 1][q]);
                if (VAR >= 2 && k + q > 0 && st_ok) sts_f64(xa + ((k * GS + q - 1) * LSP) * 8, v);
                if (k + 1 < NG) R[(k + 1) & 1][q] = VAR >= 1 ? lds_f64(xa + (((k + 1) * GS + q) * LSP) * 8) : 1e-12 * q;
                v = nv;
            }
        }
        if (VAR >= 2 && st_ok) sts_f64(xa + ((NB - 1) * LSP) * 8, v);
    }
    cyc = clock64() - t0;
    return v;
}
__global__ void k_chain_probe(double *sink) {
    __shared__ __align__(16) double sm[64 * 26 + 32];
    __shared__ uint64_t bar;
    __shared__ volatile int stop;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    for (int i = tid; i < 64 * 26 + 32; i += blockDim.x) sm[i] = 1e-9 * (i % 97);
    if (tid == 0) {
        mbar_init(&bar, 1);
        mbar_fence_init();
        stop = 0;
    }
    __syncthreads();
    if (warp == 0) {
        long long c0, c1, c2, c3;
        double a = chain_probe_run<0>(sm, lane, c0);
        a += chain_probe_run<1>(sm, lane, c1);
        a += chain_probe_run<2>(sm, lane, c2);
        if (lane == 0) stop = 1; // phase 1 over: spinners start
        __syncwarp();
        for (volatile int w = 0; w < 2000; ++w) {}
        a += chain_probe_run<2>(sm, lane, c3);
        if (lane == 0) {
            const double cells = 32.0 * 64.0;
            sink[8] = c0 / cells;
            sink[9] = c1 / cells;
            sink[10] = c2 / cells;
            sink[11] = c3 / cells;
            sink[7] = a;
            stop = 2;
            mbar_arrive(&bar);
        }
        return;
    }
    // warps 1, 2: idle until phase 1 is over, then lane 0 spins on the mbarrier like the producer / store thread do
    if (lane == 0) {
        while (stop == 0) {}
        mbar_wait(&bar, 0);
    }
}

// ---- per-group statistics (stats.cuh) ---------------------------------------------------------------------------------
constexpr int ST_MAX_Q = 64; // quantiles per call: the radix histograms of 2 + 2 nq ranks sit in shared memory

int stats_args(ccb_handle *h, int64_t N, int64_t ld, int D, int G, int nq, const double *q, const int64_t *count,
               const double *mean, const double *median, const double *quant) {
    if (D < 1 || D > CCB_MAX_D || N < 0 || ld < D) return fail(h, CCB_EINVAL, "bad rows: N=%lld ld=%lld D=%d", (long long)N,
                                                                (long long)ld, D);
    if (N >= ((int64_t)1 << 31)) return fail(h, CCB_ELIMIT, "more than 2^31 - 1 cells in one call");
    if (G < 1) return fail(h, CCB_EINVAL, "G = %d < 1", G);
    if (nq < 0 || (nq > 0 && (!q || !quant))) return fail(h, CCB_EINVAL, "bad quantile arguments");
    if (nq > ST_MAX_Q) return fail(h, CCB_ELIMIT, "%d quantiles > %d", nq, ST_MAX_Q);
    for (int j = 0; j < nq; ++j)
        if (!(q[j] >= 0.0 && q[j] <= 1.0)) return fail(h, CCB_EINVAL, "quantile %d = %g outside [0, 1]", j, q[j]);
    if (!count || !mean || !median) return fail(h, CCB_EINVAL, "null output");
    return CCB_OK;
}

// The pipeline of stats.cuh over the rows X [N][ld] (CCB_DTYPE_*) grouped by d_group [N] (device; values outside [0, G)
// are skipped).  xf: the per-column transform of the values (StXf in stats.cuh); cof: device arcsinh cofactors by column
// applied first (k_st_gather_tx), or null.  Outputs are host arrays.
// Synchronises s.  h (may be null) receives the error and counts the launches.  Arguments are checked by stats_args.
int group_stats_run(ccb_handle *h, cudaStream_t s, const void *X, int32_t dtype, int64_t N, int64_t ld, int D,
                    const int32_t *d_group, int G, int nq, const double *q, const StXf &xf, const double *cof, int64_t *count,
                    double *mean, double *median, double *quant) {
    int64_t launches = 0;
    const int R = 2 + 2 * nq;
    const unsigned gN = (unsigned)std::max<int64_t>(1, std::min<int64_t>((N + ST_THREADS - 1) / ST_THREADS, 148 * 8));
    const unsigned gG = (unsigned)std::min<int64_t>((G + 255) / 256, 148 * 8);
    // cells per group; slices; the groups that take the radix select and their slices (four scans of G + 1 entries)
    Scratch qd(s), cs(s);
    CK(h, qd.alloc((size_t)std::max(nq, 1) * 8));
    if (nq) CK(h, cudaMemcpyAsync(qd.p, q, (size_t)nq * 8, cudaMemcpyHostToDevice, s));
    CK(h, cs.alloc(((size_t)G + 4 * (size_t)G + 4 * ((size_t)G + 1) + 4) * 4));
    unsigned *cnt = cs.as<unsigned>();
    int32_t *a = reinterpret_cast<int32_t *>(cnt + G), *sc = a + 4 * (size_t)G, *tot = sc + 4 * ((size_t)G + 1);
    CK(h, cudaMemsetAsync(cnt, 0, (size_t)G * 4, s));
    const int smem_count = G <= ST_THREADS * 16 ? G * 4 : 0;
    k_st_count<<<gN, ST_THREADS, smem_count, s>>>(d_group, N, G, smem_count != 0, cnt);
    k_st_derive<<<gG, 256, 0, s>>>(cnt, G, a);
    k_st_scan<<<4, 1024, 0, s>>>(a, G, sc, G, tot);
    launches += 3;
    CKL(h);
    int32_t t4[4];
    CK(h, cudaMemcpyAsync(t4, tot, sizeof t4, cudaMemcpyDeviceToHost, s));
    CK(h, cudaStreamSynchronize(s));
    const int64_t Nv = t4[0], NS = t4[1], L = t4[2], NLS = t4[3];

    StGeom geo{};
    geo.cnt = cnt, geo.goff = sc, geo.soff = sc + (G + 1), geo.Nv = Nv, geo.D = D;
    Scratch tab(s), srt(s), ks(s), part(s), outd(s), sel_mem(s);
    CK(h, tab.alloc((size_t)(NS + L + 2 * NLS + 1) * 4));
    int32_t *slice_group = tab.as<int32_t>(), *large_group = slice_group + NS, *large_slice = large_group + L,
            *large_slice_l = large_slice + NLS;
    k_st_slices<<<gG, 256, 0, s>>>(sc, G, slice_group, large_group, large_slice, large_slice_l);
    launches++;
    geo.slice_group = slice_group;
    if (Nv > 0) {
        // stable LSD counting sort of the grouped rows by group, 8 bits a pass; the first pass drops the other rows
        int bits = 0;
        while (bits < 31 && ((int64_t)(G - 1) >> bits) != 0) ++bits;
        const int passes = std::max(1, (bits + 7) / 8);
        const int64_t nt_max = (N + ST_TILE - 1) / ST_TILE;
        CK(h, srt.alloc((size_t)(4 * Nv + 2 * 256 * nt_max + 1) * 4));
        int32_t *kb[2] = {srt.as<int32_t>(), srt.as<int32_t>() + Nv}, *vb[2] = {kb[1] + Nv, kb[1] + 2 * Nv};
        int32_t *th = vb[1] + Nv, *toff = th + 256 * nt_max;
        for (int p = 0; p < passes; ++p) {
            const int64_t n = p ? Nv : N;
            const int nt = (int)((n + ST_TILE - 1) / ST_TILE);
            int32_t *ko = kb[p & 1], *vo = vb[p & 1];
            if (p == 0) {
                k_st_sort_hist<true><<<nt, ST_THREADS, 0, s>>>(d_group, n, G, 0, th, nt);
            } else {
                k_st_sort_hist<false><<<nt, ST_THREADS, 0, s>>>(kb[(p - 1) & 1], n, G, 8 * p, th, nt);
            }
            k_st_scan<<<1, 1024, 0, s>>>(th, 0, toff, 256 * nt, tot);
            if (p == 0) {
                k_st_sort_scatter<true><<<nt, ST_THREADS, 0, s>>>(d_group, nullptr, n, G, 0, toff, nt, ko, vo);
            } else {
                k_st_sort_scatter<false><<<nt, ST_THREADS, 0, s>>>(kb[(p - 1) & 1], vb[(p - 1) & 1], n, G, 8 * p, toff, nt,
                                                                   ko, vo);
            }
            launches += 3;
        }
        geo.perm = vb[(passes - 1) & 1];
        CKL(h);
    }
    // keys [D][Nv] in group order, partial sums / NaN counts [NS][D]
    CK(h, ks.alloc(std::max<size_t>((size_t)D * Nv, 1) * 8));
    CK(h, part.alloc(std::max<size_t>((size_t)NS * D, 1) * 12));
    uint64_t *keys = ks.as<uint64_t>();
    double *psum = part.as<double>();
    int32_t *pnan = reinterpret_cast<int32_t *>(psum + (size_t)NS * D);
    if (NS > 0) {
        const size_t smem = (size_t)ST_CHUNK * (D + 1) * 8;
        if (cof && dtype == CCB_DTYPE_F32)
            k_st_gather_tx<float><<<(unsigned)NS, ST_THREADS, smem, s>>>(geo, static_cast<const float *>(X), ld, xf, cof, keys,
                                                                       psum, pnan);
        else if (cof)
            k_st_gather_tx<double><<<(unsigned)NS, ST_THREADS, smem, s>>>(geo, static_cast<const double *>(X), ld, xf, cof,
                                                                        keys, psum, pnan);
        else if (dtype == CCB_DTYPE_F32)
            k_st_gather<float><<<(unsigned)NS, ST_THREADS, smem, s>>>(geo, static_cast<const float *>(X), ld, xf, keys, psum,
                                                                    pnan);
        else
            k_st_gather<double><<<(unsigned)NS, ST_THREADS, smem, s>>>(geo, static_cast<const double *>(X), ld, xf, keys, psum,
                                                                     pnan);
        launches++;
    }
    // outputs
    const size_t GD = (size_t)G * D;
    CK(h, outd.alloc(GD * (2 + (size_t)nq) * 8));
    StOut out{};
    out.q = qd.as<double>(), out.nq = nq, out.G = G;
    out.mean = outd.as<double>(), out.median = out.mean + GD, out.quant = out.median + GD;
    k_st_small<<<(unsigned)G, ST_THREADS, 0, s>>>(geo, keys, psum, pnan, out);
    launches++;
    if (L > 0) {
        const int64_t items = L * D * R;
        CK(h, sel_mem.alloc((size_t)items * (16 + 256 * 4)));
        StSel sel{};
        sel.pre = sel_mem.as<uint64_t>();
        sel.rem = reinterpret_cast<int64_t *>(sel.pre + items);
        sel.hist = reinterpret_cast<unsigned *>(sel.rem + items);
        sel.large_group = large_group, sel.large_slice = large_slice, sel.large_slice_l = large_slice_l, sel.R = R;
        CK(h, cudaMemsetAsync(sel.hist, 0, (size_t)items * 256 * 4, s));
        const unsigned gi = (unsigned)std::min<int64_t>((items + 255) / 256, 148 * 8);
        k_st_rsel_init<<<gi, 256, 0, s>>>(geo, sel, out.q, items);
        const size_t smem = (size_t)R * (256 * 4 + 8);
        CK(h, cudaFuncSetAttribute(k_st_rsel_hist, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        for (int shift = 56; shift >= 0; shift -= 8) {
            k_st_rsel_hist<<<dim3((unsigned)NLS, (unsigned)D), ST_THREADS, smem, s>>>(geo, sel, keys, shift);
            k_st_rsel_fix<<<gi, 256, 0, s>>>(sel, items, shift);
        }
        k_st_large_finish<<<(unsigned)std::min<int64_t>((L * D + 255) / 256, 148 * 8), 256, 0, s>>>(geo, sel, psum, pnan, out,
                                                                                                     L * D);
        launches += 2 + 2 * 8;
    }
    CKL(h);
    std::vector<unsigned> hc(G);
    CK(h, cudaMemcpyAsync(hc.data(), cnt, (size_t)G * 4, cudaMemcpyDeviceToHost, s));
    CK(h, cudaMemcpyAsync(mean, out.mean, GD * 8, cudaMemcpyDeviceToHost, s));
    CK(h, cudaMemcpyAsync(median, out.median, GD * 8, cudaMemcpyDeviceToHost, s));
    if (nq) CK(h, cudaMemcpyAsync(quant, out.quant, GD * nq * 8, cudaMemcpyDeviceToHost, s));
    CK(h, cudaStreamSynchronize(s));
    for (int g = 0; g < G; ++g) count[g] = hc[g];
    if (h) h->st.kernel_launches += launches;
    return CCB_OK;
}

} // namespace

// =====================================================================================================
extern "C" {

const char *ccb_last_error(const ccb_handle *h) { return h ? h->err.c_str() : g_err.c_str(); }
void *ccb_stream(ccb_handle *h) { return h ? (void *)h->stream : nullptr; }

int ccb_create(const ccb_params *p, ccb_handle **out) {
    if (!p || !out) return fail(nullptr, CCB_EINVAL, "null argument");
    *out = nullptr;
    if (p->D < 1 || p->D > CCB_MAX_D) return fail(nullptr, CCB_ELIMIT, "D=%d outside 1..%d", p->D, CCB_MAX_D);
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0)
        return fail(nullptr, CCB_ECUDA, "no CUDA device (%s); this library has no CPU path",
                    e == cudaSuccess ? "device count 0" : cudaGetErrorString(e));
    if (p->device < 0 || p->device >= ndev) return fail(nullptr, CCB_EINVAL, "device %d of %d", p->device, ndev);
    std::unique_ptr<ccb_handle> h(new (std::nothrow) ccb_handle());
    if (!h) return fail(nullptr, CCB_ENOMEM, "host allocation failed");
    h->prm = *p;
    h->D = p->D;
    h->DP = round_dp(p->D);
    if (p->chunk > 0) h->bs_bmax = std::max(32, (p->chunk + 31) / 32 * 32); // block length cap of the BSV engine
    if (p->bsv_bmin > 0) h->bs_bmin = p->bsv_bmin;
    if (p->bsv_iters > 0) h->bs_iters = std::min(p->bsv_iters, 16);
    h->bs_use_graph = p->bsv_stream == 0;
    h->off_csr_min_m = p->off_csr_min_m;
    h->bs_bmax = std::min(h->bs_bmax, 1 << 20);
    const bool p2 = is_pow2(p->k);
    h->div_mode = p2 ? 0 : 1;
    h->wsel = p2 ? 1.0 / p->k : p->k; // exact reciprocal of a power of two, else the divisor itself
    h->cnt_gt1 = p->k > 1.0;
    int rc;
    if ((rc = enter_device(p->device))) return rc;
    CK(nullptr, create(h->stream, 0));
    CK(nullptr, alloc(h->d_ctl, sizeof(Ctl)));
    CK(nullptr, cudaMemset(h->d_ctl, 0, sizeof(Ctl)));
    CK(nullptr, alloc(h->h_ctl, sizeof(Ctl)));
    memset(h->h_ctl, 0, sizeof(Ctl));
    for (int i = 0; i < 2; ++i) {
        if ((rc = alloc_store(h.get(), h->Pm[i], 256)) || (rc = alloc_store(h.get(), h->Om[i], 8192))) return rc;
        h->P[i] = h->Pm[i].view();
        h->O[i] = h->Om[i].view();
    }
    *out = h.release();
    return CCB_OK;
}

void ccb_destroy(ccb_handle *h) {
    if (!h) return;
    cudaSetDevice(h->prm.device);
    if (h->stream) cudaStreamSynchronize(h->stream);
    delete h;
}

int ccb_get_stats(const ccb_handle *h, ccb_stats *out) {
    if (!h || !out) return fail(nullptr, CCB_EINVAL, "null argument");
    // the device-side counters are as of the last control-block read-back (every chunk / ccb_counts)
    *out = h->st;
    const Ctl &c = *h->h_ctl;
    out->upgrades = h->st_base.upgrades + c.upgrades;
    out->created = h->st_base.created + c.created;
    out->downgraded = h->st_base.downgraded + c.downgraded;
    out->deleted = h->st_base.deleted + c.deleted;
    if (h->bs.h_bc) {
        const BsCtl &b = *h->bs.h_bc, &bb = h->bc_base;
        out->bsv_blocks = bb.blocks + b.blocks;
        out->bsv_rounds = bb.iters + b.iters;
        out->bsv_mismatches = bb.mismatches + b.mismatches;
        out->bsv_cuts_unknown = bb.cuts_unknown + b.cuts_unknown;
        out->bsv_cuts_rounds = bb.cuts_iter + b.cuts_iter;
        out->bsv_cuts_capacity = bb.cuts_cap + b.cuts_cap;
        out->bsv_late_topk = bb.tk_late + b.tk_late;
        out->bsv_outlier_stage_cells = bb.rejects + b.rejects;
        out->bsv_replayed_cells = bb.replayed + b.replayed;
        out->bsv_light_rounds = bb.rounds_light + b.rounds_light;
        out->bsv_serial_cells = bb.serial_cells + b.serial_cells;
        out->nearest_pairs += bb.pairs + b.pairs;
    }
    return CCB_OK;
}

#ifdef CCB_DEBUG
// Diagnostics build only (python chronoclust_b200/build.py --debug -> libchronoclust_b200_debug.so, declared in
// csrc/debug.h): none of these symbols exists in the product library.
int64_t ccb_debug_trace(ccb_handle *h, int64_t *out, int64_t max_records) {
    if (!h || !out) return -1;
    cudaStreamSynchronize(h->stream);
    int n = 0;
    cudaMemcpyFromSymbol(&n, g_trace_n, sizeof(int));
    const int64_t m = std::min<int64_t>(std::min<int64_t>(n, CCB_TRACE_MAX), max_records);
    if (m > 0) cudaMemcpyFromSymbol(out, g_trace, (size_t)m * CCB_TRACE_WORDS * sizeof(long long));
    const int zero = 0;
    cudaMemcpyToSymbol(g_trace_n, &zero, sizeof(int));
    return n;
}

int ccb_debug_counters(ccb_handle *h, int64_t *out16, int32_t reset) {
    if (!h || !out16) return -1;
    cudaStreamSynchronize(h->stream);
    cudaMemcpyFromSymbol(out16, g_dbg_cnt, 16 * sizeof(long long));
    if (reset) {
        const long long z[16] = {0};
        cudaMemcpyToSymbol(g_dbg_cnt, z, sizeof(z));
    }
    return 0;
}

int ccb_debug_chain(ccb_handle *h, int64_t *out, int32_t max_keys) {
    if (!h || !out) return fail(h, CCB_EINVAL, "null argument");
    if (!h->ws_dbg) { // first call switches the counters on
        if (h->ws.mp_stride <= 0) return fail(h, CCB_ESTATE, "no block-speculative workspace yet");
        CK(h, cudaStreamSynchronize(h->stream));
        const size_t bytes = (size_t)h->ws.mp_stride * 8 * sizeof(int64_t);
        Dev<int64_t> dbg;
        CK(h, alloc(dbg, bytes));
        CK(h, cudaMemset(dbg, 0, bytes));
        h->ws_dbg = std::move(dbg);
        h->ws.dbg = h->ws_dbg;
        memset(out, 0, (size_t)max_keys * 8 * sizeof(int64_t));
        return CCB_OK;
    }
    CK(h, cudaStreamSynchronize(h->stream));
    const int n = std::min<int>(max_keys, h->ws.mp_stride);
    CK(h, cudaMemcpy(out, h->ws.dbg, (size_t)n * 8 * sizeof(int64_t), cudaMemcpyDeviceToHost));
    return CCB_OK;
}
#endif

int ccb_reset(ccb_handle *h) {
    int rc;
    if ((rc = enter(h)) || (rc = sync_ctl(h))) return rc;
    {
        const Ctl &c = *h->h_ctl;
        h->st_base.upgrades += c.upgrades;
        h->st_base.created += c.created;
        h->st_base.downgraded += c.downgraded;
        h->st_base.deleted += c.deleted;
    }
    memset(h->h_ctl, 0, sizeof(Ctl));
    rc = push_ctl(h);
    if (rc) return rc;
    if (h->bs.bc) {
        CK(h, cudaMemcpyAsync(h->bs.h_bc, h->bs.bc, sizeof(BsCtl), cudaMemcpyDeviceToHost, h->stream));
        CK(h, cudaStreamSynchronize(h->stream));
        const BsCtl &b = *h->bs.h_bc;
        BsCtl &bb = h->bc_base;
        bb.blocks += b.blocks, bb.iters += b.iters, bb.mismatches += b.mismatches, bb.cuts_unknown += b.cuts_unknown;
        bb.cuts_iter += b.cuts_iter, bb.cuts_cap += b.cuts_cap, bb.tk_late += b.tk_late, bb.rejects += b.rejects;
        bb.replayed += b.replayed, bb.pairs += b.pairs, bb.rounds_light += b.rounds_light, bb.serial_cells += b.serial_cells;
        const int32_t keep_B = b.next_B;
        memset(h->bs.h_bc, 0, sizeof(BsCtl));
        h->bs.h_bc->next_B = keep_B;
        CK(h, cudaMemcpyAsync(h->bs.bc, h->bs.h_bc, sizeof(BsCtl), cudaMemcpyHostToDevice, h->stream));
    }
    CK(h, cudaStreamSynchronize(h->stream));
    h->have_params = false;
    h->last.valid = false;
    h->off_M = 0;
    h->cl_off.assign(1, 0);
    h->cl_members.clear();
    h->cl_w.clear();
    return CCB_OK;
}

int ccb_enable_timing(ccb_handle *h, int32_t on) {
    if (!h) return fail(nullptr, CCB_EINVAL, "null handle");
    h->timing = on != 0;
    return CCB_OK;
}

int ccb_get_timing(ccb_handle *h, double ms[CCB_NCAT], int64_t launches[CCB_NCAT], int32_t reset) {
    if (int rc = enter(h)) return rc;
    CK(h, cudaStreamSynchronize(h->stream));
    drain_timing(h);
    for (int i = 0; i < CCB_NCAT; ++i) {
        if (ms) ms[i] = h->cat_ms[i];
        if (launches) launches[i] = h->cat_n[i];
        if (reset) {
            h->cat_ms[i] = 0;
            h->cat_n[i] = 0;
        }
    }
    return CCB_OK;
}

int ccb_set_dnrm2(ccb_handle *h, void *fn) {
    if (!h) return fail(nullptr, CCB_EINVAL, "null handle");
    h->dnrm2 = fn;
    return CCB_OK;
}

int ccb_begin_timepoint(ccb_handle *h, double mu, double omicron, int64_t pi, int32_t decay, double decay_factor) {
    int rc;
    if ((rc = enter(h))) return rc;
    h->mu = mu;
    h->omicron = omicron;
    h->pi = pi;
    h->have_params = true;
    h->last.valid = false;
    if (!decay) return CCB_OK;
    cudaStream_t s = h->stream;
    if ((rc = sync_ctl(h))) return rc;
    // every downgraded pcore MC lands in the outlier list: make room first
    const int64_t need_o = (int64_t)h->h_ctl->n_outlier + h->h_ctl->n_pcore;
    if ((rc = grow_store(h, true, h->h_ctl->n_outlier, need_o))) return rc;
    // kernel 3's plan codes: one per entry of either list
    CK(h, h->d_pnew.ensure((size_t)h->P[h->pcur].cap * 4));
    CK(h, h->d_pfin.ensure((size_t)h->P[h->pcur].cap * 4));
    CK(h, h->d_onew.ensure((size_t)h->O[h->ocur].cap * 4));
    MaintArgs ma{};
    ma.P = h->P[h->pcur];
    ma.O = h->O[h->ocur];
    ma.P2 = h->P[1 - h->pcur];
    ma.O2 = h->O[1 - h->ocur];
    ma.ctl = h->d_ctl;
    ma.p_new = h->d_pnew;
    ma.p_fin = h->d_pfin;
    ma.o_new = h->d_onew;
    ma.f = decay_factor;
    ma.beta_mu = h->prm.beta * mu;
    ma.omicron = omicron;
    ma.pi = pi;
    ma.D = h->D;
    ma.DP = h->DP;
    ma.cnt_gt1 = h->cnt_gt1;
    ma.wsel = h->wsel;
    Timed tm(h, CCB_CAT_MAINT);
    k_maint_plan<<<1, MAINT_THREADS, 0, s>>>(ma);
    CKL(h);
    const int64_t total = (int64_t)(h->h_ctl->n_pcore + h->h_ctl->n_outlier) * h->DP;
    const int gx = (int)std::min<int64_t>(std::max<int64_t>((total + 255) / 256, 1), 148 * 8);
    k_maint_gather<<<gx, 256, 0, s>>>(ma);
    CKL(h);
    k_maint_finish<<<1, 1, 0, s>>>(h->d_ctl);
    CKL(h);
    h->st.kernel_launches += 3;
    h->pcur = 1 - h->pcur;
    h->ocur = 1 - h->ocur;
    tm.stop();
    return sync_ctl(h);
}

// k_stage_rows over n rows of D columns on stream s: the instance with the arcsinh transform when cof is set
static void launch_stage_rows(cudaStream_t s, int32_t dtype, const void *src, int64_t ld_src, double *dst, int64_t ld_dst,
                              int64_t n, int D, const int32_t *cols, const double *cof, const double *scale,
                              const double *shift) {
    const int64_t total = n * D;
    const unsigned gx = (unsigned)std::min<int64_t>((total + 255) / 256, 148 * 16);
    if (cof && dtype == CCB_DTYPE_F32)
        k_stage_rows_tx<float><<<gx, 256, 0, s>>>(static_cast<const float *>(src), ld_src, dst, ld_dst, n, D, cols, cof, scale,
                                                  shift);
    else if (cof)
        k_stage_rows_tx<double><<<gx, 256, 0, s>>>(static_cast<const double *>(src), ld_src, dst, ld_dst, n, D, cols, cof,
                                                   scale, shift);
    else if (dtype == CCB_DTYPE_F32)
        k_stage_rows<float><<<gx, 256, 0, s>>>(static_cast<const float *>(src), ld_src, dst, ld_dst, n, D, cols, scale, shift);
    else
        k_stage_rows<double><<<gx, 256, 0, s>>>(static_cast<const double *>(src), ld_src, dst, ld_dst, n, D, cols, scale,
                                                shift);
}

// widen (and, with cofactors, arcsinh transform, and, with a scaler, min-max transform) n rows of dtype into double rows,
// on the handle's stream.  cols: the device column map of a column-subset ingest (output column d = source column
// cols[d]), or null; cof: the device cofactors by source column, or null
static void stage_rows(ccb_handle *h, int32_t dtype, const void *src, int64_t ld_src, double *dst, int64_t ld_dst, int64_t n,
                       const int32_t *cols, const double *cof, const double *scale, const double *shift) {
    if (n <= 0) return;
    launch_stage_rows(h->stream, dtype, src, ld_src, dst, ld_dst, n, h->D, cols, cof, scale, shift);
    h->st.kernel_launches++;
}

static int ingest_host(ccb_handle *h, const void *X, int32_t dtype, int64_t N, int64_t ld, int W, const int32_t *cols,
                       const double *cof, int32_t *assign_uid, uint8_t *stage, const double *scale, const double *shift);

// host arcsinh cofactors [n]: each 0 (the column stays linear) or positive and finite
static int check_cofactors(ccb_handle *h, const double *cof, int n) {
    for (int c = 0; c < n; ++c)
        if (!(cof[c] >= 0.0 && cof[c] <= DBL_MAX)) // (NaN fails both)
            return fail(h, CCB_EINVAL, "cofactor[%d] = %g: a cofactor is 0 (linear) or positive and finite", c, cof[c]);
    return CCB_OK;
}

// ccb_ingest_ex (cols and cofactor null, W == D), ccb_ingest_cols (cofactor null) and ccb_ingest_tx after enter(): every
// argument check, then the ingest.  cols: null (the identity; W must be D) or host [D] distinct columns of W-wide rows;
// cofactor: null or host [W] arcsinh cofactors by source column.
static int ingest_rows(ccb_handle *h, const void *X, int32_t dtype, int32_t on_device, int64_t N, int64_t ld, int W,
                       const int32_t *cols, const double *cofactor, const double *scale, const double *min_,
                       int32_t *assign_uid, uint8_t *stage) {
    int rc;
    if (!cols && W != h->D) return fail(h, CCB_EINVAL, "row width W = %d without a column map; D = %d", W, h->D);
    if (cols) {
        if (W < h->D || W > CCB_MAX_D) return fail(h, CCB_EINVAL, "row width W = %d outside [D = %d, %d]", W, h->D, CCB_MAX_D);
        uint64_t seen = 0;
        for (int d = 0; d < h->D; ++d) {
            const int32_t c = cols[d];
            if (c < 0 || c >= W) return fail(h, CCB_EINVAL, "cols[%d] = %d outside [0, W = %d)", d, c, W);
            if ((seen >> c) & 1ull) return fail(h, CCB_EINVAL, "column %d appears twice in cols", c);
            seen |= 1ull << c;
        }
    }
    if (cofactor && (rc = check_cofactors(h, cofactor, W))) return rc;
    if (dtype != CCB_DTYPE_F64 && dtype != CCB_DTYPE_F32) return fail(h, CCB_EINVAL, "unknown input dtype %d", (int)dtype);
    if (!scale != !min_) return fail(h, CCB_EINVAL, "scale and min_ must both be set or both be NULL");
    if (ld < W) return fail(h, CCB_EINVAL, "leading dimension %lld < %s = %d", (long long)ld, cols ? "W" : "D", W);
    if (N < 0 || (!X && N > 0) || (!assign_uid && N > 0)) return fail(h, CCB_EINVAL, "bad ingest arguments");
    // (the copies below run behind whatever still reads the vectors and the column map on the handle's stream)
    if (scale) {
        CK(h, h->d_scale.ensure(4 * CCB_MAX_D * sizeof(double)));
        CK(h, cudaMemcpyAsync(h->d_scale, scale, (size_t)h->D * 8, cudaMemcpyHostToDevice, h->stream));
        CK(h, cudaMemcpyAsync(h->d_scale + CCB_MAX_D, min_, (size_t)h->D * 8, cudaMemcpyHostToDevice, h->stream));
    }
    const double *d_sc = scale ? h->d_scale.p : nullptr, *d_sh = scale ? h->d_scale + CCB_MAX_D : nullptr;
    const int32_t *d_cols = nullptr;
    uint64_t colmask = 0;
    if (cols) {
        CK(h, h->d_cols.ensure(CCB_MAX_D * sizeof(int32_t)));
        CK(h, cudaMemcpyAsync(h->d_cols, cols, (size_t)h->D * 4, cudaMemcpyHostToDevice, h->stream));
        d_cols = h->d_cols;
        double by_col[2][CCB_MAX_D] = {}; // scale_ / min_ by source column, for ccb_cluster_stats over the full rows
        for (int d = 0; d < h->D; ++d) {
            colmask |= 1ull << cols[d];
            if (scale) by_col[0][cols[d]] = scale[d], by_col[1][cols[d]] = min_[d];
        }
        if (scale) CK(h, cudaMemcpyAsync(h->d_scale + 2 * CCB_MAX_D, by_col, sizeof by_col, cudaMemcpyHostToDevice, h->stream));
    }
    const double *d_cof = nullptr;
    if (cofactor) {
        CK(h, h->d_cof.ensure(CCB_MAX_D * sizeof(double)));
        CK(h, cudaMemcpyAsync(h->d_cof, cofactor, (size_t)W * 8, cudaMemcpyHostToDevice, h->stream));
        d_cof = h->d_cof;
    }
    h->last.valid = false;
    auto record = [&](const void *rows, int32_t rows_dtype, int64_t ldr, const int32_t *assign) {
        h->last.X = rows, h->last.dtype = rows_dtype, h->last.ld = ldr, h->last.W = cols ? W : h->D, h->last.N = N;
        h->last.assign = assign, h->last.colmask = colmask, h->last.scaled = scale != nullptr;
        h->last.raw_tx = cols && cofactor; // (the d_X rows the engine read are transformed already)
        h->last.valid = true;
    };
    if (!on_device) {
        // (ingest_host leaves the rows in d_X: unstaged float64 ones with the caller's leading dimension, staged ones
        // -- float32 or a column subset -- with D; the full rows it staged stay in d_stg with the caller's)
        if ((rc = ingest_host(h, X, dtype, N, ld, W, d_cols, d_cof, assign_uid, stage, d_sc, d_sh))) return rc;
        if (cols) record(h->d_stg, dtype, ld, h->d_assign);
        else record(h->d_X, CCB_DTYPE_F64, dtype == CCB_DTYPE_F32 ? h->D : ld, h->d_assign);
        return CCB_OK;
    }
    // device-resident rows: float64 without a scaler, a column map or cofactors go to the engine as they are; anything else
    // is staged into d_X (leading dimension D) by one launch -- the caller's buffer is never written
    if (dtype == CCB_DTYPE_F64 && !scale && !cols && !cofactor) {
        const double *Xd = static_cast<const double *>(X);
        if ((rc = ingest_core_bsv(h, Xd, N, ld, assign_uid, stage))) return rc;
        record(Xd, CCB_DTYPE_F64, ld, assign_uid);
        return CCB_OK;
    }
    CK(h, h->d_X.ensure(((size_t)N * h->D + 2) * 8));
    stage_rows(h, dtype, X, ld, h->d_X, h->D, N, d_cols, d_cof, d_sc, d_sh);
    CKL(h);
    if ((rc = ingest_core_bsv(h, h->d_X, N, h->D, assign_uid, stage))) return rc;
    if (cols) record(X, dtype, ld, assign_uid);
    else record(h->d_X, CCB_DTYPE_F64, h->D, assign_uid);
    return CCB_OK;
}

int ccb_ingest_ex(ccb_handle *h, const void *X, int32_t dtype, int32_t on_device, int64_t N, int64_t ld,
                  const double *scale, const double *min_, int32_t *assign_uid, uint8_t *stage) {
    int rc;
    if ((rc = enter(h))) return rc;
    return ingest_rows(h, X, dtype, on_device, N, ld, h->D, nullptr, nullptr, scale, min_, assign_uid, stage);
}

int ccb_ingest_cols(ccb_handle *h, const void *X, int32_t dtype, int32_t on_device, int64_t N, int64_t ld, int32_t W,
                    const int32_t *cols, const double *scale, const double *min_, int32_t *assign_uid, uint8_t *stage) {
    int rc;
    if ((rc = enter(h))) return rc;
    if (!cols) return fail(h, CCB_EINVAL, "null column map");
    return ingest_rows(h, X, dtype, on_device, N, ld, W, cols, nullptr, scale, min_, assign_uid, stage);
}

int ccb_ingest_tx(ccb_handle *h, const void *X, int32_t dtype, int32_t on_device, int64_t N, int64_t ld, int32_t W,
                  const int32_t *cols, const double *cofactor, const double *scale, const double *min_, int32_t *assign_uid,
                  uint8_t *stage) {
    int rc;
    if ((rc = enter(h))) return rc;
    return ingest_rows(h, X, dtype, on_device, N, ld, W, cols, cofactor, scale, min_, assign_uid, stage);
}

int ccb_ingest_device(ccb_handle *h, const double *X_dev, int64_t N, int64_t ld, int32_t *assign_uid_dev,
                      uint8_t *stage_dev) {
    return ccb_ingest_ex(h, X_dev, CCB_DTYPE_F64, 1, N, ld, nullptr, nullptr, assign_uid_dev, stage_dev);
}

int ccb_ingest(ccb_handle *h, const double *X, int64_t N, int64_t ld, int32_t *assign_uid, uint8_t *stage) {
    return ccb_ingest_ex(h, X, CCB_DTYPE_F64, 0, N, ld, nullptr, nullptr, assign_uid, stage);
}

int ccb_ingest_scaled(ccb_handle *h, const double *X_raw, int64_t N, int64_t ld, const double *scale, const double *min_,
                      int32_t *assign_uid, uint8_t *stage) {
    if (!scale || !min_) return fail(h, CCB_EINVAL, "null scaler vectors");
    return ccb_ingest_ex(h, X_raw, CCB_DTYPE_F64, 0, N, ld, scale, min_, assign_uid, stage);
}

// host rows in, per-cell results out.  float64 rows are copied into d_X as they are (leading dimension ld) and, with
// cofactors (cof: device vector) or a scaler (scale / shift: device vectors), transformed there in place; float32 rows,
// and the W-wide rows of a column-subset ingest (cols: device column map), are copied into the staging buffer and
// gathered / widened (and transformed) from there into d_X with leading dimension D.  Either happens segment by segment
// behind the segments' copies.  Arguments are checked by ingest_rows.
static int ingest_host(ccb_handle *h, const void *X, int32_t dtype, int64_t N, int64_t ld, int W, const int32_t *cols,
                       const double *cof, int32_t *assign_uid, uint8_t *stage, const double *scale, const double *shift) {
    int rc;
    if (N == 0) return CCB_OK;
    const bool f32 = dtype == CCB_DTYPE_F32, staged = f32 || cols;
    const size_t esz = f32 ? 4 : 8;
    const int64_t ldX = staged ? h->D : ld; // leading dimension of the rows in d_X
    // the rows [r0, r0 + n) of the caller occupy (n - 1) * ld + W elements: the last row's padding is not read
    auto span = [&](int64_t n) { return (size_t)((n - 1) * ld + W) * esz; };
    CK(h, h->d_X.ensure(((size_t)N * ldX + 2) * 8));
    if (staged) CK(h, h->d_stg.ensure(span(N)));
    CK(h, h->d_assign.ensure((size_t)N * 4));
    CK(h, h->d_stage.ensure((size_t)N));
    const char *src = static_cast<const char *>(X);
    char *dst = staged ? reinterpret_cast<char *>(h->d_stg.p) : reinterpret_cast<char *>(h->d_X.p); // where the copies land
    // the copied rows [r0, r0 + n) -> double rows in d_X, on the handle's stream behind the wait for their copy
    auto stage_seg = [&](int64_t r0, int64_t n) -> int {
        if (staged || cof || scale) {
            stage_rows(h, dtype, dst + r0 * ld * esz, ld, h->d_X + r0 * ldX, ldX, n, cols, cof, scale, shift);
            CKL(h);
        }
        return CCB_OK;
    };
    // segments of the input: one block's worth of rows first, then doubling, the last one takes the rest -- the engine
    // starts after a 3 MB copy instead of a 24 MB one and the copies (5x faster than the engine) stay ahead of it
    // The per-cell results travel back the same way, one segment behind the engine: through a page-locked bounce buffer
    // (the caller's arrays are ordinary pageable memory as a rule -- numpy -- and a device -> pageable copy runs at a
    // fraction of the link rate), copied out by this thread while the engine works on the next segment.  A short last
    // segment keeps the part that cannot overlap (its results) small.
    int64_t seg_end[8];
    int nseg = 1;
    seg_end[0] = N;
    if (!h->timing && N >= 262144) {
        int64_t len = h->bs_bmax, at = 0;
        nseg = 0;
        while (nseg < 6 && at + len + len < N) {
            at += len;
            seg_end[nseg++] = at;
            len *= 2;
        }
        const int64_t tail = 2 * (int64_t)h->bs_bmax;
        if (N - at > 4 * tail) seg_end[nseg++] = N - tail;
        seg_end[nseg++] = N;
    }
    if (nseg == 1) {
        {
            Timed tm(h, CCB_CAT_COPY);
            CK(h, cudaMemcpyAsync(dst, src, span(N), cudaMemcpyHostToDevice, h->stream));
        }
        if ((rc = stage_seg(0, N)) || (rc = ingest_core_bsv(h, h->d_X, N, ldX, h->d_assign, h->d_stage))) return rc;
    } else {
        // The ordered engine consumes cells front to back, so the input travels in segments on a copy stream and the
        // engine starts as soon as the first one has landed: segment k + 1 is queued right after the engine has been
        // launched on segment k (with pageable host memory the staging copy then overlaps the engine, too).
        if (!h->copy_stream) {
            Stream cs, rs;
            Event ev[8];
            CK(h, create(cs, 0));
            CK(h, create(rs, 0));
            for (Event &e : ev) CK(h, create(e, cudaEventDisableTiming));
            h->copy_stream = std::move(cs);
            h->res_stream = std::move(rs);
            std::swap(h->ev_seg, ev);
        }
        CK(h, cudaEventRecord(h->ev_seg[0], h->stream)); // earlier work on the handle's stream (previous readers of d_X)
        CK(h, cudaStreamWaitEvent(h->copy_stream, h->ev_seg[0], 0));
        auto seg_rows = [&](int k, int64_t &r0, int64_t &n) {
            r0 = k ? seg_end[k - 1] : 0;
            n = seg_end[k] - r0;
        };
        auto copy_seg = [&](int k) -> int {
            int64_t r0, n;
            seg_rows(k, r0, n);
            if (n > 0)
                CK(h, cudaMemcpyAsync(dst + r0 * ld * esz, src + r0 * ld * esz, span(n), cudaMemcpyHostToDevice, h->copy_stream));
            CK(h, cudaEventRecord(h->ev_seg[k], h->copy_stream));
            return CCB_OK;
        };
        CK(h, h->h_res.ensure((size_t)N * 5));
        int32_t *ba = reinterpret_cast<int32_t *>(h->h_res.p);
        uint8_t *bs = h->h_res + (size_t)N * 4;
        // results of segment k (its engine run is complete: ingest_core_bsv returns after a synchronisation) -> caller
        auto results_seg = [&](int k) -> int {
            int64_t r0, n;
            seg_rows(k, r0, n);
            if (n <= 0) return CCB_OK;
            CK(h, cudaMemcpyAsync(ba + r0, h->d_assign + r0, (size_t)n * 4, cudaMemcpyDeviceToHost, h->res_stream));
            if (stage) CK(h, cudaMemcpyAsync(bs + r0, h->d_stage + r0, (size_t)n, cudaMemcpyDeviceToHost, h->res_stream));
            CK(h, cudaStreamSynchronize(h->res_stream));
            memcpy(assign_uid + r0, ba + r0, (size_t)n * 4);
            if (stage) memcpy(stage + r0, bs + r0, (size_t)n);
            return CCB_OK;
        };
        if ((rc = copy_seg(0))) return rc;
        for (int k = 0; k < nseg; ++k) {
            int64_t r0, n;
            seg_rows(k, r0, n);
            CK(h, cudaStreamWaitEvent(h->stream, h->ev_seg[k], 0));
            if ((rc = stage_seg(r0, n))) return rc;
            // once the engine is running on segment k: queue the input of segment k + 1, fetch the results of segment k - 1
            const std::function<int()> next = [&]() -> int {
                int r = k + 1 < nseg ? copy_seg(k + 1) : CCB_OK;
                if (!r && k > 0) r = results_seg(k - 1);
                return r;
            };
            if ((rc = ingest_core_bsv(h, h->d_X + r0 * ldX, n, ldX, h->d_assign + r0, h->d_stage + r0, &next))) return rc;
        }
        if ((rc = results_seg(nseg - 1))) return rc;
        return CCB_OK;
    }
    {
        Timed tm(h, CCB_CAT_COPY);
        CK(h, cudaMemcpyAsync(assign_uid, h->d_assign, (size_t)N * 4, cudaMemcpyDeviceToHost, h->stream));
        if (stage) CK(h, cudaMemcpyAsync(stage, h->d_stage, (size_t)N, cudaMemcpyDeviceToHost, h->stream));
    }
    CK(h, cudaStreamSynchronize(h->stream));
    if (h->timing) drain_timing(h);
    return CCB_OK;
}

int ccb_counts(ccb_handle *h, int64_t out[4]) {
    int rc;
    if ((rc = enter(h))) return rc;
    if (!out) return fail(h, CCB_EINVAL, "null argument");
    if ((rc = sync_ctl(h))) return rc;
    out[0] = h->h_ctl->n_pcore;
    out[1] = h->h_ctl->n_outlier_alive;
    out[2] = h->h_ctl->pcore_last_id;
    out[3] = h->h_ctl->outlier_last_id;
    return CCB_OK;
}

int ccb_export_list(ccb_handle *h, int32_t which, int64_t *ids, int64_t *uids, double *w, double *cf1, double *cf2,
                    double *cen, double *pref) {
    int rc;
    if ((rc = enter(h)) || (rc = sync_ctl(h))) return rc;
    const Store &S = which ? h->O[h->ocur] : h->P[h->pcur];
    const int n = which ? h->h_ctl->n_outlier : h->h_ctl->n_pcore;
    const int D = h->D;
    if (n == 0) return CCB_OK;
    std::vector<double> hw(n), h1((size_t)n * D), h2((size_t)n * D), hc((size_t)n * D);
    std::vector<uint64_t> hm(n);
    std::vector<int64_t> hid(n);
    std::vector<int32_t> hu(n);
    CK(h, cudaMemcpy(hw.data(), S.w, (size_t)n * 8, cudaMemcpyDeviceToHost));
    CK(h, cudaMemcpy(h1.data(), S.cf1, (size_t)n * D * 8, cudaMemcpyDeviceToHost));
    CK(h, cudaMemcpy(h2.data(), S.cf2, (size_t)n * D * 8, cudaMemcpyDeviceToHost));
    CK(h, cudaMemcpy(hc.data(), S.cen, (size_t)n * D * 8, cudaMemcpyDeviceToHost));
    CK(h, cudaMemcpy(hm.data(), S.mask, (size_t)n * 8, cudaMemcpyDeviceToHost));
    CK(h, cudaMemcpy(hid.data(), S.id, (size_t)n * 8, cudaMemcpyDeviceToHost));
    CK(h, cudaMemcpy(hu.data(), S.uid, (size_t)n * 4, cudaMemcpyDeviceToHost));
    int o = 0;
    for (int j = 0; j < n; ++j) {
        if (which && hw[j] < 0.0) continue; // tombstone left by an upgrade
        if (ids) ids[o] = hid[j];
        if (uids) uids[o] = hu[j];
        if (w) w[o] = hw[j];
        for (int d = 0; d < D; ++d) {
            if (cf1) cf1[(size_t)o * D + d] = h1[(size_t)j * D + d];
            if (cf2) cf2[(size_t)o * D + d] = h2[(size_t)j * D + d];
            if (cen) cen[(size_t)o * D + d] = hc[(size_t)j * D + d];
            if (pref) pref[(size_t)o * D + d] = ((hm[j] >> d) & 1ull) ? h->prm.k : 1.0;
        }
        ++o;
    }
    return CCB_OK;
}

int ccb_import_list(ccb_handle *h, int32_t which, int64_t n, const int64_t *ids, const int64_t *uids, const double *w,
                    const double *cf1, const double *cf2, const double *cen, const double *pref) {
    int rc;
    if ((rc = enter(h))) return rc;
    if (n < 0) return fail(h, CCB_EINVAL, "bad argument");
    h->last.valid = false;
    if ((rc = sync_ctl(h)) || (rc = grow_store(h, which != 0, 0, std::max<int64_t>(n, 1)))) return rc;
    const int D = h->D;
    Store &S = which ? h->O[h->ocur] : h->P[h->pcur];
    std::vector<uint64_t> hm(n);
    std::vector<int32_t> hu(n);
    for (int64_t j = 0; j < n; ++j) {
        uint64_t m = 0;
        for (int d = 0; d < D; ++d)
            if (pref[(size_t)j * D + d] == h->prm.k && h->prm.k != 1.0) m |= 1ull << d;
        hm[j] = m;
        if (uids[j] < 0 || uids[j] >= ((int64_t)1 << 31)) return fail(h, CCB_ELIMIT, "uid outside int32");
        hu[j] = (int32_t)uids[j];
    }
    if (n) {
        CK(h, cudaMemcpy(S.w, w, (size_t)n * 8, cudaMemcpyHostToDevice));
        CK(h, cudaMemcpy(S.cf1, cf1, (size_t)n * D * 8, cudaMemcpyHostToDevice));
        CK(h, cudaMemcpy(S.cf2, cf2, (size_t)n * D * 8, cudaMemcpyHostToDevice));
        CK(h, cudaMemcpy(S.cen, cen, (size_t)n * D * 8, cudaMemcpyHostToDevice));
        CK(h, cudaMemcpy(S.mask, hm.data(), (size_t)n * 8, cudaMemcpyHostToDevice));
        CK(h, cudaMemcpy(S.id, ids, (size_t)n * 8, cudaMemcpyHostToDevice));
        CK(h, cudaMemcpy(S.uid, hu.data(), (size_t)n * 4, cudaMemcpyHostToDevice));
        k_repack_store<<<(unsigned)(((size_t)n * h->DP + 255) / 256), 256, 0, h->stream>>>(S, (int)n, D, h->DP, h->wsel);
        CKL(h);
        h->st.kernel_launches++;
    }
    if (which) {
        h->h_ctl->n_outlier = (int32_t)n;
        h->h_ctl->n_outlier_alive = (int32_t)n;
    } else {
        h->h_ctl->n_pcore = (int32_t)n;
    }
    if ((rc = push_ctl(h))) return rc;
    CK(h, cudaStreamSynchronize(h->stream));
    return CCB_OK;
}

int ccb_set_counters(ccb_handle *h, int64_t pcore_last_id, int64_t outlier_last_id) {
    int rc;
    if ((rc = enter(h)) || (rc = sync_ctl(h))) return rc;
    h->h_ctl->pcore_last_id = pcore_last_id;
    h->h_ctl->outlier_last_id = outlier_last_id;
    if ((rc = push_ctl(h))) return rc;
    CK(h, cudaStreamSynchronize(h->stream));
    return CCB_OK;
}

// ---- offline ------------------------------------------------------------------------------------------
int ccb_offline(ccb_handle *h, int64_t *n_clusters) {
    int rc;
    if ((rc = enter(h))) return rc;
    if (!h->have_params) return fail(h, CCB_ESTATE, "ccb_begin_timepoint must precede ccb_offline");
    if ((rc = sync_ctl(h))) return rc;
    cudaStream_t s = h->stream;
    const int M = h->h_ctl->n_pcore, D = h->D;
    const Store &P = h->P[h->pcur];
    const int words = (M + 31) / 32;
    h->off_M = M;
    h->cl_off.assign(1, 0);
    h->cl_members.clear();
    h->cl_w.clear();
    h->cl_cf1.clear();
    h->cl_cf2.clear();
    h->cl_cen.clear();
    h->cl_pref.clear();
    h->cl_label.assign(M, -1);
    if (n_clusters) *n_clusters = 0;
    if (M == 0) return CCB_OK;

    const double E2 = h->prm.upsilon_eps2;
    Timed tm_off(h, CCB_CAT_OFFLINE);
    uint8_t *core, *cls;
    uint32_t *nbr, *wnbr;
    int32_t *cnt, *queue, *label, *order, *cloff, *ncl;
    uint64_t *submask;
#define OBUF(var, which, n)                                                      \
    if ((rc = off_buf(h, ccb_handle::which, (size_t)(n) * sizeof(*var)))) return rc; \
    var = (decltype(var))h->ob[ccb_handle::which].p
    OBUF(core, OB_CORE, M);
    OBUF(cls, OB_CLS, M);
    OBUF(nbr, OB_NBR, (size_t)M * words);
    OBUF(wnbr, OB_WNBR, (size_t)M * words);
    OBUF(cnt, OB_CNT, M);
    OBUF(queue, OB_QUEUE, 2 * (size_t)M + 2);
    OBUF(label, OB_LABEL, M);
    OBUF(order, OB_ORDER, M);
    OBUF(cloff, OB_CLOFF, (size_t)M + 2);
    OBUF(ncl, OB_NCL, 1);
    OBUF(submask, OB_SUBMASK, M);

    k_off_core<<<(M + 127) / 128, 128, 0, s>>>(P.cf1, P.cf2, P.w, P.mask, M, D, h->prm.k, h->wsel, h->div_mode, h->cnt_gt1,
                                               h->prm.eps2, h->mu, h->pi, core);
    CKL(h);
    h->st.kernel_launches++;
    int64_t nb = 0;
    int nl = 0;
    if ((rc = off_neighbours_settled(h, s, P.cen, M, D, 0, M, h->prm.upsilon_eps, E2, h->dnrm2, nbr, cnt, &nb)))
        return rc;
    h->st.borderline_pairs += nb;
    if ((rc = launch_off_subspace(h, s, P.cen, M, D, 0, M, nbr, cnt, h->prm.delta, submask)) ||
        (rc = launch_off_weighted(h, s, P.cen, M, D, 0, M, nbr, submask, h->prm.k, E2, wnbr)) ||
        (rc = launch_off_clusters(h, s, M, wnbr, core, submask, h->cnt_gt1, h->pi, cls, queue, label, order, cloff, ncl, &nl,
                                  h->off_csr_min_m)))
        return rc;
    h->st.kernel_launches += 2 + nl;
    int32_t nc_raw = 0;
    CK(h, cudaMemcpyAsync(&nc_raw, ncl, 4, cudaMemcpyDeviceToHost, s));
    CK(h, cudaStreamSynchronize(s));
    std::vector<int32_t> hl(M), ho(M), hoff((size_t)nc_raw + 1);
    std::vector<double> kw(nc_raw), k1((size_t)nc_raw * D), k2((size_t)nc_raw * D), kc((size_t)nc_raw * D);
    std::vector<uint64_t> km(nc_raw);
    if (nc_raw > 0) {
        double *d1, *d2, *dc, *dw;
        uint64_t *omask;
        OBUF(d1, OB_D1, (size_t)nc_raw * D);
        OBUF(d2, OB_D2, (size_t)nc_raw * D);
        OBUF(dc, OB_DC, (size_t)nc_raw * D);
        OBUF(dw, OB_DW, nc_raw);
        OBUF(omask, OB_OMASK, nc_raw);
        k_off_cluster_cf<<<nc_raw, 64, 0, s>>>(P.cf1, P.cf2, P.w, D, order, cloff, h->prm.delta2, d1, d2, dc, omask, dw);
        CKL(h);
        h->st.kernel_launches++;
        CK(h, cudaMemcpyAsync(kw.data(), dw, (size_t)nc_raw * 8, cudaMemcpyDeviceToHost, s));
        CK(h, cudaMemcpyAsync(k1.data(), d1, k1.size() * 8, cudaMemcpyDeviceToHost, s));
        CK(h, cudaMemcpyAsync(k2.data(), d2, k2.size() * 8, cudaMemcpyDeviceToHost, s));
        CK(h, cudaMemcpyAsync(kc.data(), dc, kc.size() * 8, cudaMemcpyDeviceToHost, s));
        CK(h, cudaMemcpyAsync(km.data(), omask, (size_t)nc_raw * 8, cudaMemcpyDeviceToHost, s));
    }
#undef OBUF
    tm_off.stop();
    CK(h, cudaMemcpyAsync(hl.data(), label, (size_t)M * 4, cudaMemcpyDeviceToHost, s));
    CK(h, cudaMemcpyAsync(ho.data(), order, (size_t)M * 4, cudaMemcpyDeviceToHost, s));
    CK(h, cudaMemcpyAsync(hoff.data(), cloff, hoff.size() * 4, cudaMemcpyDeviceToHost, s));
    std::vector<int64_t> ids(M);
    CK(h, cudaMemcpyAsync(ids.data(), P.id, (size_t)M * 8, cudaMemcpyDeviceToHost, s));
    CK(h, cudaStreamSynchronize(s));
    if (h->timing) drain_timing(h);
    // keep clusters whose weight is > 0 (predecon.py:83); relabel
    std::vector<int32_t> remap(nc_raw, -1);
    for (int c = 0; c < nc_raw; ++c) {
        if (!(kw[c] > 0.0)) continue;
        remap[c] = (int32_t)h->cl_w.size();
        h->cl_w.push_back(kw[c]);
        for (int i = hoff[c]; i < hoff[c + 1]; ++i) h->cl_members.push_back(ids[ho[i]]);
        h->cl_off.push_back((int64_t)h->cl_members.size());
        for (int d = 0; d < D; ++d) {
            h->cl_cf1.push_back(k1[(size_t)c * D + d]);
            h->cl_cf2.push_back(k2[(size_t)c * D + d]);
            h->cl_cen.push_back(kc[(size_t)c * D + d]);
            h->cl_pref.push_back(((km[c] >> d) & 1ull) ? h->prm.k : 1.0);
        }
    }
    for (int j = 0; j < M; ++j) h->cl_label[j] = hl[j] >= 0 ? remap[hl[j]] : -1;
    if (n_clusters) *n_clusters = (int64_t)h->cl_w.size();
    return CCB_OK;
}

int ccb_cluster_sizes(ccb_handle *h, int64_t out[3]) {
    if (!h || !out) return fail(nullptr, CCB_EINVAL, "null argument");
    out[0] = (int64_t)h->cl_w.size();
    out[1] = (int64_t)h->cl_members.size();
    out[2] = h->off_M;
    return CCB_OK;
}

int ccb_export_clusters(ccb_handle *h, int64_t *off, int64_t *members, double *w, double *cf1, double *cf2, double *cen,
                        double *pref, int32_t *label) {
    if (!h) return fail(nullptr, CCB_EINVAL, "null handle");
    auto cp = [](auto *dst, const auto &v) {
        if (dst && !v.empty()) memcpy(dst, v.data(), v.size() * sizeof(v[0]));
    };
    cp(off, h->cl_off);
    cp(members, h->cl_members);
    cp(w, h->cl_w);
    cp(cf1, h->cl_cf1);
    cp(cf2, h->cl_cf2);
    cp(cen, h->cl_cen);
    cp(pref, h->cl_pref);
    cp(label, h->cl_label);
    return CCB_OK;
}

int ccb_export_offline(ccb_handle *h, uint8_t *core, uint8_t *nbr, uint8_t *wnbr, double *subw) {
    if (int rc = enter(h)) return rc;
    const int64_t M = h->off_M;
    if (M == 0) return CCB_OK;
    // read back from the offline workspace of the last ccb_offline (kept on the device until the next one)
    const int D = h->D, words = (int)((M + 31) / 32);
    std::vector<uint8_t> hcore(M);
    std::vector<uint32_t> hn((size_t)M * words), hw((size_t)M * words);
    std::vector<uint64_t> hs(M);
    CK(h, cudaStreamSynchronize(h->stream));
    CK(h, cudaMemcpy(hcore.data(), h->ob[ccb_handle::OB_CORE].p, (size_t)M, cudaMemcpyDeviceToHost));
    CK(h, cudaMemcpy(hn.data(), h->ob[ccb_handle::OB_NBR].p, hn.size() * 4, cudaMemcpyDeviceToHost));
    CK(h, cudaMemcpy(hw.data(), h->ob[ccb_handle::OB_WNBR].p, hw.size() * 4, cudaMemcpyDeviceToHost));
    CK(h, cudaMemcpy(hs.data(), h->ob[ccb_handle::OB_SUBMASK].p, (size_t)M * 8, cudaMemcpyDeviceToHost));
    for (int64_t p = 0; p < M; ++p) {
        if (core) core[p] = hcore[p];
        for (int64_t q = 0; q < M; ++q) {
            if (nbr) nbr[p * M + q] = (hn[p * words + (q >> 5)] >> (q & 31)) & 1u;
            if (wnbr) wnbr[p * M + q] = (hw[p * words + (q >> 5)] >> (q & 31)) & 1u;
        }
        if (subw)
            for (int d = 0; d < D; ++d) subw[p * D + d] = ((hs[p] >> d) & 1ull) ? h->prm.k : 1.0;
    }
    return CCB_OK;
}

// ---- FP64 pipe microbenchmark (roofline denominators; MEASURED_PEAKS.json has no FP64 figure) ----------
__global__ void k_fp64_peak(int mode, int iters, double *sink) {
    double a0 = threadIdx.x * 1e-9 + 1.0, a1 = a0 + 0.1, a2 = a0 + 0.2, a3 = a0 + 0.3;
    double a4 = a0 + 0.4, a5 = a0 + 0.5, a6 = a0 + 0.6, a7 = a0 + 0.7;
    const double m = 1.0000000001, c = 1e-12;
    if (mode == 0) { // fused multiply-add stream: 2 flop per instruction
        for (int i = 0; i < iters; ++i) {
            a0 = __fma_rn(a0, m, c); a1 = __fma_rn(a1, m, c); a2 = __fma_rn(a2, m, c); a3 = __fma_rn(a3, m, c);
            a4 = __fma_rn(a4, m, c); a5 = __fma_rn(a5, m, c); a6 = __fma_rn(a6, m, c); a7 = __fma_rn(a7, m, c);
        }
    } else { // separate multiply and add, never contracted: 1 flop per instruction (what parity allows)
        for (int i = 0; i < iters; ++i) {
            a0 = __dadd_rn(__dmul_rn(a0, m), c); a1 = __dadd_rn(__dmul_rn(a1, m), c);
            a2 = __dadd_rn(__dmul_rn(a2, m), c); a3 = __dadd_rn(__dmul_rn(a3, m), c);
            a4 = __dadd_rn(__dmul_rn(a4, m), c); a5 = __dadd_rn(__dmul_rn(a5, m), c);
            a6 = __dadd_rn(__dmul_rn(a6, m), c); a7 = __dadd_rn(__dmul_rn(a7, m), c);
        }
    }
    const double r = a0 + a1 + a2 + a3 + a4 + a5 + a6 + a7;
    if (r == 123.456) sink[0] = r;
}

// single-warp latency probes (cycles per dependent step), results in sink[1..]
__global__ void k_fp64_latency(double *sink) {
    __shared__ double sm[64 * 26];
    const int lane = threadIdx.x;
    for (int i = lane; i < 64 * 26; i += 32) sm[i] = 1e-9 * i;
    __syncwarp();
    double a = lane * 1e-9 + 1.0;
    const double c = 1e-12, m = 1.0000000001;
    long long t0 = clock64();
#pragma unroll 16
    for (int i = 0; i < 1024; ++i) a = __dadd_rn(a, c);
    long long t1 = clock64();
    const double r_add = (double)(t1 - t0) / 1024.0;
    t0 = clock64();
#pragma unroll 16
    for (int i = 0; i < 1024; ++i) a = __dmul_rn(a, m);
    t1 = clock64();
    const double r_mul = (double)(t1 - t0) / 1024.0;
    t0 = clock64();
#pragma unroll 16
    for (int i = 0; i < 1024; ++i) a = __fma_rn(a, m, c);
    t1 = clock64();
    const double r_fma = (double)(t1 - t0) / 1024.0;
    // the replay pattern: 8 loads, 8 chained adds, 8 stores in place
    t0 = clock64();
    for (int g = 0; g < 128; ++g) {
        double av[8];
        const int base = (g & 7) * 8 * 26 + (lane < 26 ? lane : 0);
#pragma unroll
        for (int q = 0; q < 8; ++q) av[q] = sm[base + q * 26];
#pragma unroll
        for (int q = 0; q < 8; ++q) {
            a = __dadd_rn(a, av[q]);
            if (lane < 26) sm[base + q * 26] = a;
        }
    }
    t1 = clock64();
    const double r_rep = (double)(t1 - t0) / 1024.0;
    float f = (float)a;
    t0 = clock64();
#pragma unroll 16
    for (int i = 0; i < 1024; ++i) f = __fadd_rn(f, 1e-6f);
    t1 = clock64();
    const double r_fadd = (double)(t1 - t0) / 1024.0;
    if (lane == 0) {
        sink[1] = r_add;
        sink[2] = r_mul;
        sink[3] = r_fma;
        sink[4] = r_rep;
        sink[5] = r_fadd;
        sink[6] = a + f;
    }
}

int ccb_fp64_peak(int32_t device, void *stream, int32_t mode, int32_t iters, int32_t blocks, double *sink,
                  double *flops_out) {
    if (int rc = enter_device(device)) return rc;
    if (mode == 3) { // probes of the replay pattern: sink[8..11] = cycles per cell (see k_chain_probe)
        k_chain_probe<<<1, 96, 0, (cudaStream_t)stream>>>(sink);
        if (flops_out) *flops_out = 0.0;
        return launched(nullptr, "k_chain_probe");
    }
    if (mode == 2) { // latency probes: sink[1..5] = cycles per dependent DADD, DMUL, DFMA, replay step, FADD
        k_fp64_latency<<<1, 32, 0, (cudaStream_t)stream>>>(sink);
        if (flops_out) *flops_out = 0.0;
        return launched(nullptr, "k_fp64_latency");
    }
    k_fp64_peak<<<blocks, 256, 0, (cudaStream_t)stream>>>(mode, iters, sink);
    if (int rc = launched(nullptr, "k_fp64_peak")) return rc;
    if (flops_out) *flops_out = (double)blocks * 256.0 * (double)iters * 8.0 * 2.0; // 8 chains x (mul + add)
    return CCB_OK;
}

// ---- stateless device-pointer entry points ------------------------------------------------------------
int ccb_nearest(int32_t device, void *stream, const double *X, int64_t N, int64_t ld, int32_t D, const double *cen,
                const uint64_t *prefmask, int64_t M, double k, int32_t *slot, double *dist) {
    if (D < 1 || D > CCB_MAX_D || N < 0 || M < 0 || ld < D) return fail(nullptr, CCB_EINVAL, "bad ccb_nearest arguments");
    if (int rc = enter_device(device)) return rc;
    cudaStream_t s = (cudaStream_t)stream;
    if (N == 0) return CCB_OK;
    if (M == 0) {
        cudaMemsetAsync(slot, 0xff, (size_t)N * 4, s);
        return CCB_OK;
    }
    const int DP = round_dp(D);
    const bool p2 = is_pow2(k);
    const double wsel = p2 ? 1.0 / k : k;
    // scratch: packed rows + per-slab candidates, sized by the split the launch will use
    int max_slabs = 1;
    {
        int ok = 0;
        CCB_DISPATCH_DP(DP, {
            int gx, slab_mcs;
            nearest_static_split<kDP, 1>(p2 ? 0 : 1, N, (int)M, MAX_SLABS, gx, slab_mcs, max_slabs);
            ok = 1;
        })
        if (!ok) return fail(nullptr, CCB_ELIMIT, "unsupported dimensionality %d", D);
    }
    Scratch cw(s), sd(s), si(s);
    CK(nullptr, cw.alloc((size_t)M * DP * sizeof(double2)));
    CK(nullptr, sd.alloc((size_t)N * max_slabs * 8));
    CK(nullptr, si.alloc((size_t)N * max_slabs * 4));
    k_pack_cw<<<(unsigned)(((size_t)M * DP + 255) / 256), 256, 0, s>>>(cen, prefmask, M, D, DP, wsel, cw.as<double2>());
    return launch_nearest<1>(nullptr, s, DP, p2 ? 0 : 1, X, nullptr, nullptr, 0, N, ld, D, cw.as<double2>(), (int)M,
                             sd.as<double>(), si.as<int32_t>(), dist, slot, max_slabs, nullptr);
}

int ccb_assoc_nearest(int32_t device, void *stream, const double *cur_cen, const uint64_t *cur_prefmask, int64_t Q,
                      const double *prev_cen, int64_t P, int32_t D, double k, int32_t *best, double *dist) {
    return ccb_assoc_nearest2(device, stream, cur_cen, cur_prefmask, Q, prev_cen, P, D, k, best, dist, nullptr);
}

int ccb_assoc_nearest2(int32_t device, void *stream, const double *cur_cen, const uint64_t *cur_prefmask, int64_t Q,
                       const double *prev_cen, int64_t P, int32_t D, double k, int32_t *best, double *dist, double *dist2) {
    if (D < 1 || D > CCB_MAX_D || Q < 0 || P < 0 || Q >= ((int64_t)1 << 31) || P >= ((int64_t)1 << 31))
        return fail(nullptr, CCB_EINVAL, "bad ccb_assoc_nearest arguments");
    if (int rc = enter_device(device)) return rc;
    cudaStream_t s = (cudaStream_t)stream;
    if (Q == 0) return CCB_OK;
    if (P == 0) {
        cudaMemsetAsync(best, 0xff, (size_t)Q * 4, s);
        return CCB_OK;
    }
    const int DP = round_dp(D);
    const bool p2 = is_pow2(k);
    int ok = 0;
    CCB_DISPATCH_DP(DP, {
        const int gx = (int)((Q + ASSOC_THREADS - 1) / ASSOC_THREADS);
        if (p2) k_assoc<kDP, false><<<gx, ASSOC_THREADS, 0, s>>>(cur_cen, cur_prefmask, (int)Q, prev_cen, (int)P, D, k, 1.0 / k, best, dist, dist2);
        else k_assoc<kDP, true><<<gx, ASSOC_THREADS, 0, s>>>(cur_cen, cur_prefmask, (int)Q, prev_cen, (int)P, D, k, k, best, dist, dist2);
        ok = 1;
    })
    if (!ok) return fail(nullptr, CCB_ELIMIT, "unsupported dimensionality %d", D);
    return launched(nullptr, "k_assoc launch");
}

int ccb_colminmax_ex(int32_t device, void *stream, const void *X_dev, int32_t dtype, int64_t N, int64_t ld, int32_t D,
                     double *min_dev, double *max_dev) {
    if (dtype != CCB_DTYPE_F64 && dtype != CCB_DTYPE_F32) return fail(nullptr, CCB_EINVAL, "unknown input dtype %d", (int)dtype);
    if (D < 1 || D > CCB_MAX_D || N < 0 || ld < D) return fail(nullptr, CCB_EINVAL, "bad ccb_colminmax arguments");
    if (int rc = enter_device(device)) return rc;
    cudaStream_t s = (cudaStream_t)stream;
    Scratch sc(s);
    CK(nullptr, sc.alloc(2 * (size_t)D * 8));
    unsigned long long *okey = sc.as<unsigned long long>();
    cudaMemsetAsync(okey, 0xff, (size_t)D * 8, s);   // running minima: largest key
    cudaMemsetAsync(okey + D, 0x00, (size_t)D * 8, s); // running maxima: smallest key
    const int64_t total = N * D;
    const unsigned gx = (unsigned)std::min<int64_t>((total + 255) / 256, 148 * 8);
    if (total > 0 && dtype == CCB_DTYPE_F32)
        k_colminmax<float><<<gx, 256, 0, s>>>(static_cast<const float *>(X_dev), N, ld, D, okey);
    else if (total > 0)
        k_colminmax<double><<<gx, 256, 0, s>>>(static_cast<const double *>(X_dev), N, ld, D, okey);
    k_colminmax_finish<<<1, 64, 0, s>>>(okey, D, min_dev, max_dev);
    return launched(nullptr, "k_colminmax");
}

int ccb_arcsinh(int32_t device, void *stream, const void *X_dev, int32_t dtype, int64_t N, int64_t ld, int32_t D,
                const double *cofactor, double *out_dev) {
    if (dtype != CCB_DTYPE_F64 && dtype != CCB_DTYPE_F32) return fail(nullptr, CCB_EINVAL, "unknown input dtype %d", (int)dtype);
    if (D < 1 || D > CCB_MAX_D || N < 0 || ld < D || !cofactor || (N > 0 && (!X_dev || !out_dev)))
        return fail(nullptr, CCB_EINVAL, "bad ccb_arcsinh arguments");
    if (int rc = check_cofactors(nullptr, cofactor, D)) return rc;
    if (int rc = enter_device(device)) return rc;
    if (N == 0) return CCB_OK;
    cudaStream_t s = (cudaStream_t)stream;
    Scratch sc(s);
    CK(nullptr, sc.alloc((size_t)D * 8));
    CK(nullptr, cudaMemcpyAsync(sc.p, cofactor, (size_t)D * 8, cudaMemcpyHostToDevice, s));
    launch_stage_rows(s, dtype, X_dev, ld, out_dev, D, N, D, nullptr, sc.as<double>(), nullptr, nullptr);
    return launched(nullptr, "k_stage_rows (ccb_arcsinh)");
}

int ccb_colminmax(int32_t device, void *stream, const double *X_dev, int64_t N, int64_t ld, int32_t D, double *min_dev,
                  double *max_dev) {
    return ccb_colminmax_ex(device, stream, X_dev, CCB_DTYPE_F64, N, ld, D, min_dev, max_dev);
}

int ccb_off_neighbours(int32_t device, void *stream, const double *cen, int64_t M, int32_t D, int64_t r0, int64_t r1,
                       double E, double E2, void *dnrm2, uint32_t *nbr, int32_t *cnt, int64_t *n_border) {
    if (D < 1 || D > CCB_MAX_D || M < 0 || r0 < 0 || r1 < r0 || r1 > M || !n_border)
        return fail(nullptr, CCB_EINVAL, "bad arguments");
    if (int rc = enter_device(device)) return rc;
    return off_neighbours_settled(nullptr, (cudaStream_t)stream, cen, (int)M, D, (int)r0, (int)r1, E, E2, dnrm2, nbr, cnt,
                                  n_border);
}

int ccb_off_subspace(int32_t device, void *stream, const double *cen, int64_t M, int32_t D, int64_t r0, int64_t r1,
                     const uint32_t *nbr, const int32_t *cnt, double delta, uint64_t *submask) {
    if (D < 1 || D > CCB_MAX_D || M < 0 || r0 < 0 || r1 < r0 || r1 > M) return fail(nullptr, CCB_EINVAL, "bad arguments");
    if (int rc = enter_device(device)) return rc;
    return launch_off_subspace(nullptr, (cudaStream_t)stream, cen, (int)M, D, (int)r0, (int)r1, nbr, cnt, delta, submask);
}

int ccb_off_weighted(int32_t device, void *stream, const double *cen, int64_t M, int32_t D, int64_t r0, int64_t r1,
                     const uint32_t *nbr, const uint64_t *submask_all, double k, double E2, uint32_t *wnbr) {
    if (D < 1 || D > CCB_MAX_D || M < 0 || r0 < 0 || r1 < r0 || r1 > M) return fail(nullptr, CCB_EINVAL, "bad arguments");
    if (int rc = enter_device(device)) return rc;
    return launch_off_weighted(nullptr, (cudaStream_t)stream, cen, (int)M, D, (int)r0, (int)r1, nbr, submask_all, k, E2, wnbr);
}

int ccb_off_clusters(int32_t device, void *stream, int64_t M, const uint32_t *wnbr, const uint8_t *core,
                     const uint64_t *submask_all, double k, int64_t pi, int32_t csr_min_m, int32_t *label, int32_t *order,
                     int32_t *cl_off, int32_t *n_cl) {
    if (M < 0) return fail(nullptr, CCB_EINVAL, "bad arguments");
    if (int rc = enter_device(device)) return rc;
    cudaStream_t s = (cudaStream_t)stream;
    Scratch cls(s), queue(s);
    CK(nullptr, cls.alloc((size_t)std::max<int64_t>(M, 1)));
    CK(nullptr, queue.alloc((2 * (size_t)M + 2) * 4));
    int nl = 0;
    return launch_off_clusters(nullptr, s, (int)M, wnbr, core, submask_all, k > 1.0, pi, cls.as<uint8_t>(), queue.as<int32_t>(),
                               label, order, cl_off, n_cl, &nl, csr_min_m);
}

int ccb_offc_rowinfo(int32_t device, void *stream, const uint32_t *wnbr_rows, int64_t M, int64_t r0, int64_t r1, uint8_t *iso,
                     int32_t *nnz) {
    if (M < 0 || r0 < 0 || r1 < r0 || r1 > M) return fail(nullptr, CCB_EINVAL, "bad arguments");
    if (int rc = enter_device(device)) return rc;
    return launch_offc_rowinfo(nullptr, (cudaStream_t)stream, wnbr_rows, (int)M, (int)r0, (int)r1, iso, nnz);
}

int ccb_offc_fill(int32_t device, void *stream, const uint32_t *wnbr_rows, int64_t M, int64_t r0, int64_t r1,
                  const uint8_t *iso_all, const int64_t *off_all, int32_t *col) {
    if (M < 0 || r0 < 0 || r1 < r0 || r1 > M) return fail(nullptr, CCB_EINVAL, "bad arguments");
    if (int rc = enter_device(device)) return rc;
    return launch_offc_fill(nullptr, (cudaStream_t)stream, wnbr_rows, (int)M, (int)r0, (int)r1, iso_all, off_all, col);
}

int ccb_off_clusters_csr(int32_t device, void *stream, int64_t M, const int64_t *off, const int32_t *col, const uint8_t *iso,
                         const uint8_t *core, const uint64_t *submask_all, double k, int64_t pi, int32_t *label, int32_t *order,
                         int32_t *cl_off, int32_t *n_cl) {
    if (M < 0 || M >= ((int64_t)1 << 31)) return fail(nullptr, CCB_EINVAL, "bad arguments");
    if (int rc = enter_device(device)) return rc;
    cudaStream_t s = (cudaStream_t)stream;
    if (M == 0) {
        cudaMemsetAsync(n_cl, 0, 4, s);
        cudaMemsetAsync(cl_off, 0, 4, s);
        return CCB_OK;
    }
    int64_t total = 0; // list lengths decide between the walks
    const int rc = csr_total(nullptr, s, off, (int)M, &total);
    return rc ? rc
              : off_clusters_csr(nullptr, s, (int)M, off, col, total, iso, core, submask_all, k > 1.0, pi, label, order, cl_off,
                                 n_cl);
}

int ccb_group_stats(int32_t device, void *stream, const void *X, int32_t dtype, int64_t N, int64_t ld, int32_t D,
                    const int32_t *group, int32_t G, int32_t nq, const double *q, int64_t *count, double *mean, double *median,
                    double *quant) {
    if (dtype != CCB_DTYPE_F64 && dtype != CCB_DTYPE_F32) return fail(nullptr, CCB_EINVAL, "unknown input dtype %d", (int)dtype);
    if (int rc = stats_args(nullptr, N, ld, D, G, nq, q, count, mean, median, quant)) return rc;
    if (N > 0 && (!X || !group)) return fail(nullptr, CCB_EINVAL, "null rows or groups");
    if (int rc = enter_device(device)) return rc;
    return group_stats_run(nullptr, (cudaStream_t)stream, X, dtype, N, ld, D, group, G, nq, q, StXf{}, nullptr, count, mean, median,
                           quant);
}

int ccb_cluster_stats(ccb_handle *h, const int32_t *group_of_pcore, int64_t n_pcore, int32_t G, int32_t nq, const double *q,
                      int64_t *count, double *mean, double *median, double *quant) {
    int rc;
    if ((rc = enter(h))) return rc;
    if (!h->last.valid)
        return fail(h, CCB_ESTATE, "no ingest since the last ccb_begin_timepoint / ccb_reset / ccb_import_list");
    if (G < 0 || G == INT32_MAX) return fail(h, CCB_EINVAL, "G = %d", G);
    if ((rc = stats_args(h, h->last.N, h->last.ld, h->last.W, G + 1, nq, q, count, mean, median, quant))) return rc;
    if ((rc = sync_ctl(h))) return rc;
    const int np = h->h_ctl->n_pcore;
    if (n_pcore != np) return fail(h, CCB_EINVAL, "n_pcore = %lld, the pcore list holds %d", (long long)n_pcore, np);
    if (np > 0 && !group_of_pcore) return fail(h, CCB_EINVAL, "null group_of_pcore");
    for (int p = 0; p < np; ++p)
        if (group_of_pcore[p] >= G) return fail(h, CCB_EINVAL, "group_of_pcore[%d] = %d >= G = %d", p, group_of_pcore[p], G);
    cudaStream_t s = h->stream;
    const int64_t N = h->last.N, nlut = std::max<int64_t>(h->h_ctl->outlier_last_id, 1);
    Scratch sc(s);
    CK(h, sc.alloc(((size_t)nlut + np + N) * 4));
    int32_t *lut = sc.as<int32_t>(), *gop = lut + nlut, *group = gop + np;
    const unsigned gx = (unsigned)std::max<int64_t>(1, std::min<int64_t>((std::max<int64_t>(nlut, N) + 255) / 256, 148 * 8));
    k_st_lut_fill<<<gx, 256, 0, s>>>(lut, nlut, G);
    if (np > 0) {
        CK(h, cudaMemcpyAsync(gop, group_of_pcore, (size_t)np * 4, cudaMemcpyHostToDevice, s));
        k_st_lut_pcore<<<(np + 255) / 256, 256, 0, s>>>(h->P[h->pcur].uid, gop, np, nlut, G, lut);
        h->st.kernel_launches++;
    }
    k_st_cell_group<<<gx, 256, 0, s>>>(h->last.assign, N, lut, nlut, G, group);
    h->st.kernel_launches += 2;
    CKL(h);
    StXf xf{};
    if (h->last.scaled && h->last.colmask) { // raw full rows: the clustering columns are transformed forth and back
        xf.scale = h->d_scale + 2 * CCB_MAX_D, xf.shift = h->d_scale + 3 * CCB_MAX_D, xf.mask = h->last.colmask, xf.fwd = 1;
    } else if (h->last.scaled) { // the scaled rows the engine read: transformed back
        xf.scale = h->d_scale, xf.shift = h->d_scale + CCB_MAX_D, xf.mask = ~0ull >> (64 - h->D);
    }
    return group_stats_run(h, s, h->last.X, h->last.dtype, N, h->last.ld, h->last.W, group, G + 1, nq, q, xf,
                           h->last.raw_tx ? h->d_cof.p : nullptr, count, mean,
                           median, quant);
}

} // extern "C"
