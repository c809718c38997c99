// engine.cuh -- KERNEL 2, second generation: the BLOCK-SPECULATIVE VERSIONED COMMIT ("BSV").
//
// Replaces the ordered per-cell loop of HDDStream.online_microcluster_maintenance
// (clustering/hddstream.py:220-237: _add_to_pcore :288-343, _add_to_outlier :345-395,
// _upgrade_outlier_microcluster :397-430, _create_new_outlier_cluster :434-462, with the Microcluster maths
// of objects/microcluster.py:89-153, 213-233 and utilities/mc_functions.py:14-56) -- bit for bit, but with
// the work of a block of B consecutive cells spread over the whole GPU.  tests/proto/bsv_proto.c is the
// CPU model of exactly this scheme (validated against the reference's golden vectors).
//
// A cell's decision is a target KEY:  j < Mp                  absorbed by pcore MC j
//                                     Mp + o  (o < Mo0)       absorbed by outlier MC o of the snapshot
//                                     KNEW + c (c <= i)       absorbed by the MC that cell c of this block
//                                                             creates (c == i: the cell itself creates it)
// with KNEW = Mp + Mo0.  One block runs
//   S   k_bs_spec      speculate from the snapshot: nearest feasible pcore MC (candidate), SAFE / CONTESTED (+ the
//                      snapshot's verdict as a prediction for the replay); it also hands out the top-K slots of the cells
//                      that may reach the outlier stage and counts the candidates per (tile, pcore MC) for round 1
//       k_nearest      top-K of the snapshot outlier list for those cells (kernel 1, nearest.cuh)
//       k_bs_spec_o    speculated outlier decision
//   then up to ITMAX rounds of
//   L   k_bs_tilecnt / k_bs_pscan / k_bs_pscatter   ordered candidate list of every pcore MC
//   C   k_bs_chain_p   per pcore MC, its candidates in input order: CF1 += x, CF2 += x*x, W += 1 as dependent
//                      fp64 adds (the only inherently serial work: ~1 DADD latency per cell); CONTESTED cells
//                      take the radius test in place (a division-free fast test, the exact one when that cannot
//                      call it; runs of them two per step or eight per pass along predicted verdicts); the state
//                      after every absorb is kept (VERSION)
//       k_bs_olist     sort (key, cell) of the pcore-rejected cells -> outlier-side chains
//       k_bs_chain_o   the same replay for modified snapshot outlier MCs and MCs created in this block
//   D   k_bs_derive_p / k_bs_derive_o   centroid, preference mask, radius^2 of every version (cell-parallel)
//   V   k_bs_verify_p  every cell recomputes its pcore decision against the version every pcore MC had just
//       k_bs_verify_o  before it; rejected cells recompute the outlier decision (nearest unmodified snapshot
//                      MC from the top-K list -- or the bound its last entry gives when all of them are stale --
//                      against every modified / created MC at its version)
//   M   k_bs_decide    first cell whose exact decision differs from the speculation = end of the exact
//                      prefix (induction: every earlier cell saw exact versions).  The recomputed decisions
//                      become the next speculation; if they only move cells between outlier-side keys the next
//                      round re-runs the outlier side alone (LIGHT round); an upgrade ends the block at that cell.
//   and finally k_bs_commit writes the exact prefix back (rows, per-cell results, then the block's bookkeeping).
// All control flow lives in device memory (BsCtl): the whole loop of one ingest call is one CUDA graph with two
// device-driven WHILE nodes (api.cu: build_graph), inside which   kernel 1 + S_o  ||  L + C_p   and then
// D_p + V_p  ||  olist + C_o + D_o   run as parallel branches (disjoint data).
#pragma once
#include <limits.h>

#include "common.cuh"
#include "online.cuh"

namespace ccb {

constexpr int BS_KEY_NONE = -4;    // no outlier-side decision recorded
constexpr int BS_KEY_NEED = -3;    // reaches the outlier stage but has no top-K list yet
constexpr int BS_KEY_PENDING = -5; // rejected by the pcore stage in V, outlier stage not evaluated yet
constexpr int BS_KEY_UNKNOWN = -1; // every listed snapshot candidate was modified earlier in the block
constexpr int BS_RMAX = 4096;      // cells per block that may reach the outlier stage
constexpr int BS_TOPK = 8;
constexpr int BS_COLD_B = 512;     // length of a block that starts without any microcluster
// plist entry = cell | flags: CONTESTED (exact radius test inside the chain) and, for a CONTESTED cell, the PREDICTED verdict
// of that test (the snapshot's in round 1, the previous round's afterwards) -- a hint for the replay, never a result
constexpr int BS_PL_CONT = (int)0x80000000, BS_PL_PREJ = 0x40000000, BS_PL_CELL = 0x3fffffff;

struct BsCtl {
    int64_t N, pos;
    int32_t Bcur, Beff, next_B, Bmin, Bmax;
    int32_t active, phase, it, itmax; // phase 0: iterating, 1: commit pending
    int32_t Mp, Mo0;
    int32_t nneed, tk_lo, tk_hi; // need-list length; range of entries whose top-K list is to be computed
    int32_t nneed_raw;           // slots k_bs_spec asked for (more than BS_RMAX: its last CTA re-does the list in cell order)
    int32_t nh, hnew0, no;       // hot outlier-side keys, index of the first created-in-block key, members
    int32_t npend;
    int32_t m_commit, upgrade;
    int32_t need_grow, done;
    int32_t ticket; // k_bs_pscan: CTAs finished (last one computes the key offsets)
    int32_t ticket_o; // k_bs_olist: likewise (the last one builds the key segments)
    int32_t ticket_c; // k_bs_commit: likewise (the last one finishes the block)
    int32_t ticket_s; // k_bs_spec: likewise (the last one closes the need list)
    int32_t tc_done;  // the per-(tile, key) candidate counts of round 1 were made by k_bs_spec (k_bs_tilecnt has nothing to do)
    int32_t o_big;    // outlier-side keys of this round with more members than a CTA of k_bs_chain_o derives itself
    int32_t m_exact;  // cells below this are exact since an earlier round of the block (first mismatch of the previous round)
    int32_t pclean; // refinement round whose pcore side (candidates, CONTESTED flags, accepts) is that of the round before
    int32_t m0, up0; // this round: first cell whose exact decision differs from the speculation / first upgrading cell
                     // (atomicMin by the verify kernels, consumed and reset by k_bs_decide; INT_MAX = none)
    int64_t blocks, iters, mismatches, cuts_unknown, cuts_iter, cuts_cap, tk_late, rejects, replayed, pairs;
    int64_t rounds_light; // refinement rounds that re-ran the outlier side only
    int64_t serial_cells; // sum over the pcore replays of the LONGEST chain's members: the dependent-add floor of kernel 2
};

struct BsWs {
    int32_t *pcand, *ospec, *tkpos, *dec, *eff, *newrank, *pend, *plist;
    int32_t *pbest; // [bmax] nearest feasible pcore MC at the exact versions (k_bs_verify_p), for cells the pcore stage rejects
    uint8_t *pflag, *prej, *upf;
    double *ver;  // [bmax][lsp] VERSION records: CF1 at [0, D), CF2 at [dp, dp + D), W at [2 dp]; lsp = 2 dp + 2
    double *vcen, *vr2;
    uint64_t *vmask;
    int32_t *tilecnt, *tbase, *poff; // [ntiles + 1][mp_stride], [ntiles + 1][mp_stride], [mp_stride + 1]
    int32_t *pcnt;                   // [mp_stride + 1] candidates of every pcore key (poff is padded to multiples of 4)
    double *xg;                      // [bmax + 4 * mp_stride][lsp] ADDEND records in plist order: x, x*x, 1.0 (layout of ver)
    double *verp;                    // [bmax + 4 * mp_stride][lsp] VERSION records of the pcore chains, in plist order
    int32_t *vpos;                   // [bmax] plist position of every pcore candidate
    int32_t *nrows, *ncell;          // [BS_RMAX] absolute row / block-relative cell of the need list
    double *tk_dist;
    int32_t *tk_idx; // [BS_RMAX][BS_TOPK]
    int32_t *hkey, *hoff, *omem, *hrank; // hrank[h]: real creations before created-in-block key h (h >= hnew0; hrank[nh]: all)
    int32_t *hfirst;                     // [BS_RMAX + 1] first member of every outlier-side key
    unsigned long long *okeys;           // [BS_RMAX] (key, cell) of the pcore-rejected cells, sorted (k_bs_olist)
    int32_t *firstmember; // [O.cap], INT_MAX = unmodified in this block
    int64_t *dbg; // optional [mp_stride][8] per-key cycle counters of k_bs_chain_p (diagnostics), or nullptr
    int32_t mp_stride, bmax, dp, lsp;
};
__device__ __forceinline__ double *ver_cf1(const BsWs &w, int i) { return w.ver + (size_t)i * w.lsp; }
__device__ __forceinline__ double *ver_cf2(const BsWs &w, int i) { return w.ver + (size_t)i * w.lsp + w.dp; }
__device__ __forceinline__ double &ver_w(const BsWs &w, int i) { return w.ver[(size_t)i * w.lsp + 2 * w.dp]; }
// VERSION record of a member of a PCORE chain: where k_bs_chain_p's bulk store left it (plist order)
__device__ __forceinline__ const double *pver(const BsWs &w, int i) { return w.verp + (size_t)w.vpos[i] * w.lsp; }

// What changes from one ccb_ingest call to the next.  Stream launches pass it inside Eng; CUDA-graph launches (whose
// kernel arguments are baked in) read it from device memory through Eng::io.
struct EngIo {
    const double *X; // first two fields = XRef (kernel 1 reads them through the same pointer)
    int64_t ld;
    int32_t *assign;
    uint8_t *stage;
    double theta; // SAFE needs: snapshot distance <= theta (+inf: no distance condition) ...
    double r2safe; // ... and snapshot radius^2 of the tentative MC <= r2safe (a margin below eps^2)
    double r2rej;  // snapshot radius^2 above this: speculate REJECTED without entering the chain (+inf: never)
    Num nm;
};

struct Eng {
    const double *X;
    int64_t ld;
    Store P, O;
    Num nm;
    Ctl *ctl;
    BsCtl *bc;
    BsWs ws;
    int32_t *assign;
    uint8_t *stage;
    double theta, r2safe, r2rej;
    const EngIo *io;                 // nullptr: the fields above are current
    unsigned long long h_outer, h_inner; // cudaGraphConditionalHandle of the block loop / round loop, 0 = stream launches
    __device__ __forceinline__ void fetch() {
        if (io) {
            X = io->X;
            ld = io->ld;
            assign = io->assign;
            stage = io->stage;
            theta = io->theta;
            r2safe = io->r2safe;
            r2rej = io->r2rej;
            nm = io->nm;
        }
    }
};

// ---------------------------------------------------------------------------------------------------
// thread-sequential arithmetic (one thread, dimensions in index order)

template <int DP>
__device__ __forceinline__ void load_row(const double *row, int D, double (&x)[DP]) {
#pragma unroll
    for (int d = 0; d < DP; ++d) x[d] = d < D ? row[d] : 0.0;
}

// mc_functions.py:35-43 with the cell in registers
template <int DP>
__device__ __forceinline__ double dist_regs(const double (&x)[DP], const double *__restrict__ c, uint64_t mask,
                                            const Num &nm) {
    double acc = 0.0;
#pragma unroll
    for (int d = 0; d < DP; ++d) {
        if (d < nm.D) {
            double t = dsub(x[d], c[d]);
            t = dmul(t, t);
            if ((mask >> d) & 1ull) t = nm.div_mode ? ddiv(t, nm.k) : dmul(t, nm.wsel);
            acc = dadd(acc, t);
        }
    }
    return acc;
}

// get_copy_with_new_point + calculate_projected_radius_squared (microcluster.py:213-233, mc_functions.py:45-56)
// by one thread.  Returns r^2; wn = W + 1, nmask = preference mask of the tentative MC.
template <int DP>
__device__ __forceinline__ double tent_regs(const double *__restrict__ cf1, const double *__restrict__ cf2, double w,
                                            const double (&x)[DP], const Num &nm, double &wn, uint64_t &nmask) {
    wn = dadd(w, 1.0);
    double s = 0.0;
    uint64_t mk = 0ull;
#pragma unroll
    for (int d = 0; d < DP; ++d) {
        if (d < nm.D) {
            const double c1 = dadd(cf1[d], x[d]);
            const double c2 = dadd(cf2[d], dmul(x[d], x[d]));
            const double a = ddiv(c2, wn);
            const double c = ddiv(c1, wn);
            const double var = dsub(a, dmul(c, c));
            const bool bit = var <= nm.delta2;
            mk |= (uint64_t)bit << d;
            s = dadd(s, bit ? (nm.div_mode ? ddiv(var, nm.k) : dmul(var, nm.wsel)) : var);
        }
    }
    nmask = mk;
    return s;
}

// feasibility gate of _add_to_pcore (hddstream.py:315-321) with the cell in registers
template <int DP>
__device__ __forceinline__ bool feasible_regs(const double *__restrict__ cf1, const double *__restrict__ cf2, double w,
                                              const double (&x)[DP], const Num &nm) {
    const double w1 = dadd(w, 1.0);
    int cnt = 0;
#pragma unroll
    for (int d = 0; d < DP; ++d) {
        if (d < nm.D) {
            const double a = ddiv(dadd(cf2[d], dmul(x[d], x[d])), w1);
            double b = ddiv(dadd(cf1[d], x[d]), w1);
            b = dmul(b, b);
            cnt += (dsub(a, b) <= nm.delta2);
        }
    }
    return (int64_t)cnt <= nm.pi;
}

__device__ __forceinline__ unsigned lanemask_lt() { return (1u << (threadIdx.x & 31)) - 1u; }

// latest element < i of the ascending list l[0..n), or -1
__device__ __forceinline__ int latest_before(const int32_t *__restrict__ l, int n, int i) {
    int lo = 0, hi = n;
    while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        if (l[mid] < i) lo = mid + 1;
        else hi = mid;
    }
    return lo ? l[lo - 1] : -1;
}

// ---------------------------------------------------------------------------------------------------
__global__ void k_bs_init(BsCtl *bc, int64_t N, int32_t itmax, int32_t bmin, int32_t bmax) {
    bc->N = N;
    bc->pos = 0;
    bc->done = N <= 0;
    bc->need_grow = 0;
    bc->active = 0;
    bc->itmax = itmax;
    bc->Bmin = bmin;
    bc->Bmax = bmax;
    if (bc->next_B < bmin) bc->next_B = bmin;
    if (bc->next_B > bmax) bc->next_B = bmax;
}

__global__ void k_bs_begin(Eng e) {
    e.fetch();
    CCB_TS(0);
    CCB_PDL();
    BsCtl *bc = e.bc;
    bc->active = 0;
    bc->tk_lo = bc->tk_hi = 0; // an idle block must not leave kernel 1 any work
    bc->m0 = bc->up0 = INT_MAX;
    do {
        if (bc->done || bc->need_grow) break;
        if (bc->pos >= bc->N) {
            bc->done = 1;
            break;
        }
        const int Mp = e.ctl->n_pcore, Mo0 = e.ctl->n_outlier;
        if ((int64_t)Mo0 + BS_RMAX + 1 > e.O.cap) {
            bc->need_grow = 1;
            break;
        }
        if (Mp + 1 > e.P.cap || Mp + 1 > e.ws.mp_stride) {
            bc->need_grow = 2;
            break;
        }
        const int64_t left = bc->N - bc->pos;
        // no microcluster at all (the first cells of a run): every cell of the block would be checked against every MC the
        // cells in front of it may create -- quadratic in the block length -- while the exact prefix grows by a few hundred
        // cells per block at best; a short block costs a quarter per round
        const int32_t want = (Mp + Mo0 == 0) ? min(bc->next_B, BS_COLD_B) : bc->next_B;
        bc->Bcur = (int32_t)(left < want ? left : want);
        bc->Beff = bc->Bcur;
        bc->Mp = Mp;
        bc->Mo0 = Mo0;
        bc->nneed = 0;
        bc->nneed_raw = 0;
        bc->tc_done = 0;
        bc->nh = bc->hnew0 = bc->no = 0;
        bc->npend = 0;
        bc->it = 0;
        bc->phase = 0;
        bc->m_commit = 0;
        bc->upgrade = 0;
        bc->pclean = 0;
        bc->m_exact = 0;
        bc->active = 1;
    } while (0);
    // graph launches: the round loop runs iff the block is active; an idle block also ends the block loop
    if (e.h_inner) cudaGraphSetConditional(e.h_inner, bc->active ? 1u : 0u);
    if (e.h_outer && !bc->active) cudaGraphSetConditional(e.h_outer, 0u);
}

// ---- S ----------------------------------------------------------------------------------------------
constexpr int BS_THREADS = 128;

// BS_SPLIT lanes share one cell: lane p of the group scans pcore MCs p, p + BS_SPLIT, ... and the group reduces
// (distance, list position) lexicographically -- the first strictly smaller MC of the sequential scan.  The grid of
// one block is small (32 768 cells); splitting the MC axis quadruples the warps that hide the dependent-add latency.
constexpr int BS_SPLIT = 4;

__device__ __forceinline__ void group_argmin(double &d, int &j) { // over BS_SPLIT adjacent lanes; j < 0: no candidate
#pragma unroll
    for (int o = 1; o < BS_SPLIT; o <<= 1) {
        const double od = __shfl_xor_sync(0xffffffffu, d, o);
        const int oj = __shfl_xor_sync(0xffffffffu, j, o);
        if (oj >= 0 && (j < 0 || od < d || (od == d && oj < j))) {
            d = od;
            j = oj;
        }
    }
}

constexpr int BS_CTA1 = 1024;

__device__ __forceinline__ int block_exclusive_scan_1024(int v, int *s_warp, int &total) {
    // inclusive scan inside the warp, then across the 32 warp totals
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    int inc = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const int t = __shfl_up_sync(0xffffffffu, inc, o);
        if (lane >= o) inc += t;
    }
    if (lane == 31) s_warp[warp] = inc;
    __syncthreads();
    if (warp == 0) {
        int w = s_warp[lane];
        int winc = w;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int t = __shfl_up_sync(0xffffffffu, winc, o);
            if (lane >= o) winc += t;
        }
        s_warp[lane] = winc - w;   // exclusive offset of each warp
        if (lane == 31) s_warp[32] = winc; // grand total
    }
    __syncthreads();
    total = s_warp[32];
    const int r = s_warp[warp] + inc - v;
    __syncthreads();
    return r;
}

template <int NT>
__device__ __forceinline__ int block_exclusive_scan_t(int v, int *s_warp, int &total) { // NT threads, NT / 32 <= 32 warps
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    int inc = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const int t = __shfl_up_sync(0xffffffffu, inc, o);
        if (lane >= o) inc += t;
    }
    if (lane == 31) s_warp[warp] = inc;
    __syncthreads();
    if (warp == 0) {
        const int w = lane < NT / 32 ? s_warp[lane] : 0;
        int winc = w;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int t = __shfl_up_sync(0xffffffffu, winc, o);
            if (lane >= o) winc += t;
        }
        s_warp[lane] = winc - w;
        if (lane == 31) s_warp[32] = winc;
    }
    __syncthreads();
    total = s_warp[32];
    const int r = s_warp[warp] + inc - v;
    __syncthreads();
    return r;
}

// Ordered need list (the rare case: more than BS_RMAX cells of the block are not SAFE): slots are handed out again in
// cell order and the block is truncated at the first cell that does not fit (bounds the outlier-stage work of one block).
// Runs in the last CTA of k_bs_spec (NT threads).
template <int NT>
__device__ __forceinline__ void bs_need_ordered(const Eng &e, BsCtl *bc, int *s_warp, int *s_cut) {
    const int B = bc->Bcur, tid = threadIdx.x;
    const int per = (B + NT - 1) / NT;
    const int lo = min(B, tid * per), hi = min(B, lo + per);
    if (tid == 0) *s_cut = B;
    int cnt = 0;
    for (int i = lo; i < hi; ++i) cnt += e.ws.pflag[i] != 0;
    int total;
    int base = block_exclusive_scan_t<NT>(cnt, s_warp, total);
    const int32_t row0 = (int32_t)bc->pos;
    for (int i = lo; i < hi; ++i) {
        if (!e.ws.pflag[i]) continue;
        if (base < BS_RMAX) {
            e.ws.tkpos[i] = base;
            e.ws.nrows[base] = row0 + i;
            e.ws.ncell[base] = i;
        } else {
            e.ws.tkpos[i] = -1;
            if (base == BS_RMAX) *s_cut = i; // exactly one thread sees the first overflowing cell
        }
        ++base;
    }
    __syncthreads();
    if (tid == 0) {
        bc->Beff = *s_cut;
        bc->nneed = min(total, BS_RMAX);
    }
}

// S: one CTA = one tile of 32 cells, BS_SPLIT lanes per cell.  Besides the speculation itself the kernel hands out the
// top-K slots of the cells that are not SAFE, counts the tile's candidates per pcore key (k_bs_tilecnt's work in the first
// round) and, in its last CTA, closes the need list -- three launches of round 1 folded into this one.
template <int DP>
__global__ void __launch_bounds__(BS_THREADS, DP <= 16 ? 7 : 1) k_bs_spec(Eng e) {
    e.fetch();
    CCB_TS(1);
    CCB_PDL();
    __shared__ int s_warp[33];
    __shared__ int s_last, s_cut;
    BsCtl *bc = e.bc;
    if (!bc->active) return;
    const int Bcur = bc->Bcur;
    if ((int)blockIdx.x * (BS_THREADS / BS_SPLIT) >= Bcur) return; // (whole CTAs)
    const int gt = blockIdx.x * BS_THREADS + threadIdx.x;
    const int i = gt / BS_SPLIT, part = gt % BS_SPLIT;
    const bool live = i < Bcur;
    const Num nm = e.nm;
    const int D = nm.D, Mp_all = bc->Mp, Mp = live ? Mp_all : 0;
    // this tile's row of the per-(tile, key) candidate counts
    int32_t *trow = e.ws.tilecnt + (size_t)blockIdx.x * e.ws.mp_stride;
    for (int j = threadIdx.x; j < Mp_all; j += BS_THREADS) trow[j] = 0;
    __syncthreads();
    double x[DP];
    load_row<DP>(e.X + (bc->pos + (live ? i : 0)) * e.ld, D, x);
    int best = -1;
    double bd = 0.0;
    for (int j = part; j < Mp; j += BS_SPLIT) {
        if (nm.pi_active && !feasible_regs<DP>(e.P.cf1 + (size_t)j * D, e.P.cf2 + (size_t)j * D, e.P.w[j], x, nm)) continue;
        const double dv = dist_regs<DP>(x, e.P.cen + (size_t)j * D, e.P.mask[j], nm);
        if (!(dv != dv) && (best < 0 || dv < bd)) {
            best = j;
            bd = dv;
        }
    }
    group_argmin(bd, best); // (every lane of the group holds the result)
    // radius^2 of the tentative MC (microcluster.py:213-233, mc_functions.py:45-56) on the snapshot: the group's lanes share
    // the 2 D divisions (lane p: dimensions p, p + BS_SPLIT, ...), lane 0 sums the terms in index order
    const int lane = threadIdx.x & 31, gbase = lane & ~(BS_SPLIT - 1);
    constexpr int TPL = (DP + BS_SPLIT - 1) / BS_SPLIT;
    double term[TPL];
    {
        const int b = best >= 0 ? best : 0;
        const double *cf1 = e.P.cf1 + (size_t)b * D, *cf2 = e.P.cf2 + (size_t)b * D;
        const double wn = dadd(best >= 0 ? e.P.w[b] : 0.0, 1.0);
#pragma unroll
        for (int u = 0; u < TPL; ++u) {
            const int d = part + u * BS_SPLIT;
            double t = 0.0;
            if (d < D && best >= 0) {
                // (x is a register array: select the coordinate without dynamic indexing)
                double xv = 0.0;
#pragma unroll
                for (int dd = 0; dd < DP; ++dd)
                    if (dd == d) xv = x[dd];
                const double a = ddiv(dadd(cf2[d], dmul(xv, xv)), wn);
                const double c = ddiv(dadd(cf1[d], xv), wn);
                const double var = dsub(a, dmul(c, c));
                t = (var <= nm.delta2) ? (nm.div_mode ? ddiv(var, nm.k) : dmul(var, nm.wsel)) : var;
            }
            term[u] = t;
        }
    }
    double r2s = 0.0;
#pragma unroll
    for (int d = 0; d < DP; ++d) {
        const double t = __shfl_sync(0xffffffffu, term[d / BS_SPLIT], gbase + (d % BS_SPLIT));
        if (d < D) r2s = dadd(r2s, t);
    }
    const bool mine = part == 0 && live;
    int flag = mine ? 1 : 0;
    if (mine && best >= 0) {
        if (bd <= e.theta && r2s <= e.r2safe) {
            flag = 0;
        } else {
            if (r2s > nm.eps2) flag = 3; // CONTESTED, and the snapshot predicts "rejected" (bit 1: BS_PL_PREJ in plist)
            // far beyond the radius limit on the snapshot: speculate "rejected by the pcore stage" right away instead of
            // sending the cell through the serial chain for an exact test; k_bs_verify_p checks it like everything else
            if (r2s > e.r2rej) best = -1;
        }
    }
    // need list: every cell that is not SAFE takes a top-K slot right here (one atomic per warp; the order of the slots
    // is immaterial).  Should the block need more than BS_RMAX slots, the last CTA hands them out again in cell order and
    // truncates the block (bs_need_ordered).
    const unsigned fm = __ballot_sync(0xffffffffu, flag != 0);
    int slot = -1;
    if (fm) {
        int base = 0;
        if (lane == __ffs(fm) - 1) base = atomicAdd(&bc->nneed_raw, __popc(fm));
        base = __shfl_sync(0xffffffffu, base, __ffs(fm) - 1);
        if (flag) slot = base + __popc(fm & ((1u << lane) - 1u));
    }
    if (mine) {
        e.ws.pcand[i] = best;
        e.ws.pflag[i] = (uint8_t)flag;
        e.ws.prej[i] = best < 0;
        e.ws.ospec[i] = BS_KEY_NONE;
        if (slot >= 0 && slot < BS_RMAX) {
            e.ws.tkpos[i] = slot;
            e.ws.nrows[slot] = (int32_t)bc->pos + i;
            e.ws.ncell[slot] = i;
        } else {
            e.ws.tkpos[i] = -1;
        }
        if (best >= 0) atomicAdd(&trow[best], 1);
    }
    // ---- the last CTA of the block closes the need list
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) s_last = atomicAdd(&bc->ticket_s, 1) == (Bcur + BS_THREADS / BS_SPLIT - 1) / (BS_THREADS / BS_SPLIT) - 1;
    __syncthreads();
    if (!s_last) return;
    __threadfence();
    const int raw = *(volatile int32_t *)&bc->nneed_raw;
    if (raw <= BS_RMAX) { // the usual case: the slots handed out above stand
        if (threadIdx.x == 0) {
            bc->Beff = Bcur;
            bc->nneed = raw;
            bc->tc_done = 1; // the tile counts above are those of the whole block
        }
    } else {
        bs_need_ordered<BS_THREADS>(e, bc, s_warp, &s_cut);
    }
    if (threadIdx.x == 0) {
        bc->ticket_s = 0;
        bc->tk_lo = 0;
        bc->tk_hi = bc->nneed;
        bc->rejects += bc->nneed;
        bc->pairs += (int64_t)bc->nneed * bc->Mo0;
    }
}

// speculated outlier-stage decision of the need list: nearest snapshot MC + radius test on the snapshot state
__global__ void __launch_bounds__(BS_THREADS) k_bs_spec_o(Eng e) {
    e.fetch();
    CCB_TS(5);
    CCB_PDL();
    const BsCtl *bc = e.bc;
    if (!bc->active || bc->phase != 0 || bc->it != 0) return; // first round of a block only
    const int t = blockIdx.x * BS_THREADS + threadIdx.x;
    if (t >= bc->nneed) return;
    const int i = e.ws.ncell[t];
    const Num nm = e.nm;
    const int D = nm.D;
    const int KNEW = bc->Mp + bc->Mo0;
    int key = KNEW + i;
    const int o = bc->Mo0 > 0 ? e.ws.tk_idx[(size_t)t * BS_TOPK] : -1;
    if (o >= 0) {
        const double *x = e.X + (bc->pos + i) * e.ld;
        const double *cf1 = e.O.cf1 + (size_t)o * D, *cf2 = e.O.cf2 + (size_t)o * D;
        const double wn = dadd(e.O.w[o], 1.0);
        double s = 0.0;
        for (int d = 0; d < D; ++d) {
            const double xv = x[d];
            const double a = ddiv(dadd(cf2[d], dmul(xv, xv)), wn);
            const double c = ddiv(dadd(cf1[d], xv), wn);
            const double var = dsub(a, dmul(c, c));
            s = dadd(s, (var <= nm.delta2) ? (nm.div_mode ? ddiv(var, nm.k) : dmul(var, nm.wsel)) : var);
        }
        if (s <= nm.eps2) key = bc->Mp + o;
    }
    e.ws.ospec[i] = key;
}

// ---- L ----------------------------------------------------------------------------------------------
// per (tile of 32 cells, pcore key): number of candidates
__global__ void __launch_bounds__(BS_THREADS) k_bs_tilecnt(Eng e) {
    e.fetch();
    CCB_TS(6);
    CCB_PDL();
    const BsCtl *bc = e.bc;
    if (!bc->active || bc->phase != 0 || bc->pclean) return;
    if (bc->it == 0 && bc->tc_done) return; // round 1 of an untruncated block: k_bs_spec counted
    const int lane = threadIdx.x & 31;
    const int t = blockIdx.x * (BS_THREADS / 32) + (threadIdx.x >> 5);
    const int ntiles = (bc->Beff + 31) >> 5;
    if (t >= ntiles) return;
    const int i = t * 32 + lane;
    const int c = i < bc->Beff ? e.ws.pcand[i] : -1;
    const int Mp = bc->Mp;
    int32_t *row = e.ws.tilecnt + (size_t)t * e.ws.mp_stride;
    for (int j0 = 0; j0 < Mp; j0 += 32) {
        int my = 0;
        const int jn = min(32, Mp - j0);
        for (int jj = 0; jj < jn; ++jj) {
            const unsigned b = __ballot_sync(0xffffffffu, c == j0 + jj);
            if (lane == jj) my = __popc(b);
        }
        if (lane < jn) row[j0 + lane] = my;
    }
}

// per key (one CTA each): exclusive prefix of the tile counts (in place) and the key's total; the last CTA to
// finish turns the totals into the (padded) key offsets
__global__ void __launch_bounds__(BS_CTA1, 1) k_bs_pscan(Eng e) {
    e.fetch();
    CCB_TS(7);
    CCB_PDL();
    __shared__ int s_warp[33];
    __shared__ int s_last, s_max;
    BsCtl *bc = e.bc;
    if (!bc->active || bc->phase != 0 || bc->pclean) return;
    const int Mp = bc->Mp, stride = e.ws.mp_stride;
    const int j = blockIdx.x;
    if (j >= Mp) return;
    const int ntiles = (bc->Beff + 31) >> 5;
    int carry = 0;
    for (int t0 = 0; t0 < ntiles; t0 += BS_CTA1) {
        const int t = t0 + threadIdx.x;
        const int v = t < ntiles ? e.ws.tilecnt[(size_t)t * stride + j] : 0;
        int total;
        const int ex = block_exclusive_scan_1024(v, s_warp, total);
        if (t < ntiles) e.ws.tilecnt[(size_t)t * stride + j] = carry + ex;
        carry += total;
    }
    if (threadIdx.x == 0) {
        e.ws.pcnt[j] = carry;
        __threadfence();
        s_last = atomicAdd(&bc->ticket, 1) == Mp - 1;
    }
    __syncthreads();
    if (!s_last) return;
    __threadfence();
    // exclusive scan of the totals, each rounded up to a multiple of 4 entries so that every key's segment of
    // plist / xg starts 16-byte aligned (bulk-copy requirement of the chain kernel)
    carry = 0;
    if (threadIdx.x == 0) s_max = 0;
    int mx = 0;
    for (int j0 = 0; j0 < Mp; j0 += BS_CTA1) {
        const int jj = j0 + threadIdx.x;
        const int raw = jj < Mp ? ((volatile int32_t *)e.ws.pcnt)[jj] : 0;
        mx = max(mx, raw);
        const int v = (raw + 3) & ~3;
        int total;
        const int ex = block_exclusive_scan_1024(v, s_warp, total);
        if (jj < Mp) e.ws.poff[jj] = carry + ex;
        carry += total;
    }
    mx = __reduce_max_sync(0xffffffffu, mx);
    if ((threadIdx.x & 31) == 0 && mx > 0) atomicMax(&s_max, mx);
    __syncthreads();
    if (threadIdx.x == 0) {
        e.ws.poff[Mp] = carry;
        bc->ticket = 0;
        bc->serial_cells += s_max;
        CCB_DBG(g_trace_ts[21] = s_max;)
    }
}

// plist[pos] = cell | CONTESTED << 31 and xg[pos] = the cell's ADDEND record (x, x*x, 1.0), pos in (key, cell) order.
// One CTA per tile of 32 cells: warp 0 places the cells (lane = cell), then each of the four warps writes eight of the
// records, lane = element of the record (coalesced rows), four records in flight at a time so that the row loads overlap
// instead of paying one global-memory latency per record.
__global__ void __launch_bounds__(BS_THREADS) k_bs_pscatter(Eng e) {
    e.fetch();
    CCB_TS(8);
    CCB_PDL();
    __shared__ int s_pos[32];
    const BsCtl *bc = e.bc;
    if (!bc->active || bc->phase != 0 || bc->pclean) return;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int t = blockIdx.x;
    const int ntiles = (bc->Beff + 31) >> 5;
    if (t >= ntiles) return;
    if (warp == 0) {
        const int i = t * 32 + lane;
        const int c = i < bc->Beff ? e.ws.pcand[i] : -1;
        const unsigned peers = __match_any_sync(0xffffffffu, c);
        int pos = -1;
        if (c >= 0) {
            const int rank = __popc(peers & lanemask_lt());
            pos = e.ws.poff[c] + e.ws.tilecnt[(size_t)t * e.ws.mp_stride + c] + rank;
            const int pf = e.ws.pflag[i];
            e.ws.plist[pos] = i | (pf ? BS_PL_CONT : 0) | ((pf & 2) ? BS_PL_PREJ : 0);
            e.ws.vpos[i] = pos;
        }
        s_pos[lane] = pos;
    }
    __syncthreads();
    const int D = e.nm.D, dp = e.ws.dp, lsp = e.ws.lsp;
    const double *Xt = e.X + (bc->pos + (int64_t)t * 32) * e.ld;
    constexpr int QU = 4, PER = 32 / (BS_THREADS / 32);
    for (int q0 = warp * PER; q0 < (warp + 1) * PER; q0 += QU) {
        int pq[QU];
#pragma unroll
        for (int u = 0; u < QU; ++u) pq[u] = s_pos[q0 + u];
        for (int el0 = 0; el0 < lsp; el0 += 32) {
            const int el = el0 + lane;
            double v[QU];
#pragma unroll
            for (int u = 0; u < QU; ++u) {
                v[u] = 0.0;
                if (pq[u] >= 0 && el < lsp) {
                    const double *src = Xt + (int64_t)(q0 + u) * e.ld;
                    if (el < D) v[u] = src[el];
                    else if (el >= dp && el < dp + D) v[u] = src[el - dp];
                    else if (el == 2 * dp) v[u] = 1.0;
                }
            }
#pragma unroll
            for (int u = 0; u < QU; ++u)
                if (pq[u] >= 0 && el < lsp) {
                    const double x = v[u];
                    e.ws.xg[(size_t)pq[u] * lsp + el] = (el >= dp && el < dp + D) ? dmul(x, x) : x;
                }
        }
    }
}

// ---- C ----------------------------------------------------------------------------------------------
// The replay of a key's members in input order is the only inherently serial work of the whole engine -- one
// dependent DADD per cell and dimension -- so both chain kernels are written for latency: cells are taken eight
// at a time, their coordinates and indices are fetched from shared memory up front, only the CF adds are chained.
// Lane d of the replaying warp owns dimensions d and d + 32.
//
// k_bs_chain_o: OUTLIER-SIDE keys (modified snapshot outlier MCs and MCs created in this block), one CTA per key;
// members are few and scattered, so warps 1-3 gather the next batch with cp.async (index list first, then the
// rows) while warp 0 replays the current one.
__device__ __forceinline__ void derive_version(const Eng &e, const Num &nm, int i, const double *rec); // (section D)

template <int DP>
struct ChainCfg {
    static constexpr int NB = DP <= 16 ? 128 : (DP <= 32 ? 64 : 32);
};
constexpr int BS_CHAIN_PRODUCERS = BS_THREADS - 32;

// one key; every thread of the CTA passes the same 1 + (batches) barriers, so the caller may loop over keys
template <int DP>
__device__ __forceinline__ void bs_chain_o_key(const Eng &e, const BsCtl *bc, int key_idx,
                                               double (&xs)[2][ChainCfg<DP>::NB][DP], int (&mi)[2][ChainCfg<DP>::NB]) {
    constexpr int NB = ChainCfg<DP>::NB;
    constexpr int GS = 8;
    const Num nm = e.nm;
    const int D = nm.D;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int Mp = bc->Mp, KNEW = bc->Mp + bc->Mo0;
    const int32_t *mem;
    int n;
    const double *s1 = nullptr, *s2 = nullptr;
    double w = 0.0;
    mem = e.ws.omem + e.ws.hoff[key_idx];
    n = e.ws.hoff[key_idx + 1] - e.ws.hoff[key_idx];
    {
        const int key = e.ws.hkey[key_idx];
        if (key < KNEW) {
            const int o = key - Mp;
            s1 = e.O.cf1 + (size_t)o * D;
            s2 = e.O.cf2 + (size_t)o * D;
            w = e.O.w[o];
        }
    }
    if (n <= 0) return;
    const double *Xb = e.X + bc->pos * e.ld;
    const bool vec16 = ((D & 1) == 0) && ((e.ld & 1) == 0) && ((reinterpret_cast<uintptr_t>(e.X) & 15) == 0);
    const int nb = (n + NB - 1) / NB;

    // ---- producers: batch b -> buffer b & 1
    auto produce = [&](int b) {
        const int buf = b & 1, cnt = min(NB, n - b * NB);
        const int pt = tid - 32;
        for (int m = pt; m < cnt; m += BS_CHAIN_PRODUCERS) {
            const int i = mem[b * NB + m];
            mi[buf][m] = i;
        }
        asm volatile("bar.sync 1, %0;" ::"n"(BS_CHAIN_PRODUCERS) : "memory");
        if (vec16) {
            const int hd = D >> 1;
            for (int idx = pt; idx < cnt * hd; idx += BS_CHAIN_PRODUCERS) {
                const int m = idx / hd, d2 = (idx - m * hd) * 2;
                asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(smem_u32(&xs[buf][m][d2])),
                             "l"(Xb + (int64_t)mi[buf][m] * e.ld + d2)
                             : "memory");
            }
        } else {
            for (int idx = pt; idx < cnt * D; idx += BS_CHAIN_PRODUCERS) {
                const int m = idx / D, d = idx - m * D;
                cp_async8(&xs[buf][m][d], Xb + (int64_t)mi[buf][m] * e.ld + d);
            }
        }
        asm volatile("cp.async.commit_group;\ncp.async.wait_group 0;" ::: "memory");
    };

    if (warp != 0) {
        produce(0);
        __syncthreads();
        for (int b = 0; b < nb; ++b) {
            if (b + 1 < nb) produce(b + 1);
            __syncthreads();
        }
        return;
    }

    // ---- consumer (warp 0): lane = element of the VERSION record (CF1 | CF2 | W, the layout of ver), as in
    // k_bs_chain_p: absorbing a cell is ONE dependent add for the lane that owns the element and one coalesced store of the
    // record to ver[cell]; the addend of a CF2 lane is x * x (off the chain).  (Round 1 kept one dimension per lane: three
    // adds, three scattered stores and their address arithmetic per member -- 40 us for the 2 000-member keys of the cold
    // start, with 12 of 32 lanes busy.)
    constexpr int LSP = 2 * DP + 2, NE = (2 * DP + 1 + 31) / 32; // elements per lane
    double v[NE];
    int src[NE];  // which coordinate of the cell feeds element e (-1: the weight lane, addend 1.0; -2: idle)
    bool sq[NE];
#pragma unroll
    for (int h = 0; h < NE; ++h) {
        const int el = lane + 32 * h;
        src[h] = -2;
        sq[h] = false;
        v[h] = 0.0;
        if (el < D) {
            src[h] = el;
            v[h] = s1 ? s1[el] : 0.0;
        } else if (el >= DP && el < DP + D) {
            src[h] = el - DP;
            sq[h] = true;
            v[h] = s2 ? s2[el - DP] : 0.0;
        } else if (el == 2 * DP) {
            src[h] = -1;
            v[h] = w;
        }
    }
    // (the warp issues in order: addresses and addends are made before the dependent adds start, and the lane's base
    // pointer is held in an opaque register so that it is not re-derived from special registers per member)
    double *ver_lane = e.ws.ver + lane;
    asm volatile("" : "+l"(ver_lane));
    bool st[NE];
#pragma unroll
    for (int h = 0; h < NE; ++h) st[h] = src[h] != -2;
    __syncthreads(); // batch 0 staged
    for (int b = 0; b < nb; ++b) {
        const int cur = b & 1;
        const int cnt = min(NB, n - b * NB);
        for (int m0 = 0; m0 < cnt; m0 += GS) {
            const int g = min(GS, cnt - m0);
            double *rec[GS];
            double a[GS][NE];
#pragma unroll
            for (int q = 0; q < GS; ++q) {
                const int mq = min(m0 + q, cnt - 1); // (past the end of a ragged group: a valid slot, never stored)
                rec[q] = ver_lane + (size_t)mi[cur][mq] * LSP;
#pragma unroll
                for (int h = 0; h < NE; ++h) {
                    const double x = src[h] >= 0 ? xs[cur][mq][src[h]] : 1.0;
                    a[q][h] = sq[h] ? dmul(x, x) : x;
                    asm volatile("" : "+d"(a[q][h]));
                }
                asm volatile("" : "+l"(rec[q]));
            }
            if (g == GS) {
#pragma unroll
                for (int q = 0; q < GS; ++q)
#pragma unroll
                    for (int h = 0; h < NE; ++h) {
                        v[h] = dadd(v[h], a[q][h]);
                        if (st[h]) rec[q][32 * h] = v[h];
                    }
            } else {
#pragma unroll
                for (int q = 0; q < GS - 1; ++q)
                    if (q < g) { // warp-uniform
#pragma unroll
                        for (int h = 0; h < NE; ++h) {
                            v[h] = dadd(v[h], a[q][h]);
                            if (st[h]) rec[q][32 * h] = v[h];
                        }
                    }
            }
        }
        __syncthreads();
    }
}

template <int DP>
__global__ void __launch_bounds__(BS_THREADS) k_bs_chain_o(Eng e) {
    e.fetch();
    CCB_TS(13);
    CCB_PDL();
    __shared__ __align__(16) double xs[2][ChainCfg<DP>::NB][DP];
    __shared__ int mi[2][ChainCfg<DP>::NB];
    const BsCtl *bc = e.bc;
    if (!bc->active || bc->phase != 0) return;
    const int nh = bc->nh;
    for (int key_idx = blockIdx.x; key_idx < nh; key_idx += gridDim.x) {
        bs_chain_o_key<DP>(e, bc, key_idx, xs, mi);
        // D (derive) of this key's versions right here when the key is small -- the steady state: one to three members per
        // key -- so that k_bs_derive_o has nothing left to do; a key with more members than the CTA has threads is left
        // to that kernel, which spreads them over the whole GPU (the CTA is in step here: see bs_chain_o_key)
        const int off = e.ws.hoff[key_idx], n = e.ws.hoff[key_idx + 1] - off;
        if (n <= BS_THREADS) {
            if ((int)threadIdx.x < n) {
                const int i = e.ws.omem[off + threadIdx.x];
                derive_version(e, e.nm, i, e.ws.ver + (size_t)i * e.ws.lsp);
            }
        } else if (threadIdx.x == 0) {
            atomicAdd(&e.bc->o_big, 1);
        }
    }
}

// k_bs_chain_p: PCORE keys (CONTESTED members take the exact radius test in place).  The candidates of a key lie
// CONTIGUOUSLY in plist / xg (k_bs_pscatter) as ADDEND records a = (x, x*x, 1.0), and an MC is the record
// v = (CF1, CF2, W): absorbing a cell is v += a, element-wise -- ONE dependent DADD per cell for the lane that
// owns the element.  Three warps, specialised:
//   producer  one thread streams the records through a ring of shared-memory stages with 1-D bulk TMA copies
//             (cp.async.bulk + mbarrier complete_tx);
//   replay    warp 0, lane = record element: a <- LDS, v += a, v -> STS over the addend it just consumed (the stage
//             now holds the VERSION after every cell);
//   store     one thread sends every finished stage -- 64 consecutive VERSION records of the key -- to verp[plist position]
//             with ONE bulk TMA store and releases the stage (k_bs_derive_p hands the records on to ver[cell], cell-parallel).
// A single warp cannot hide instruction latency, so everything that is not the dependent add lives elsewhere, and the
// replay code itself is written for in-order issue: one LDS and one STS hide in the shadow of every dependent DADD.
__device__ __forceinline__ void mbar_arrive(uint64_t *bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void tma_store_1d(void *dst_gmem, const void *src_smem, uint32_t bytes) {
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(dst_gmem), "r"(smem_u32(src_smem)),
                 "r"(bytes)
                 : "memory");
}

__device__ __forceinline__ double lds_f64(uint32_t a) {
    double v;
    asm volatile("ld.shared.f64 %0, [%1];" : "=d"(v) : "r"(a));
    return v;
}
__device__ __forceinline__ void sts_f64(uint32_t a, double v) {
    asm volatile("st.shared.f64 [%0], %1;" ::"r"(a), "d"(v) : "memory");
}
__device__ __forceinline__ int4 lds_v4(uint32_t a) {
    int4 v;
    asm volatile("ld.shared.v4.s32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(a));
    return v;
}

template <int DP>
struct ChainPCfg {
    static constexpr int LSP = 2 * DP + 2;
    static constexpr int NH = (LSP + 31) / 32;
    static constexpr int NB = DP <= 16 ? 64 : 32;
    static constexpr int S = DP <= 48 ? 8 : 6;
    static constexpr size_t SMEM = (size_t)S * NB * (LSP * 8 + 4) + 3 * S * 8 + 2 * DP * 8 + 128;
};
// warp 0 replays, lane 0 of warp 1 streams the addends in, lane 0 of warp 2 streams the versions out, warp 4 (the replay
// warp's scheduler) warms the instruction cache of the rare path and exits; warp 3 only fills the CTA up
constexpr int BS_CHAINP_THREADS = 160;

// Exact radius test of the tentative MC nv = v + a (mc_functions.py:45-56) for a CONTESTED cell, by the whole replay
// warp (lane = record element).  Deliberately NOT inlined: the replay warp runs alone on its scheduler, so every cold
// instruction-cache line it touches is a full miss it cannot hide; one small shared copy keeps the footprint of the
// rare path at a few hundred instructions.  NH == 1: the record is one register per lane (nv0); otherwise it is read
// back from the stage at rec_addr (this lane's element 0 of the record, shared-window address).
// Lane d computes the d-th term (two IEEE divisions, off each other's critical path); the D terms are then summed in index
// order by every lane from warp shuffles -- no memory round trip; with D == DP the sum is a straight chain of D adds.
template <int DP, int NH>
__device__ __noinline__ bool bs_radius_test(double nv0, uint32_t rec_addr, int lane, int D, double delta2, double eps2,
                                            int div_mode, double k, double wsel) {
    constexpr int NT = DP > 32 ? 2 : 1; // terms per lane
    double wn, c1[NT], c2[NT];
    if (NH == 1) { // fetch CF2', W' by shuffle
        wn = __shfl_sync(0xffffffffu, nv0, 2 * DP);
        c1[0] = nv0;
        c2[0] = __shfl_sync(0xffffffffu, nv0, (lane + DP) & 31);
    } else {
        __syncwarp();
        wn = lds_f64(rec_addr - lane * 8 + 2 * DP * 8);
#pragma unroll
        for (int h = 0; h < NT; ++h) {
            const bool rd = lane + 32 * h < D;
            c1[h] = rd ? lds_f64(rec_addr + 32 * h * 8) : 1.0;
            c2[h] = rd ? lds_f64(rec_addr + (DP + 32 * h) * 8) : 1.0;
        }
    }
    double term[NT];
#pragma unroll
    for (int h = 0; h < NT; ++h) {
        const bool act = lane + 32 * h < D;
        // idle lanes carry 1.0: their (discarded) quotients stay on the fast path of the division
        const double q2 = ddiv(act ? c2[h] : 1.0, wn);
        const double c = ddiv(act ? c1[h] : 1.0, wn);
        const double var = dsub(q2, dmul(c, c));
        const bool bit = act && (var <= delta2);
        double t = var;
        if (div_mode) { // warp-uniform; a real branch, so that a power-of-two k never pays for this division
            asm volatile("");
            const double tq = ddiv(var, k);
            t = bit ? tq : var;
        } else {
            t = bit ? dmul(var, wsel) : var;
        }
        term[h] = t;
    }
    double r2 = 0.0;
    if (D == DP) {
#pragma unroll
        for (int d = 0; d < DP; ++d) r2 = dadd(r2, __shfl_sync(0xffffffffu, term[d >> 5], d & 31));
    } else {
#pragma unroll 1
        for (int d = 0; d < D; ++d) {
            const double t0 = __shfl_sync(0xffffffffu, term[0], d & 31);
            const double t1 = NT > 1 ? __shfl_sync(0xffffffffu, term[NT - 1], d & 31) : 0.0;
            r2 = dadd(r2, d < 32 ? t0 : t1);
        }
    }
    return r2 <= eps2;
}

// FAST radius test of a CONTESTED cell: the same decision from ~1/5 of the latency, or "undecided".  Returns 1 (radius^2 of
// the tentative MC <= eps^2: absorbed), 0 (rejected) or 2 (too close to call: the caller runs bs_radius_test).
// Multiplied through by W'^2 the test of mc_functions.py:45-56 reads  sum_d w_d (CF2'_d W' - CF1'_d^2)  <=  eps^2 W'^2
// with w_d = 1/k where CF2'_d W' - CF1'_d^2 <= delta^2 W'^2, else 1 -- no division.  Lane d evaluates its term in fp64 (one
// DMUL + one DFMA), scales it so that the right-hand side is at most TH = 2^25 (2^23 for DP > 16), rounds it to an integer and
// the warp adds the integers with ONE redux.sync instead of a chain of D shuffles and dependent adds.  DP > 16: the integer
// is split into a high and a low part (two redux.sync) to keep 2^-20 units.
// Bound.  In these units the fast sum and the reference's r^2 W'^2 fs each differ from the exact value by at most ~6 ulp per
// term of CF2'_d W' fs (the rounding of CF2' W' and of the fma; of CF2'/W', (CF1'/W')^2 and their difference), which sum
// to <= 12 * 2^-53 * TH * sum_d (CF2'_d / W') / eps^2, plus the rounding of the integer (1/2 a term unsplit, 2^-21 split)
// and ~D ulp of thr for the reference's own sum.  The decision is taken only when the sum is mg units clear of the
// threshold, mg = (D + 8 unsplit, 0.01 split) + 2^-48 * TH * sum_d (CF2_d / W) / eps^2 from the chain's start state (the
// tentative records of a chain stay near its centroid; the factor 32 over 2^-53 leaves 2.5x for that drift), and when no
// variance is within 2^-24 (relative) of delta^2; anything else -- including NaNs -- is "undecided".  So the decision is
// the reference's at any distance from the origin where the preference test itself is still resolvable (CF2 W / (delta^2
// W^2) < ~2^27, i.e. coordinates below ~1e4 delta); far from the origin the fast test only leaves more records undecided.
// A wrong decision could not corrupt results in any case: k_bs_verify_p recomputes every decision of the chain with the
// reference's exact arithmetic (a wrong one would merely cost a round), and the first member of every chain always takes
// the exact test, so every block advances.
struct ChainFast {
    double F;    // TH / Wmax^2, Wmax = W at the start of the chain + its members + 1 (>= every W' of the chain)
    double fs;   // F / eps^2: scale of the terms
    double invk; // weight of a preferred dimension (approximate for a k that is not a power of two)
    double delta2;
    double mg;   // clearance a decision needs, in integer units (see the bound above)
};
template <int DP, int NH>
__device__ __forceinline__ int bs_radius_fast(double nv0, uint32_t rec_addr, int lane, int D, const ChainFast cf) {
    constexpr int NT = DP > 32 ? 2 : 1; // terms per lane
    constexpr bool SPLIT = DP > 16;
    constexpr int CL = SPLIT ? (1 << 24) : (1 << 26);
    double wn, c1[NT], c2[NT];
    if (NH == 1) {
        wn = __shfl_sync(0xffffffffu, nv0, 2 * DP);
        c1[0] = nv0;
        c2[0] = __shfl_sync(0xffffffffu, nv0, (lane + DP) & 31);
    } else {
        __syncwarp();
        wn = lds_f64(rec_addr - lane * 8 + 2 * DP * 8);
#pragma unroll
        for (int h = 0; h < NT; ++h) {
            const bool rd = lane + 32 * h < D;
            c1[h] = rd ? lds_f64(rec_addr + 32 * h * 8) : 0.0;
            c2[h] = rd ? lds_f64(rec_addr + (DP + 32 * h) * 8) : 0.0;
        }
    }
    const double wn2 = dmul(wn, wn);
    const double thr = dmul(wn2, cf.F);
    const double d2w = dmul(cf.delta2, wn2);
    const double tol = dmul(d2w, 0x1p-24);
    // integer thresholds, off the critical path (they depend on W' only): absorbed below t_lo, rejected above t_hi
    const int t_lo = __double2int_rd(dsub(thr, cf.mg)), t_hi = __double2int_ru(dadd(thr, cf.mg));
    int hi_sum = 0, lo_sum = 0;
    bool amb = false;
#pragma unroll
    for (int h = 0; h < NT; ++h) {
        const bool act = lane + 32 * h < D;
        const double t = __fma_rn(-c1[h], c1[h], dmul(c2[h], wn));
        const double diff = dsub(t, d2w);
        amb = amb || (act && !(fabs(diff) > tol));
        const double tk = dmul(t, cf.invk);
        const double v = dmul(diff <= 0.0 ? tk : t, cf.fs);
        int hi = __double2int_rn(v); // saturates; NaN -> 0 (caught by amb above)
        hi = max(min(hi, CL), -(1 << 20));
        hi_sum += act ? hi : 0;
        if (SPLIT) {
            const int lo = __double2int_rn(dmul(dsub(v, (double)hi), 0x1p20));
            lo_sum += act ? max(min(lo, 1 << 20), -(1 << 20)) : 0;
        }
    }
    const int S = __reduce_add_sync(0xffffffffu, hi_sum);
    if (__any_sync(0xffffffffu, amb)) return 2;
    if (SPLIT) {
        const int L = __reduce_add_sync(0xffffffffu, lo_sum);
        const double tot = dadd((double)S, dmul((double)L, 0x1p-20));
        if (tot < dsub(thr, cf.mg)) return 1;
        if (tot > dadd(thr, cf.mg)) return 0;
        return 2;
    }
    return S < t_lo ? 1 : (S > t_hi ? 0 : 2);
}

__device__ __forceinline__ void fence_proxy_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// one group of GS = 8 cells that holds a CONTESTED cell or is the ragged tail of the key: its addends are fetched up
// front, then the cells go one by one, the CONTESTED ones through the exact radius test on their tentative record.  Kept
// out of line (one copy; see bs_radius_test).
template <int NH>
struct ChainRec {
    double v[NH];
};
template <int DP, int NH>
__device__ __noinline__ ChainRec<NH> bs_chain_slow_group(ChainRec<NH> rec, uint32_t ga, uint32_t ma_g, unsigned cg, int ncell,
                                                         int lane, int D, double delta2, double eps2, int div_mode, double k,
                                                         double wsel, uint8_t *prej, const ChainFast cf, int exact_first) {
    constexpr int LSP = 2 * DP + 2, GS = 8;
    double(&v)[NH] = rec.v;
    bool st_ok[NH];
#pragma unroll
    for (int h = 0; h < NH; ++h) st_ok[h] = lane + 32 * h < LSP;
    double R[GS][NH];
    unsigned rej = 0u;
#pragma unroll
    for (int q = 0; q < GS; ++q)
#pragma unroll
        for (int h = 0; h < NH; ++h) R[q][h] = lds_f64(ga + (q * LSP + 32 * h) * 8); // (stale past ncell: never used)
#pragma unroll
    for (int q = 0; q < GS; ++q) {
        if (q < ncell) { // warp-uniform
            const uint32_t ra = ga + q * (LSP * 8);
            double nv[NH];
#pragma unroll
            for (int h = 0; h < NH; ++h) {
                nv[h] = dadd(v[h], R[q][h]);
                if (st_ok[h]) sts_f64(ra + 32 * h * 8, nv[h]);
            }
            bool keep = true;
            if ((cg >> q) & 1u) {
                int r = (q == 0 && exact_first) ? 2 : bs_radius_fast<DP, NH>(nv[0], ra, lane, D, cf);
                if (r == 2) r = bs_radius_test<DP, NH>(nv[0], ra, lane, D, delta2, eps2, div_mode, k, wsel) ? 1 : 0;
                keep = r != 0;
                rej |= (keep ? 0u : 1u) << q;
            }
            if (keep) { // the record of a rejected cell is never read as a version
#pragma unroll
                for (int h = 0; h < NH; ++h) v[h] = nv[h];
            }
        }
    }
    // the verdicts of the group's CONTESTED cells, lane q = cell q: one divergent region per group, not one per cell
    if (lane < GS && ((cg >> lane) & 1u) && lane < ncell) {
        int raw;
        asm volatile("ld.shared.s32 %0, [%1];" : "=r"(raw) : "r"(ma_g + lane * 4));
        prej[raw & BS_PL_CELL] = (uint8_t)((rej >> lane) & 1u);
    }
    return rec;
}

// The same group when the record is one register per lane (NH == 1: DP <= 12) and CONTESTED cells come in runs -- the cold
// start and the saturated parameter corners, where whole chains are CONTESTED: TWO cells per step.  The verdict of cell q + 1
// depends on that of cell q only through which state it is added to, so its test is evaluated for BOTH outcomes of cell q
// next to cell q's own test (three independent instruction streams for the in-order warp instead of one dependent one)
// and the right one is picked afterwards: ~1/2 of the latency per CONTESTED cell.  Anything the fast test cannot call
// (and the first member of a chain) takes the one-by-one path with the exact test.  A rolled loop: the code stays small.
struct ChainRecD {
    double v;
    int dev; // CONTESTED cells of the group whose verdict differed from the prediction
};
template <int DP>
__device__ __noinline__ ChainRecD bs_chain_slow_group_pairs(ChainRecD rec, uint32_t ga, uint32_t ma_g, unsigned cg, unsigned pg,
                                                            int ncell, int lane, int D, double delta2, double eps2, int div_mode,
                                                            double k, double wsel, uint8_t *prej, uint8_t *pflag,
                                                            const ChainFast cf, int exact_first) {
    constexpr int LSP = 2 * DP + 2, GS = 8;
    double v = rec.v;
    const bool st_ok = lane < LSP;
    unsigned rej = 0u;
    double a0 = lds_f64(ga), a1 = lds_f64(ga + LSP * 8); // (a1 is stale when ncell == 1: never used)
#pragma unroll 1
    for (int q = 0; q < ncell; q += 2) { // two cells per trip
        const uint32_t ra = ga + q * (LSP * 8);
        // the addends of the next trip (clamped: never used past the group)
        const double a2 = lds_f64(ga + min(q + 2, GS - 1) * (LSP * 8)), a3 = lds_f64(ga + min(q + 3, GS - 1) * (LSP * 8));
        const bool hasB = q + 1 < ncell;
        const bool cA = (cg >> q) & 1u, cB = hasB && ((cg >> (q + 1)) & 1u);
        const double nvA = dadd(v, a0);
        if (st_ok) sts_f64(ra, nvA);
        int rA = 1, rB = 1;
        double nvB;
        bool done = false;
        if (cA && cB && !(q == 0 && exact_first)) {
            const double nvB1 = dadd(nvA, a1), nvB0 = dadd(v, a1);
            rA = bs_radius_fast<DP, 1>(nvA, ra, lane, D, cf);
            const int rB1 = bs_radius_fast<DP, 1>(nvB1, ra, lane, D, cf);
            const int rB0 = bs_radius_fast<DP, 1>(nvB0, ra, lane, D, cf);
            rB = rA ? rB1 : rB0;
            nvB = rA ? nvB1 : nvB0;
            done = rA != 2 && rB != 2;
        }
        if (!done) { // one by one
            if (cA) {
                rA = (q == 0 && exact_first) ? 2 : bs_radius_fast<DP, 1>(nvA, ra, lane, D, cf);
                if (rA == 2) rA = bs_radius_test<DP, 1>(nvA, ra, lane, D, delta2, eps2, div_mode, k, wsel) ? 1 : 0;
            }
            nvB = dadd(rA ? nvA : v, a1);
            if (cB) {
                rB = bs_radius_fast<DP, 1>(nvB, ra, lane, D, cf);
                if (rB == 2) rB = bs_radius_test<DP, 1>(nvB, ra + LSP * 8, lane, D, delta2, eps2, div_mode, k, wsel) ? 1 : 0;
            }
        }
        if (hasB) {
            if (st_ok) sts_f64(ra + LSP * 8, nvB);
            v = rB ? nvB : (rA ? nvA : v);
            rej |= ((cA && !rA) ? 1u : 0u) << q | ((cB && !rB) ? 1u : 0u) << (q + 1);
        } else {
            v = rA ? nvA : v;
            rej |= ((cA && !rA) ? 1u : 0u) << q;
        }
        a0 = a2;
        a1 = a3;
    }
    if (lane < GS && ((cg >> lane) & 1u) && lane < ncell) { // verdicts + next round's predictions
        int raw;
        asm volatile("ld.shared.s32 %0, [%1];" : "=r"(raw) : "r"(ma_g + lane * 4));
        const unsigned r = (rej >> lane) & 1u;
        prej[raw & BS_PL_CELL] = (uint8_t)r;
        pflag[raw & BS_PL_CELL] = (uint8_t)(1u | (r << 1));
    }
    rec.v = v;
    rec.dev = __popc((rej ^ pg) & cg & ((1u << ncell) - 1u));
    return rec;
}

// The same group, EIGHT cells per pass (NH == 1).  Every CONTESTED cell carries a predicted verdict (BS_PL_PREJ: the
// snapshot's in round 1, its own verdict of the round before afterwards).  A pass lays the tentative records of the cells
// q0 .. 7 along the predicted pattern (a predicted-rejected cell leaves the state alone, so runs of them are not even
// chained), runs the fast tests of all of them side by side -- independent instruction streams, their integer sums through
// back-to-back redux.sync, ONE redux for all "too close to call" flags -- and compares with the prediction: the cells in
// front of the first deviation are final, the deviating cell itself is final too (its record was built on the right
// state; an undecided one takes the exact test), and the next pass starts behind it.  With mostly right predictions that
// is one pass of ~400 cycles per eight cells instead of eight dependent tests.  Nothing here can change a result: every
// verdict is the fast test's (decision-exact by its clearance, re-checked by k_bs_verify_p) or the exact test's.
template <int DP>
__device__ __noinline__ ChainRecD bs_chain_slow_group_batch(ChainRecD rec, uint32_t ga, uint32_t ma_g, unsigned cg, unsigned pg,
                                                            int ncell, int lane, int D, double delta2, double eps2, int div_mode,
                                                            double k, double wsel, uint8_t *prej, uint8_t *pflag,
                                                            const ChainFast cf, int exact_first) {
    constexpr int LSP = 2 * DP + 2, GS = 8;
    constexpr int CL = 1 << 26;
    double v = rec.v;
    int ndev = 0;
    const bool st_ok = lane < LSP, act = lane < D;
    const unsigned live = (1u << ncell) - 1u;
    cg &= live;
    const unsigned pred = pg & cg; // predicted rejections
    unsigned rej = 0u;             // verdicts
    double a[GS];
#pragma unroll
    for (int q = 0; q < GS; ++q) a[q] = lds_f64(ga + q * (LSP * 8)); // (stale past ncell: never used)
    int q0 = 0;
    if (exact_first && (cg & 1u)) { // the first member of a chain takes the exact test: every block advances
        const double nv = dadd(v, a[0]);
        if (st_ok) sts_f64(ga, nv);
        if (bs_radius_test<DP, 1>(nv, ga, lane, D, delta2, eps2, div_mode, k, wsel)) v = nv;
        else rej |= 1u;
        q0 = 1;
    }
#pragma unroll 1
    while (q0 < ncell) {
        const unsigned todo = live & ~((1u << q0) - 1u); // cells of this pass
        const unsigned adv = todo & ~pred;               // ... that are predicted to join the chain
        double nv[GS], sb[GS];                           // tentative record of cell q, state in front of it
        {
            // the state runs through a pure chain of adds: a cell that does not join adds -0.0, the exact identity of
            // IEEE addition in round-to-nearest (x + -0.0 == x for every x, signed zeros included)
            double ae[GS];
#pragma unroll
            for (int q = 0; q < GS; ++q) ae[q] = ((adv >> q) & 1u) ? a[q] : -0.0;
            double st = v;
#pragma unroll
            for (int q = 0; q < GS; ++q) {
                sb[q] = st;
                nv[q] = dadd(st, a[q]);
                st = dadd(st, ae[q]);
            }
        }
        // fast tests of all eight records (bs_radius_fast, NT == 1, unsplit), reductions apart
        int hs[GS], tlo[GS], thi[GS];
        unsigned ambm = 0u;
#pragma unroll
        for (int q = 0; q < GS; ++q) {
            const double wn = __shfl_sync(0xffffffffu, nv[q], 2 * DP);
            const double c2 = __shfl_sync(0xffffffffu, nv[q], (lane + DP) & 31);
            const double c1 = nv[q];
            const double wn2 = dmul(wn, wn);
            const double thr = dmul(wn2, cf.F);
            const double d2w = dmul(cf.delta2, wn2);
            const double tol = dmul(d2w, 0x1p-24);
            tlo[q] = __double2int_rd(dsub(thr, cf.mg));
            thi[q] = __double2int_ru(dadd(thr, cf.mg));
            const double t = __fma_rn(-c1, c1, dmul(c2, wn));
            const double diff = dsub(t, d2w);
            if (act && !(fabs(diff) > tol)) ambm |= 1u << q;
            const double tk = dmul(t, cf.invk);
            const double vv = dmul(diff <= 0.0 ? tk : t, cf.fs);
            int hi = __double2int_rn(vv); // saturates; NaN -> 0 (caught by ambm)
            hi = max(min(hi, CL), -(1 << 20));
            hs[q] = act ? hi : 0;
        }
#pragma unroll
        for (int q = 0; q < GS; ++q) hs[q] = __reduce_add_sync(0xffffffffu, hs[q]);
        ambm = __reduce_or_sync(0xffffffffu, ambm);
        unsigned accm = 0u, rejm = 0u;
#pragma unroll
        for (int q = 0; q < GS; ++q) {
            accm |= (hs[q] < tlo[q] ? 1u : 0u) << q;
            rejm |= (hs[q] > thi[q] ? 1u : 0u) << q;
        }
        accm &= ~ambm;
        rejm &= ~ambm;
        const unsigned und = ~(accm | rejm);
        const unsigned dev = ((rejm & ~pred) | (accm & pred) | und) & cg & todo; // verdict != prediction, or none
        const int qs = dev ? __ffs(dev) - 1 : ncell;                              // first deviating cell
        const int qe = min(qs, ncell - 1);
#pragma unroll
        for (int q = 0; q < GS; ++q)
            if (q >= q0 && q <= qe && st_ok) sts_f64(ga + q * (LSP * 8), nv[q]);
        rej |= pred & todo & ((1u << qs) - 1u);
        // state behind cell qe when the cells in front of it went as predicted and qe itself as `keep` says
        double nq = nv[0], sq = sb[0];
#pragma unroll
        for (int q = 1; q < GS; ++q) {
            nq = q == qe ? nv[q] : nq;
            sq = q == qe ? sb[q] : sq;
        }
        bool keep;
        if (dev) {
            ++ndev;
            if ((und >> qs) & 1u) keep = bs_radius_test<DP, 1>(nq, ga + qs * (LSP * 8), lane, D, delta2, eps2, div_mode, k, wsel);
            else keep = (accm >> qs) & 1u;
            rej |= (keep ? 0u : 1u) << qs;
        } else {
            keep = !((pred >> qe) & 1u);
        }
        v = keep ? nq : sq;
        q0 = qs + 1;
    }
    if (lane < GS && ((cg >> lane) & 1u)) { // verdicts of the CONTESTED cells (lane q = cell q) + next round's prediction
        int raw;
        asm volatile("ld.shared.s32 %0, [%1];" : "=r"(raw) : "r"(ma_g + lane * 4));
        const unsigned r = (rej >> lane) & 1u;
        prej[raw & BS_PL_CELL] = (uint8_t)r;
        pflag[raw & BS_PL_CELL] = (uint8_t)(1u | (r << 1));
    }
    rec.v = v;
    rec.dev = ndev;
    return rec;
}

// 32 consecutive cells without a CONTESTED one inside a stage that holds one elsewhere: the straight-line schedule of the
// clean stage (dependent add, store of the version before, load one batch ahead), out of line -- one copy, used rarely.
template <int DP, int NH>
__device__ __noinline__ ChainRec<NH> bs_chain_clean32(ChainRec<NH> rec, uint32_t xa, int lane) {
    constexpr int LSP = 2 * DP + 2, GS = 8, NG = 4;
    double(&v)[NH] = rec.v;
    bool st_ok[NH];
#pragma unroll
    for (int h = 0; h < NH; ++h) st_ok[h] = lane + 32 * h < LSP;
    double R[2][GS][NH];
#pragma unroll
    for (int q = 0; q < GS; ++q)
#pragma unroll
        for (int h = 0; h < NH; ++h) R[0][q][h] = lds_f64(xa + (q * LSP + 32 * h) * 8);
#pragma unroll
    for (int k = 0; k < NG; ++k) {
#pragma unroll
        for (int q = 0; q < GS; ++q) {
            double nv[NH];
#pragma unroll
            for (int h = 0; h < NH; ++h) nv[h] = dadd(v[h], R[k & 1][q][h]);
            if (k + q > 0) {
#pragma unroll
                for (int h = 0; h < NH; ++h)
                    if (st_ok[h]) sts_f64(xa + ((k * GS + q - 1) * LSP + 32 * h) * 8, v[h]);
            }
            if (k + 1 < NG) {
#pragma unroll
                for (int h = 0; h < NH; ++h) R[(k + 1) & 1][q][h] = lds_f64(xa + (((k + 1) * GS + q) * LSP + 32 * h) * 8);
            }
#pragma unroll
            for (int h = 0; h < NH; ++h) v[h] = nv[h];
        }
    }
#pragma unroll
    for (int h = 0; h < NH; ++h)
        if (st_ok[h]) sts_f64(xa + ((NG * GS - 1) * LSP + 32 * h) * 8, v[h]);
    return rec;
}

template <int DP>
__global__ void __launch_bounds__(BS_CHAINP_THREADS) k_bs_chain_p(Eng e) {
    e.fetch();
    CCB_TS(9);
    CCB_PDL();
    using Cfg = ChainPCfg<DP>;
    constexpr int NB = Cfg::NB, S = Cfg::S, GS = 8, NH = Cfg::NH, LSP = Cfg::LSP, NG = NB / GS;
    static_assert(NB == 32 || NB == 64, "the CONTESTED flags of a stage are gathered by one or two ballots");
    extern __shared__ __align__(128) unsigned char bs_smem[];
    double *xs = reinterpret_cast<double *>(bs_smem);              // [S][NB][LSP]
    int *ms = reinterpret_cast<int *>(xs + (size_t)S * NB * LSP);  // [S][NB]
    uint64_t *full = reinterpret_cast<uint64_t *>(ms + S * NB);    // [S] producer -> replay
    uint64_t *done = full + S;                                     // [S] replay -> store thread
    uint64_t *empty = done + S;                                    // [S] store thread -> producer
    const BsCtl *bc = e.bc;
    if (!bc->active || bc->phase != 0 || bc->pclean) return;
    const Num nm = e.nm;
    const int D = nm.D;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int j = blockIdx.x;
    if (j >= bc->Mp) return;
    const int n = e.ws.pcnt[j];
    if (n <= 0) return;
    const int p0 = e.ws.poff[j];
    const double *xg = e.ws.xg + (size_t)p0 * LSP;
    const int32_t *pl = e.ws.plist + p0;
    const int nb = (n + NB - 1) / NB;
    if (tid == 0) {
        for (int s = 0; s < S; ++s) {
            mbar_init(&full[s], 1);
            mbar_init(&done[s], 1);
            mbar_init(&empty[s], 1);
        }
        mbar_fence_init();
    }
    __syncthreads();
    if (warp == 1) { // ---- producer
        if (lane == 0) {
            CCB_DBG(long long tw = 0;)
            for (int b = 0; b < nb; ++b) {
                const int s = b % S;
                if (b >= S) {
                    CCB_DBG(const long long t0 = clock64();)
                    mbar_wait(&empty[s], ((b / S) - 1) & 1);
                    CCB_DBG(tw += clock64() - t0;)
                }
                const int cnt = min(NB, n - b * NB);
                const uint32_t bx = (uint32_t)cnt * LSP * 8u, bi = (uint32_t)((cnt + 3) & ~3) * 4u;
                mbar_expect_tx(&full[s], bx + bi);
                tma_load_1d(xs + (size_t)s * NB * LSP, xg + (size_t)b * NB * LSP, bx, &full[s]);
                tma_load_1d(ms + s * NB, pl + b * NB, bi, &full[s]);
            }
            CCB_DBG((void)tw;)
        }
        return;
    }
    if (warp == 2) { // ---- store thread: verp[plist position] <- the versions left in the stage, one bulk copy per stage
        if (lane == 0) {
            CCB_DBG(long long tw = 0; const long long tbeg = clock64();)
            double *vp = e.ws.verp + (size_t)p0 * LSP;
            for (int b = 0; b < nb; ++b) {
                const int s = b % S;
                {
                    CCB_DBG(const long long t0 = clock64();)
                    mbar_wait(&done[s], (b / S) & 1);
                    CCB_DBG(tw += clock64() - t0;)
                }
                const int cnt = min(NB, n - b * NB);
                tma_store_1d(vp + (size_t)b * NB * LSP, xs + (size_t)s * NB * LSP, (uint32_t)cnt * LSP * 8u);
                asm volatile("cp.async.bulk.commit_group;" ::: "memory");
                if (b > 0) { // the copy before this one has read its stage: hand that stage back to the producer
                    asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory");
                    mbar_arrive(&empty[(b - 1) % S]);
                }
            }
            asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); // shared memory must outlive the copies
            CCB_DBG((void)tw; (void)tbeg;)
        }
        return;
    }
    if (warp != 0) {
        if (warp == 4) { // (the replay warp's scheduler: it is still waiting for its first stage)
            // one pass through the rare-path code on dummy data: its instruction-cache lines are then on this SM before the
            // replay warp (which cannot hide a miss) meets its first CONTESTED cell
            const bool r = bs_radius_test<DP, NH>(1.0, smem_u32(xs) + lane * 8, lane, D, nm.delta2, nm.eps2, nm.div_mode, nm.k,
                                                  nm.wsel);
            if (r && D < 0) e.ws.prej[0] = 1; // never taken; keeps the call alive
        }
        return;
    }
    // ---- replay (warp 0): lane owns elements lane + 32 h of the record
    double v[NH];
#pragma unroll
    for (int h = 0; h < NH; ++h) {
        const int el = lane + 32 * h;
        double x = 0.0;
        if (el < D) x = e.P.cf1[(size_t)j * D + el];
        else if (el >= DP && el < DP + D) x = e.P.cf2[(size_t)j * D + el - DP];
        else if (el == 2 * DP) x = e.P.w[j];
        v[h] = x;
    }
    ChainFast cfast;
    {
        constexpr double TH = DP > 16 ? 0x1p23 : 0x1p25;
        const double wmax = dadd(e.P.w[j], (double)(n + 1));
        cfast.F = ddiv(TH, dmul(wmax, wmax));
        cfast.fs = ddiv(cfast.F, nm.eps2);
        cfast.invk = nm.div_mode ? ddiv(1.0, nm.k) : nm.wsel;
        cfast.delta2 = nm.delta2;
        // sum_d CF2_d / W of the chain's start state (any order: it only feeds the error bound of the clearance)
        double q2 = 0.0;
#pragma unroll
        for (int h = 0; h < NH; ++h) {
            const int el = lane + 32 * h;
            q2 = dadd(q2, el >= DP && el < DP + D ? v[h] : 0.0);
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) q2 = dadd(q2, __shfl_xor_sync(0xffffffffu, q2, o));
        cfast.mg = dadd(DP > 16 ? 0.01 : (double)(D + 8), dmul(0x1p-48 * TH, ddiv(ddiv(q2, e.P.w[j]), nm.eps2)));
    }
    bool bmode = bc->it > 0; // (see the CONTESTED groups below)
    CCB_DBG(long long t_wait = 0, t_slow = 0, n_cont = 0, t_head = 0, t_tail = 0, n_clean = 0; const long long t_beg = clock64();)
    // The replay warp issues in order and is alone on its scheduler: every dependent instruction costs its full latency.
    // Everything below is arranged for that.  Addresses and the lane number are held in OPAQUE registers (otherwise the
    // compiler re-derives them from special registers -- S2R / S2UR, tens of cycles each -- inside the loop).
    uint32_t xs_lane = smem_u32(xs) + lane * 8, ms_base = smem_u32(ms);
    int lane_o = lane;
    asm volatile("" : "+r"(xs_lane), "+r"(ms_base), "+r"(lane_o));
    bool st_ok[NH];
#pragma unroll
    for (int h = 0; h < NH; ++h) st_ok[h] = lane_o + 32 * h < LSP;

    for (int b = 0; b < nb; ++b) {
        const int s = b % S;
        {
            CCB_DBG(const long long t0 = clock64();)
            mbar_wait(&full[s], (b / S) & 1);
            CCB_DBG(t_wait += clock64() - t0;)
        }
        CCB_DBG(const long long t_h0 = clock64();)
        const int cnt = __shfl_sync(0xffffffffu, min(NB, n - b * NB), 0); // warp-uniform for the compiler, too
        uint32_t xa = xs_lane + s * (NB * LSP * 8), ma = ms_base + s * (NB * 4);
        asm volatile("" : "+r"(xa), "+r"(ma));
        // CONTESTED flags of the whole stage: lane l looks at cells l and l + 32
        unsigned c_lo, c_hi = 0u, p_lo = 0u, p_hi = 0u;
        {
            int f0, f1 = 0;
            asm volatile("ld.shared.s32 %0, [%1];" : "=r"(f0) : "r"(ma + lane_o * 4));
            if (NB > 32) asm volatile("ld.shared.s32 %0, [%1];" : "=r"(f1) : "r"(ma + (lane_o + 32) * 4));
            c_lo = __ballot_sync(0xffffffffu, f0 < 0 && lane_o < cnt);
            if (NB > 32) c_hi = __ballot_sync(0xffffffffu, f1 < 0 && lane_o + 32 < cnt);
            if (NH == 1 && (c_lo | c_hi)) { // predicted verdicts of the CONTESTED cells (bs_chain_slow_group_batch)
                p_lo = __ballot_sync(0xffffffffu, (f0 & BS_PL_PREJ) != 0);
                if (NB > 32) p_hi = __ballot_sync(0xffffffffu, (f1 & BS_PL_PREJ) != 0);
            }
        }
        CCB_DBG(t_head += clock64() - t_h0;)
        if (cnt == NB && (c_lo | c_hi) == 0u) {
            CCB_DBG(++n_clean;)
            // ---- CLEAN FULL STAGE: straight-line code with immediate offsets.  Cell c: the dependent add, then -- in its
            // latency shadow -- the store of the version cell c - 1 left and the load of an addend one batch ahead.
            double R[2][GS][NH];
#pragma unroll
            for (int q = 0; q < GS; ++q)
#pragma unroll
                for (int h = 0; h < NH; ++h) R[0][q][h] = lds_f64(xa + (q * LSP + 32 * h) * 8);
#pragma unroll
            for (int k = 0; k < NG; ++k) {
#pragma unroll
                for (int q = 0; q < GS; ++q) {
                    double nv[NH];
#pragma unroll
                    for (int h = 0; h < NH; ++h) nv[h] = dadd(v[h], R[k & 1][q][h]);
                    if (k + q > 0) {
#pragma unroll
                        for (int h = 0; h < NH; ++h)
                            if (st_ok[h]) sts_f64(xa + ((k * GS + q - 1) * LSP + 32 * h) * 8, v[h]);
                    }
                    if (k + 1 < NG) {
#pragma unroll
                        for (int h = 0; h < NH; ++h) R[(k + 1) & 1][q][h] = lds_f64(xa + (((k + 1) * GS + q) * LSP + 32 * h) * 8);
                    }
#pragma unroll
                    for (int h = 0; h < NH; ++h) v[h] = nv[h];
                }
            }
#pragma unroll
            for (int h = 0; h < NH; ++h)
                if (st_ok[h]) sts_f64(xa + ((NB - 1) * LSP + 32 * h) * 8, v[h]);
        } else {
            // ---- stage with CONTESTED cells or the ragged tail: group by group; a clean full group is eight chained adds
            // through registers, any other group goes cell by cell (out of line), CONTESTED cells through the exact radius
            // test on their tentative record
            CCB_DBG(const long long t_s0 = clock64(); n_cont += __popc(c_lo) + __popc(c_hi);)
            const int ng = (cnt + GS - 1) / GS;
#pragma unroll 1
            for (int g = 0; g < ng; ++g) {
                if (NB == 64 && (g & 3) == 0 && cnt - g * GS >= 32 && (g ? c_hi : c_lo) == 0u) {
                    // this half of the stage is clean: 32 cells of straight-line code
                    ChainRec<NH> rec;
#pragma unroll
                    for (int h = 0; h < NH; ++h) rec.v[h] = v[h];
                    rec = bs_chain_clean32<DP, NH>(rec, xa + g * (GS * LSP * 8), lane_o);
#pragma unroll
                    for (int h = 0; h < NH; ++h) v[h] = rec.v[h];
                    g += 3;
                    continue;
                }
                uint32_t ga = xa + g * (GS * LSP * 8);
                asm volatile("" : "+r"(ga));
                const unsigned cg = ((g < 4 ? c_lo : c_hi) >> (8 * (g & 3))) & 0xffu;
                const int ncell = min(GS, cnt - g * GS);
                if (cg == 0u && ncell == GS) {
                    double R[GS][NH];
#pragma unroll
                    for (int q = 0; q < GS; ++q)
#pragma unroll
                        for (int h = 0; h < NH; ++h) R[q][h] = lds_f64(ga + (q * LSP + 32 * h) * 8);
#pragma unroll
                    for (int q = 0; q < GS; ++q)
#pragma unroll
                        for (int h = 0; h < NH; ++h) {
                            v[h] = dadd(v[h], R[q][h]);
                            if (st_ok[h]) sts_f64(ga + (q * LSP + 32 * h) * 8, v[h]);
                        }
                } else {
                    ChainRec<NH> rec;
#pragma unroll
                    for (int h = 0; h < NH; ++h) rec.v[h] = v[h];
                    if constexpr (NH == 1) {
                        if (__popc(cg) >= 2) {
                            // runs of CONTESTED cells: eight per pass along the predicted verdicts while the predictions hold
                            // (refinement rounds: a cell's verdict of the round before), two per step otherwise (round 1 on
                            // a young MC: the snapshot's predictions are worth little) -- the last group's count decides
                            const unsigned pgm = ((g < 4 ? p_lo : p_hi) >> (8 * (g & 3))) & 0xffu;
                            ChainRecD rd;
                            rd.v = v[0];
                            rd.dev = 0;
                            if (bmode)
                                rd = bs_chain_slow_group_batch<DP>(rd, ga, ma + g * (GS * 4), cg, pgm, ncell, lane_o, D, nm.delta2,
                                                                   nm.eps2, nm.div_mode, nm.k, nm.wsel, e.ws.prej, e.ws.pflag, cfast,
                                                                   (b | g) == 0);
                            else
                                rd = bs_chain_slow_group_pairs<DP>(rd, ga, ma + g * (GS * 4), cg, pgm, ncell, lane_o, D, nm.delta2,
                                                                   nm.eps2, nm.div_mode, nm.k, nm.wsel, e.ws.prej, e.ws.pflag, cfast,
                                                                   (b | g) == 0);
                            rec.v[0] = rd.v;
                            CCB_DBG(if (lane_o == 0) {
                                atomicAdd(&g_dbg_cnt[bmode ? 0 : 2], 1ull);             // groups taken eight / two at a time
                                atomicAdd(&g_dbg_cnt[bmode ? 1 : 3], (unsigned long long)rd.dev); // ... and their deviations
                                atomicAdd(&g_dbg_cnt[4], (unsigned long long)__popc(cg));
                                atomicAdd(&g_dbg_cnt[5], (unsigned long long)__popc(pgm & cg)); // predicted rejections
                            })
                            bmode = rd.dev <= 1;
                        } else
                            rec = bs_chain_slow_group<DP, NH>(rec, ga, ma + g * (GS * 4), cg, ncell, lane_o, D, nm.delta2, nm.eps2,
                                                              nm.div_mode, nm.k, nm.wsel, e.ws.prej, cfast, (b | g) == 0);
                    } else {
                        rec = bs_chain_slow_group<DP, NH>(rec, ga, ma + g * (GS * 4), cg, ncell, lane_o, D, nm.delta2, nm.eps2,
                                                          nm.div_mode, nm.k, nm.wsel, e.ws.prej, cfast, (b | g) == 0);
                    }
#pragma unroll
                    for (int h = 0; h < NH; ++h) v[h] = rec.v[h];
                }
            }
            CCB_DBG(t_slow += clock64() - t_s0;)
        }
        // the versions were written through the generic proxy; the bulk copy reads them through the async proxy
        CCB_DBG(const long long t_t0 = clock64();)
        __syncwarp();
        fence_proxy_async_smem();
        __syncwarp();
        if (lane_o == 0) mbar_arrive(&done[s]);
        CCB_DBG(t_tail += clock64() - t_t0;)
    }
    CCB_DBG(if (lane == 0) atomicMax((unsigned long long *)&g_trace_ts[20], (unsigned long long)globaltimer_ns());)
    CCB_DBG(if (e.ws.dbg && lane == 0) {
        e.ws.dbg[j * 8 + 0] = n;
        e.ws.dbg[j * 8 + 1] = clock64() - t_beg;
        e.ws.dbg[j * 8 + 2] = t_wait;
        e.ws.dbg[j * 8 + 3] = t_slow;
        e.ws.dbg[j * 8 + 4] = n_cont;
        e.ws.dbg[j * 8 + 5] = t_head;  // (the store thread's slots: it only waits)
        e.ws.dbg[j * 8 + 6] = t_tail;
        e.ws.dbg[j * 8 + 7] = n_clean;
    })
}

// ---- outlier-side member lists: sort (key, cell) of the pcore-rejected cells --------------------------
// RANK SORT over the whole GPU.  The composite (key, cell) values are distinct, so the sorted position of an entry is the
// number of smaller entries.  Every CTA compacts the same entry list into its shared memory (a few thousand slots of the
// need list at most), then ranks its own slice of the entries -- BS_OL_TPE threads per entry, each counting over a strided
// part of the array (broadcast reads) -- and writes the entries to their places in global memory; the last CTA to finish
// (ticket) turns the sorted array into the key segments.  A single CTA spent 55 us in a bitonic sort of 4096 entries;
// 148 CTAs need ~2 us for the 16.7 M comparisons.
constexpr int BS_OL_THREADS = 512, BS_OL_TPE = 16, BS_OL_CTAS = 148;

__global__ void __launch_bounds__(BS_OL_THREADS, 1) k_bs_olist(Eng e) {
    e.fetch();
    CCB_TS(12);
    CCB_PDL();
    constexpr int NT = BS_OL_THREADS, TPE = BS_OL_TPE, EPP = NT / TPE; // entries ranked per pass
    __shared__ unsigned long long keys[BS_RMAX];
    __shared__ int s_warp[33];
    __shared__ int s_last;
    BsCtl *bc = e.bc;
    if (!bc->active || bc->phase != 0) return;
    const int tid = threadIdx.x;
    const int Mp = bc->Mp, KNEW = bc->Mp + bc->Mo0;
    const int nneed = bc->nneed, Beff = bc->Beff;
    // only as many CTAs as the list can keep busy take part (a few hundred entries: a dozen CTAs); the rest leave at once
    const int ncta = max(1, min((int)gridDim.x, (nneed + EPP - 1) / EPP));
    if ((int)blockIdx.x >= ncta) return;
    // ---- every CTA: the entry list, in need-list order (the same in every CTA)
    constexpr int SPT = BS_RMAX / NT; // slots per thread
    unsigned long long mine[SPT];
    int cnt = 0;
#pragma unroll
    for (int u = 0; u < SPT; ++u) {
        const int t = tid * SPT + u;
        mine[u] = ~0ull;
        if (t < nneed) {
            const int i = e.ws.ncell[t];
            if (i < Beff && e.ws.prej[i]) {
                const int sp = e.ws.ospec[i];
                if (sp >= 0) {
                    mine[u] = ((unsigned long long)(unsigned)sp << 32) | (unsigned)i;
                    ++cnt;
                }
            }
        }
    }
    int n;
    int pos = block_exclusive_scan_t<NT>(cnt, s_warp, n);
#pragma unroll
    for (int u = 0; u < SPT; ++u)
        if (mine[u] != ~0ull) keys[pos++] = mine[u];
    __syncthreads();
    // ---- rank of this CTA's slice
    const int sub = tid % TPE, slot = tid / TPE;
    for (int e0 = blockIdx.x * EPP; e0 < n; e0 += ncta * EPP) { // (block-uniform bounds)
        const int en = e0 + slot;
        const unsigned long long my = en < n ? keys[en] : 0ull;
        int rank = 0;
        if (en < n)
            for (int q = sub; q < n; q += TPE) rank += keys[q] < my;
#pragma unroll
        for (int o = TPE / 2; o > 0; o >>= 1) rank += __shfl_xor_sync(0xffffffffu, rank, o);
        if (en < n && sub == 0) e.ws.okeys[rank] = my;
    }
    // ---- the last CTA to get here builds the segments
    __threadfence();
    __syncthreads();
    if (tid == 0) s_last = atomicAdd(&bc->ticket_o, 1) == ncta - 1;
    __syncthreads();
    if (!s_last) return;
    __threadfence();
    for (int t = tid; t < n; t += NT) keys[t] = ((volatile unsigned long long *)e.ws.okeys)[t];
    // forget the modified-flags of the previous round
    for (int h = tid; h < bc->nh; h += NT) {
        const int key = e.ws.hkey[h];
        if (key < KNEW) e.ws.firstmember[key - Mp] = INT_MAX;
    }
    __syncthreads();
    // heads of the key segments, in key order (= list order: snapshot slots, then creations by creator), and the rank of
    // every created-in-block key among the REAL creations, in key (= creator) order.  A key is real when its first member
    // is its creator; a stale speculation can leave phantom keys (members, but the creator decided otherwise) -- those
    // lie beyond the first mismatch and get no rank.  Both counts ride in one scan (heads | real creations << 16).
    __shared__ int s_hnew0;
    if (tid == 0) s_hnew0 = INT_MAX;
    const int per = (n + NT - 1) / NT;
    const int lo = min(n, tid * per), hi = min(n, lo + per);
    cnt = 0;
    for (int t = lo; t < hi; ++t) {
        const int key = (int)(keys[t] >> 32), i = (int)(keys[t] & 0xffffffffu);
        if ((t == 0) || ((keys[t] >> 32) != (keys[t - 1] >> 32))) cnt += 1 + ((key >= KNEW && i == key - KNEW) ? (1 << 16) : 0);
    }
    int total;
    const int ex = block_exclusive_scan_t<NT>(cnt, s_warp, total);
    int h = ex & 0xffff, rk = ex >> 16;
    const int nh = total & 0xffff, nreal = total >> 16;
    for (int t = lo; t < hi; ++t) {
        const int key = (int)(keys[t] >> 32), i = (int)(keys[t] & 0xffffffffu);
        e.ws.omem[t] = i;
        if ((t == 0) || ((keys[t] >> 32) != (keys[t - 1] >> 32))) {
            e.ws.hkey[h] = key;
            e.ws.hoff[h] = t;
            e.ws.hfirst[h] = i;
            if (key < KNEW) {
                e.ws.firstmember[key - Mp] = i;
            } else {
                atomicMin(&s_hnew0, h);
                const bool real = i == key - KNEW;
                e.ws.hrank[h] = rk; // real creations before this key
                if (real) e.ws.newrank[i] = rk++;
            }
            ++h;
        }
    }
    __syncthreads();
    const int hnew0 = min(s_hnew0, nh);
    if (tid == 0) {
        bc->nh = nh;
        bc->no = n;
        bc->hnew0 = hnew0;
        bc->ticket_o = 0;
        bc->o_big = 0;
        e.ws.hoff[nh] = n;
        e.ws.hrank[nh] = nreal;
    }
}

// ---- D ----------------------------------------------------------------------------------------------
// centroid, preference mask and r^2 of VERSION i (two IEEE divisions per dimension, off the serial path).  rec: where the
// chain kernel left the record -- ver[i] (outlier side) or verp[plist position] (pcore side, see pver)
__device__ __forceinline__ void derive_version(const Eng &e, const Num &nm, int i, const double *rec) {
    const int D = nm.D, dp = e.ws.dp;
    const double w = rec[2 * dp];
    double *cen = e.ws.vcen + (size_t)i * D;
    double s = 0.0;
    uint64_t mk = 0ull;
    for (int d = 0; d < D; ++d) {
        const double a = ddiv(rec[dp + d], w);
        const double c = ddiv(rec[d], w);
        cen[d] = c;
        const double var = dsub(a, dmul(c, c));
        const bool bit = var <= nm.delta2;
        mk |= (uint64_t)bit << d;
        s = dadd(s, bit ? (nm.div_mode ? ddiv(var, nm.k) : dmul(var, nm.wsel)) : var);
    }
    e.ws.vmask[i] = mk;
    e.ws.vr2[i] = s;
}

// PCORE side: the versions k_bs_chain_p left (accepted members of the pcore chains) and the per-tile bases.  Runs, with
// k_bs_verify_p behind it, next to k_bs_olist -> k_bs_chain_o -> k_bs_derive_o (disjoint cells); skipped in a light round.
__global__ void __launch_bounds__(BS_THREADS) k_bs_derive_p(Eng e) {
    e.fetch();
    CCB_TS(10);
    CCB_PDL();
    const BsCtl *bc = e.bc;
    if (!bc->active || bc->phase != 0 || bc->pclean) return;
    const int i = blockIdx.x * BS_THREADS + threadIdx.x;
    {
        // tbase[t][j] = latest ACCEPTED member of pcore chain j before tile t (t == ntiles: of the whole block)
        const int Mp = bc->Mp, stride = e.ws.mp_stride, ntiles = (bc->Beff + 31) >> 5;
        const int total = (ntiles + 1) * Mp;
        for (int idx = i; idx < total; idx += gridDim.x * BS_THREADS) {
            const int t = idx / Mp, j = idx - t * Mp;
            const int lo = e.ws.poff[j];
            int pos = lo + (t < ntiles ? e.ws.tilecnt[(size_t)t * stride + j] : e.ws.pcnt[j]);
            while (pos > lo && e.ws.prej[e.ws.plist[pos - 1] & BS_PL_CELL]) --pos;
            e.ws.tbase[(size_t)t * stride + j] = pos > lo ? (e.ws.plist[pos - 1] & BS_PL_CELL) : -1;
        }
    }
    if (i >= bc->Beff || e.ws.pcand[i] < 0 || e.ws.prej[i]) return; // not an accepted member of a pcore chain
    derive_version(e, e.nm, i, pver(e.ws, i));
}

// OUTLIER side: the versions k_bs_chain_o left (members of the outlier-side keys, in omem)
__global__ void __launch_bounds__(BS_THREADS) k_bs_derive_o(Eng e) {
    e.fetch();
    CCB_TS(14);
    CCB_PDL();
    const BsCtl *bc = e.bc;
    if (!bc->active || bc->phase != 0) return;
    if (!bc->o_big) return; // every key was small: k_bs_chain_o derived its versions itself
    const int no = bc->no;
    for (int t = blockIdx.x * BS_THREADS + threadIdx.x; t < no; t += gridDim.x * BS_THREADS) {
        const int i = e.ws.omem[t];
        derive_version(e, e.nm, i, e.ws.ver + (size_t)i * e.ws.lsp);
    }
}

// ---- V ----------------------------------------------------------------------------------------------
// pcore stage, one CTA per tile of 32 cells (lane = cell): for every pcore MC the version it had just before each cell =
// the latest accepted member of its chain inside the tile (ballot) or before the tile (tbase).  The CTA's four warps
// take the pcore MCs j = w, w + 4, ... and warp 0 reduces (distance, list position) lexicographically = the first
// strictly smaller MC of the sequential scan; four times the warps to hide the dependent loads and adds.
constexpr int BS_VP_THREADS = 128; // (eight warps with two MCs in flight were measured slower: 37.6 vs 27.2 us, r2m)
template <int DP>
__global__ void __launch_bounds__(BS_VP_THREADS, DP <= 16 ? 5 : 1) k_bs_verify_p(Eng e) {
    e.fetch();
    CCB_TS(11);
    CCB_PDL();
    constexpr int NW = BS_VP_THREADS / 32, U = 1;
    __shared__ double s_bd[NW][32];
    __shared__ int s_best[NW][32], s_prev[NW][32];
    BsCtl *bc = e.bc;
    if (!bc->active || bc->phase != 0 || bc->pclean) return; // light round: eff / dec / pend of the pcore side stand
    const int lane = threadIdx.x & 31, part = threadIdx.x >> 5;
    const int t = blockIdx.x;
    const int Beff = bc->Beff;
    if (t * 32 >= Beff) return;
    if (t * 32 + 32 <= bc->m_exact) return; // exact since an earlier round: eff / dec of these cells stand
    const Num nm = e.nm;
    const int D = nm.D, Mp = bc->Mp;
    const int i = t * 32 + lane;
    const bool live = i < Beff;
    double x[DP];
    load_row<DP>(e.X + (bc->pos + (live ? i : t * 32)) * e.ld, D, x);
    const int myc = live ? e.ws.pcand[i] : -1;
    const bool myrej = live ? (e.ws.prej[i] != 0) : true;
    const int acc_key = (myc >= 0 && !myrej) ? myc : -1;
    const int eff = !live ? BS_KEY_NONE : (myrej ? e.ws.ospec[i] : myc);
    if (live && part == 0) e.ws.eff[i] = eff;
    int best = -1, bprev = -1;
    double bd = 0.0;
    const unsigned lt = lanemask_lt();
    const int32_t *tb = e.ws.tbase + (size_t)t * e.ws.mp_stride;
    for (int j0 = part; j0 < Mp; j0 += NW * U) {
        int prev[U];
        const double *cen[U];
        uint64_t mask[U];
        bool on[U];
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const int j = j0 + u * NW;
            on[u] = j < Mp; // warp-uniform
            const unsigned lower = __ballot_sync(0xffffffffu, on[u] && acc_key == j) & lt;
            prev[u] = lower ? (t * 32 + 31 - __clz(lower)) : (on[u] ? tb[j] : -1);
        }
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const int j = on[u] ? j0 + u * NW : 0;
            cen[u] = prev[u] >= 0 ? e.ws.vcen + (size_t)prev[u] * D : e.P.cen + (size_t)j * D;
            mask[u] = prev[u] >= 0 ? e.ws.vmask[prev[u]] : e.P.mask[j];
        }
#pragma unroll
        for (int u = 0; u < U; ++u) {
            if (!on[u]) continue;
            const int j = j0 + u * NW;
            bool feas = true;
            if (nm.pi_active) {
                const double *rec = prev[u] >= 0 ? pver(e.ws, prev[u]) : nullptr;
                const double *c1 = rec ? rec : e.P.cf1 + (size_t)j * D;
                const double *c2 = rec ? rec + e.ws.dp : e.P.cf2 + (size_t)j * D;
                const double w = rec ? rec[2 * e.ws.dp] : e.P.w[j];
                feas = feasible_regs<DP>(c1, c2, w, x, nm);
            }
            const double dv = dist_regs<DP>(x, cen[u], mask[u], nm);
            if (feas && !(dv != dv) && (best < 0 || dv < bd)) { // (j ascends within the warp: strict < keeps the first)
                best = j;
                bd = dv;
                bprev = prev[u];
            }
        }
    }
    s_bd[part][lane] = bd;
    s_best[part][lane] = best;
    s_prev[part][lane] = bprev;
    __syncthreads();
    if (part != 0 || !live) return;
#pragma unroll
    for (int p = 1; p < NW; ++p) {
        const int ob = s_best[p][lane];
        const double od = s_bd[p][lane];
        if (ob >= 0 && (best < 0 || od < bd || (od == bd && ob < best))) {
            best = ob;
            bd = od;
            bprev = s_prev[p][lane];
        }
    }
    bool acc = false;
    if (best >= 0) {
        if (eff == best) {
            acc = e.ws.vr2[i] <= nm.eps2; // this very absorb is version i of the chain
        } else {
            const double *rec = bprev >= 0 ? pver(e.ws, bprev) : nullptr;
            const double *c1 = rec ? rec : e.P.cf1 + (size_t)best * D;
            const double *c2 = rec ? rec + e.ws.dp : e.P.cf2 + (size_t)best * D;
            const double w = rec ? rec[2 * e.ws.dp] : e.P.w[best];
            double wn;
            uint64_t nmask;
            acc = tent_regs<DP>(c1, c2, w, x, nm, wn, nmask) <= nm.eps2;
        }
    }
    e.ws.upf[i] = 0;
    int mm = INT_MAX;
    if (acc) {
        e.ws.dec[i] = best;
        if (best != eff) mm = i;
    } else { // decided by k_bs_verify_o, which also reports its mismatch
        e.ws.dec[i] = BS_KEY_PENDING;
        e.ws.pbest[i] = best;
        e.ws.pend[atomicAdd(&bc->npend, 1)] = i;
    }
    // first cell of the tile whose exact decision differs from the speculation -> one atomicMin per tile
    const unsigned am = __activemask();
    mm = __reduce_min_sync(am, mm);
    if (mm != INT_MAX && lane == __ffs(am) - 1) atomicMin(&bc->m0, mm);
}

// outlier stage of the cells the pcore stage rejected.  Two layouts of the same work: with few pending cells (the steady
// state: a few hundred per block) one CTA per cell -- the scan over the modified / created keys is a chain of dependent
// loads per key (member list, version, centroid), so it is spread over 128 threads; with thousands of pending cells (cold
// start, saturated parameter corners) one WARP per cell, no block barriers.  Cells below the exact prefix of the previous
// rounds (bc->m_exact) are final and skipped.

// (1) nearest snapshot MC not modified before cell i, from the top-K list, by one warp: lane s looks at entry s.  If every
// listed candidate is stale the nearest clean MC is unknown, but no clean MC is nearer than the last list entry (BOUND):
// the decision still stands when a modified / created MC, at its exact version, beats that bound.
__device__ __forceinline__ void bs_vo_topk(const Eng &e, int i, int Mp, int Mo0, int lane, double &bd0, int &bkey0, int &status,
                                           int &bounded, double &bound) {
    bd0 = 0.0, bound = 0.0;
    bkey0 = INT_MAX, status = 0, bounded = 0; // status 2: NEED
    if (Mo0 <= 0) return;
    const int tk = e.ws.tkpos[i];
    if (tk < 0) {
        status = 2;
        return;
    }
    int o = -1;
    double dv = 0.0;
    bool clean = false;
    if (lane < BS_TOPK) {
        o = e.ws.tk_idx[(size_t)tk * BS_TOPK + lane];
        dv = e.ws.tk_dist[(size_t)tk * BS_TOPK + lane];
        clean = o >= 0 && e.ws.firstmember[o] >= i;
    }
    const unsigned valid = __ballot_sync(0xffffffffu, lane < BS_TOPK && o >= 0); // a prefix of the list
    const unsigned cl = __ballot_sync(0xffffffffu, clean);
    if (cl) {
        const int s = __ffs(cl) - 1;
        bd0 = __shfl_sync(0xffffffffu, dv, s);
        bkey0 = Mp + __shfl_sync(0xffffffffu, o, s);
    } else if (valid == (1u << BS_TOPK) - 1u) {
        bounded = 1;
        bound = __shfl_sync(0xffffffffu, dv, BS_TOPK - 1);
    }
}

// (2) lanes [sub, sub + step, ...) of the hot keys: every MC modified or created earlier in the block, at its version just
// before cell i
template <int DP>
__device__ __forceinline__ void bs_vo_scan(const Eng &e, const Num &nm, const double (&x)[DP], int i, int nh, int sub, int step,
                                           double &bd, int &bkey, int &bver) {
    const int D = nm.D;
    bd = 0.0;
    bkey = INT_MAX, bver = -1;
    for (int h = sub; h < nh; h += step) {
        if (e.ws.hfirst[h] >= i) continue;
        const int off = e.ws.hoff[h], cnt = e.ws.hoff[h + 1] - off;
        const int v = cnt == 1 ? e.ws.omem[off] : latest_before(e.ws.omem + off, cnt, i);
        const double dv = dist_regs<DP>(x, e.ws.vcen + (size_t)v * D, e.ws.vmask[v], nm);
        const int key = e.ws.hkey[h];
        if (!(dv != dv) && (bkey == INT_MAX || dv < bd || (dv == bd && key < bkey))) {
            bd = dv;
            bkey = key;
            bver = v;
        }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const double od = __shfl_xor_sync(0xffffffffu, bd, o);
        const int ok = __shfl_xor_sync(0xffffffffu, bkey, o);
        const int ov = __shfl_xor_sync(0xffffffffu, bver, o);
        if (ok != INT_MAX && (bkey == INT_MAX || od < bd || (od == bd && ok < bkey))) {
            bd = od;
            bkey = ok;
            bver = ov;
        }
    }
}

// (3) the decision, by one warp (lane = dimension in the tentative absorb)
template <int DP>
__device__ __forceinline__ void bs_vo_decide(const Eng &e, BsCtl *bc, const Num &nm, int i, int lane, int Mp, int KNEW, int Beff,
                                             int status, int bounded, double bound, double bd, int bkey, int bver) {
    const int D = nm.D;
    int dec, up = 0;
    if (status) {
        dec = BS_KEY_NEED;
    } else if (bounded && !(bkey != INT_MAX && bd < bound)) {
        dec = BS_KEY_UNKNOWN;
    } else {
        dec = KNEW + i;
        if (bkey != INT_MAX) {
            const double *c1, *c2;
            double w;
            if (bver >= 0) {
                c1 = ver_cf1(e.ws, bver);
                c2 = ver_cf2(e.ws, bver);
                w = ver_w(e.ws, bver);
            } else {
                const int o = bkey - Mp;
                c1 = e.O.cf1 + (size_t)o * D;
                c2 = e.O.cf2 + (size_t)o * D;
                w = e.O.w[o];
            }
            LaneMc m, o2;
            double xl[2];
#pragma unroll
            for (int h = 0; h < 2; ++h) {
                const int d = lane + 32 * h;
                m.cf1[h] = d < D ? c1[d] : 1.0;
                m.cf2[h] = d < D ? c2[d] : 1.0;
                m.cen[h] = 0.0;
                xl[h] = d < D ? e.X[(bc->pos + i) * e.ld + d] : 0.0;
            }
            double wn;
            uint64_t nmask;
            if (tentative_absorb_t<DP>(m, w, xl, nm, o2, wn, nmask)) {
                dec = bkey;
                const int pd = nm.cnt_gt1 ? popc64(nmask) : 0;
                up = (wn >= nm.beta_mu) && ((int64_t)pd <= nm.pi); // hddstream.py:413-418
            }
        }
    }
    if (lane == 0) {
        e.ws.dec[i] = dec;
        e.ws.upf[i] = (uint8_t)up;
        if (i < Beff) { // (a light round after a truncation still lists cells behind the cut)
            if (dec != e.ws.eff[i]) atomicMin(&bc->m0, i);
            if (up) atomicMin(&bc->up0, i);
        }
    }
}

template <int DP>
__global__ void __launch_bounds__(BS_THREADS) k_bs_verify_o(Eng e) {
    e.fetch();
    CCB_TS(15);
    CCB_PDL();
    constexpr int NW = BS_THREADS / 32;
    __shared__ double s_bd[NW];
    __shared__ int s_bkey[NW], s_bver[NW];
    BsCtl *bc = e.bc;
    if (!bc->active || bc->phase != 0) return;
    const Num nm = e.nm;
    const int D = nm.D, Mp = bc->Mp, Mo0 = bc->Mo0, KNEW = Mp + Mo0;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int npend = bc->npend, nh = bc->nh, Beff = bc->Beff, m_exact = bc->m_exact;
    if (npend > (int)gridDim.x) {
        // ---- one warp per cell
        for (int pidx = blockIdx.x * NW + warp; pidx < npend; pidx += gridDim.x * NW) {
            const int i = e.ws.pend[pidx];
            if (i < m_exact) continue;
            double x[DP];
            load_row<DP>(e.X + (bc->pos + i) * e.ld, D, x);
            double bd0, bound, bd;
            int bkey0, status, bounded, bkey, bver;
            bs_vo_topk(e, i, Mp, Mo0, lane, bd0, bkey0, status, bounded, bound);
            bs_vo_scan<DP>(e, nm, x, i, nh, lane, 32, bd, bkey, bver);
            if (!(bkey != INT_MAX && (bkey0 == INT_MAX || bd < bd0 || (bd == bd0 && bkey < bkey0)))) {
                bd = bd0;
                bkey = bkey0;
                bver = -1;
            }
            bs_vo_decide<DP>(e, bc, nm, i, lane, Mp, KNEW, Beff, status, bounded, bound, bd, bkey, bver);
        }
        return;
    }
    // ---- one CTA per cell
    for (int pidx = blockIdx.x; pidx < npend; pidx += gridDim.x) {
        const int i = e.ws.pend[pidx];
        if (i < m_exact) continue; // (block-uniform)
        double x[DP];
        load_row<DP>(e.X + (bc->pos + i) * e.ld, D, x);
        double bd0 = 0.0, bound = 0.0;
        int bkey0 = INT_MAX, status = 0, bounded = 0;
        if (warp == 0) bs_vo_topk(e, i, Mp, Mo0, lane, bd0, bkey0, status, bounded, bound);
        double bd;
        int bkey, bver;
        bs_vo_scan<DP>(e, nm, x, i, nh, tid, BS_THREADS, bd, bkey, bver);
        if (lane == 0) {
            s_bd[warp] = bd;
            s_bkey[warp] = bkey;
            s_bver[warp] = bver;
        }
        __syncthreads();
        if (warp == 0) { // the rest is one warp's work
            bd = bd0;
            bkey = bkey0;
            bver = -1;
#pragma unroll
            for (int w = 0; w < NW; ++w) {
                const double od = s_bd[w];
                const int ok = s_bkey[w];
                if (ok != INT_MAX && (bkey == INT_MAX || od < bd || (od == bd && ok < bkey))) {
                    bd = od;
                    bkey = ok;
                    bver = s_bver[w];
                }
            }
            bs_vo_decide<DP>(e, bc, nm, i, lane, Mp, KNEW, Beff, status, bounded, bound, bd, bkey, bver);
        }
        __syncthreads(); // the shared slots are reused by the next cell
    }
}

// ---- M ----------------------------------------------------------------------------------------------
#ifdef CCB_DEBUG
// diagnostics build: one record per round / per block (see tools/trace_rounds.py for the layout)
__device__ void bs_trace_round(const BsCtl *bc, int kind, int m0, int Beff_in, int nneed_in, const BsWs *ws = nullptr) {
    const int r = atomicAdd(&g_trace_n, 1);
    if (r < CCB_TRACE_MAX) {
        long long *t = g_trace[r];
        t[0] = kind; // 0 refine, 1 commit decided, 2 block finished
        t[1] = bc->pos;
        t[2] = bc->Bcur;
        t[3] = Beff_in;
        t[4] = bc->it;
        t[5] = nneed_in;
        t[6] = bc->npend;
        t[7] = bc->nh;
        t[8] = bc->no;
        t[9] = m0;
        t[10] = bc->upgrade;
        t[11] = bc->pclean; // (of the NEXT round when kind == 0)
        t[12] = bc->m_commit;
        t[13] = bc->Mp;
        t[14] = bc->Mo0;
        t[15] = bc->hnew0;
        t[16] = bc->nneed;
        t[17] = bc->Beff;
        t[18] = globaltimer_ns();
        for (int k = 0; k < CCB_TRACE_SLOTS; ++k) t[20 + k] = g_trace_ts[k];
        t[19] = bc->Mo0;
        if (ws && kind < 2 && m0 >= 0 && m0 < Beff_in) { // the first mismatching cell, as the round left it
            t[60] = ws->dec[m0];
            t[61] = ws->eff[m0];
            t[62] = ws->pcand[m0];
            t[63] = (ws->pflag[m0] != 0) | (ws->prej[m0] << 1) | ((long long)(unsigned)ws->ospec[m0] << 8) | ((long long)ws->tkpos[m0] << 40);
        }
    }
    for (int k = 3; k < CCB_TRACE_SLOTS; ++k) g_trace_ts[k] = 0;
}
#endif
__device__ __forceinline__ int block_min_1024(int v, int *s_warp) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = min(v, __shfl_xor_sync(0xffffffffu, v, o));
    if ((threadIdx.x & 31) == 0) s_warp[threadIdx.x >> 5] = v;
    __syncthreads();
    v = s_warp[threadIdx.x & 31];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = min(v, __shfl_xor_sync(0xffffffffu, v, o));
    __syncthreads();
    return v;
}

__global__ void __launch_bounds__(BS_CTA1, 1) k_bs_decide(Eng e) {
    e.fetch();
    CCB_TS(16);
    CCB_PDL();
    __shared__ int s_warp[33];
    __shared__ int s_act, s_cut;
    BsCtl *bc = e.bc;
    if (!bc->active || bc->phase != 0) return;
    const int tid = threadIdx.x;
    const int Beff = bc->Beff, Mp = bc->Mp, KNEW = bc->Mp + bc->Mo0;
    // first cell whose exact decision differs from the speculation, first upgrade inside the exact prefix: both were
    // reduced with atomicMin by the verify kernels; consume and re-arm them
    __shared__ int s_m0, s_up;
    if (tid == 0) {
        s_m0 = min(bc->m0, Beff);
        s_up = bc->up0;
        bc->m0 = bc->up0 = INT_MAX;
    }
    __syncthreads();
    const int m0 = s_m0;
    const int up = s_up < m0 ? s_up : INT_MAX;
    constexpr int SU = 8;
    if (tid == 0) {
        int act = 0; // 0 refine, 1 commit
        bc->iters += 1;
        bc->replayed += bc->pclean ? bc->npend : Beff;
        if (up != INT_MAX) {
            bc->m_commit = up + 1;
            bc->upgrade = 1;
            act = 1;
        } else if (m0 == Beff) {
            bc->m_commit = Beff;
            act = 1;
        } else {
            bc->mismatches += 1;
            const int d0 = e.ws.dec[m0];
            if (d0 == BS_KEY_UNKNOWN) {
                bc->m_commit = m0;
                bc->cuts_unknown += 1;
                act = 1;
            } else if (bc->it + 1 >= bc->itmax) {
                bc->m_commit = m0;
                bc->cuts_iter += 1;
                act = 1;
            }
        }
        s_act = act;
        s_cut = Beff;
    }
    __syncthreads();
    if (s_act == 1) {
        if (tid == 0) {
            bc->phase = 1;
            bc->tk_lo = bc->tk_hi = 0;
            if (e.h_inner) cudaGraphSetConditional(e.h_inner, 0u);
            CCB_DBG(bs_trace_round(bc, 1, m0, Beff, bc->nneed, &e.ws);)
        }
        return;
    }
    CCB_DBG(__shared__ long long s_dbg[4]; if (tid == 0) {
        s_dbg[0] = e.ws.dec[m0];
        s_dbg[1] = e.ws.eff[m0];
        s_dbg[2] = e.ws.pcand[m0];
        s_dbg[3] = (e.ws.pflag[m0] != 0) | (e.ws.prej[m0] << 1) | ((long long)(unsigned)e.ws.ospec[m0] << 8) | ((long long)e.ws.tkpos[m0] << 40);
    })
    // ---- refinement: the recomputed decisions of [m0, Beff) become the next speculation
    int cut = Beff;
    for (int i0 = m0 + tid; i0 < Beff && cut == Beff; i0 += BS_CTA1 * SU) {
        int dv[SU];
#pragma unroll
        for (int u = 0; u < SU; ++u) {
            const int i = i0 + u * BS_CTA1;
            dv[u] = i < Beff ? e.ws.dec[i] : 0;
        }
#pragma unroll
        for (int u = SU - 1; u >= 0; --u)
            if (dv[u] == BS_KEY_UNKNOWN) cut = i0 + u * BS_CTA1;
    }
    cut = block_min_1024(cut, s_warp);
    // A refinement that only moves cells between OUTLIER-SIDE keys leaves the pcore side of the next round exactly
    // as it is now (same candidates, flags, accepts, hence the same pcore versions, eff / dec of the accepted cells
    // and the same list of pcore-rejected cells): that round re-runs the outlier side only (bc->pclean).
    //
    // Pass 1, all threads striding, no barriers: every differing cell that does NOT need a new top-K slot takes its
    // recomputed decision as the next speculation.  (If pass 2 truncates the block, cells behind the cut have been
    // rewritten for nothing: they are outside the block from now on and every block starts from a fresh speculation.)
    const int nneed_old = bc->nneed;
    const int32_t row0 = (int32_t)bc->pos;
    int base = nneed_old;
    int dirty = 0, any_want = 0;
    constexpr int PU = 4;
    for (int i0 = m0 + tid; i0 < cut; i0 += BS_CTA1 * PU) {
        int dv[PU], ev[PU];
#pragma unroll
        for (int u = 0; u < PU; ++u) {
            const int i = i0 + u * BS_CTA1;
            dv[u] = i < cut ? e.ws.dec[i] : 0;
            ev[u] = i < cut ? e.ws.eff[i] : 0;
        }
#pragma unroll
        for (int u = 0; u < PU; ++u) {
            const int i = i0 + u * BS_CTA1, dc = dv[u], ef = ev[u];
            if (dc == ef) continue; // (also the padding past cut)
            const bool want = dc == BS_KEY_NEED || (dc >= 0 && dc < Mp && e.ws.pcand[i] != dc && !e.ws.pflag[i]);
            if (want) {
                any_want = 1;
                continue;
            }
            if (dc < Mp) {
                e.ws.pcand[i] = dc;
            } else {
                e.ws.ospec[i] = dc;
                e.ws.pflag[i] = 1;
                // speculated "absorbed by a pcore MC", exact "rejected by the pcore stage": the exact test was the one of the
                // NEAREST pcore MC at its exact version, which need not be the speculated one -- the replay has to put the
                // cell to the test in that chain (the chain it sat in may well accept it again, round after round)
                if (ef < Mp) {
                    const int pb = e.ws.pbest[i];
                    e.ws.pcand[i] = pb;
                    if (pb < 0) e.ws.prej[i] = 1; // no feasible pcore MC at all: straight to the outlier stage
                }
            }
            if (ef >= Mp && dc >= Mp) e.ws.eff[i] = dc; // what k_bs_verify_p would record for this (rejected) cell
            else dirty = 1;
        }
    }
    any_want = __syncthreads_or(any_want);
    // Pass 2, only when some cell needs a (new) top-K slot -- a cell that reaches the outlier stage without a list, or a
    // SAFE cell whose nearest pcore MC changed (it becomes CONTESTED, which needs a fallback outlier decision should the
    // chain reject it): slots are handed out in cell order, 1024 cells at a time; the block is truncated at the first
    // cell that finds the list full.
    for (int c0 = m0; any_want && c0 < cut; c0 += BS_CTA1) {
        const int i = c0 + tid;
        int dc = 0;
        bool want = false;
        if (i < cut) {
            dc = e.ws.dec[i];
            want = dc != e.ws.eff[i] &&
                   (dc == BS_KEY_NEED || (dc >= 0 && dc < Mp && e.ws.pcand[i] != dc && !e.ws.pflag[i]));
        }
        const int nwant = __syncthreads_count(want);
        if (!nwant) continue; // uniform
        int total;
        const int slot = base + block_exclusive_scan_1024(want ? 1 : 0, s_warp, total);
        if (want && slot >= BS_RMAX) atomicMin(&s_cut, i);
        __syncthreads();
        if (want && i < s_cut) {
            e.ws.tkpos[i] = slot;
            e.ws.nrows[slot] = row0 + i;
            e.ws.ncell[slot] = i;
            e.ws.ospec[i] = KNEW + i; // provisional: create; the next round decides with the top-K list
            e.ws.pflag[i] = 1;
            if (dc != BS_KEY_NEED) e.ws.pcand[i] = dc;
            dirty = 1;
        }
        base += nwant;
        if (s_cut < Beff) break; // uniform: s_cut was read after the barrier
    }
    dirty = __syncthreads_or(dirty);
    const int Bnew = min(cut, s_cut);
    if (tid == 0) {
        if (Bnew <= m0) { // the first mismatching cell itself cannot be refined: commit the exact prefix
            bc->m_commit = m0;
            bc->cuts_cap += 1;
            bc->phase = 1;
            bc->tk_lo = bc->tk_hi = 0;
        } else {
            const int nneed_new = min(base, BS_RMAX);
            bc->tk_lo = nneed_old;
            bc->tk_hi = nneed_new;
            bc->nneed = nneed_new;
            bc->tk_late += nneed_new - nneed_old;
            bc->pairs += (int64_t)(nneed_new - nneed_old) * bc->Mo0;
            bc->Beff = Bnew;
            bc->m_exact = m0; // every cell before the first mismatch saw exact versions: final from here on
            bc->it += 1;
            bc->pclean = dirty ? 0 : 1;
            if (dirty) bc->npend = 0; // a light round keeps the list of pcore-rejected cells
            else bc->rounds_light += 1;
        }
        if (e.h_inner) cudaGraphSetConditional(e.h_inner, bc->phase == 0 ? 1u : 0u);
        CCB_DBG(bs_trace_round(bc, 0, m0, Beff, nneed_old, nullptr); if (g_trace_n - 1 < CCB_TRACE_MAX) for (int q = 0; q < 4; ++q) g_trace[g_trace_n - 1][60 + q] = s_dbg[q];)
    }
}

// ---- commit -----------------------------------------------------------------------------------------
// one warp per key: the last version before m_commit becomes the stored state of the MC
__device__ __forceinline__ void commit_row(const Eng &e, const BsCtl *bc, const Num &nm, int kidx, int lane, int Mp, int Mo0,
                                           int KNEW, int m) {
    const int D = nm.D, DP = nm.DP;
    if (kidx < Mp) {
        const int j = kidx, tm = m >> 5;
        const int i = tm * 32 + lane;
        const bool accd = i < m && e.ws.pcand[i] == j && !e.ws.prej[i];
        const unsigned mk = __ballot_sync(0xffffffffu, accd);
        const int v = mk ? (tm * 32 + 31 - __clz(mk)) : e.ws.tbase[(size_t)tm * e.ws.mp_stride + j];
        if (v < 0) return;
        const double *rec = pver(e.ws, v);
        for (int d = lane; d < D; d += 32) {
            e.P.cf1[(size_t)j * D + d] = rec[d];
            e.P.cf2[(size_t)j * D + d] = rec[e.ws.dp + d];
            e.P.cen[(size_t)j * D + d] = e.ws.vcen[(size_t)v * D + d];
        }
        if (lane == 0) {
            e.P.w[j] = rec[2 * e.ws.dp];
            e.P.mask[j] = e.ws.vmask[v];
        }
        return;
    }
    const int h = kidx - Mp;
    if (h >= bc->nh) return;
    const int32_t *mem = e.ws.omem + e.ws.hoff[h];
    if (mem[0] >= m) return;
    const int v = latest_before(mem, e.ws.hoff[h + 1] - e.ws.hoff[h], m);
    const int key = e.ws.hkey[h];
    const bool created = key >= KNEW;
    if (created && mem[0] != key - KNEW) return; // phantom key (cannot reach into the exact prefix)
    const int rank = created ? e.ws.newrank[key - KNEW] : 0;
    const int slot = created ? Mo0 + rank : key - Mp;
    const uint64_t mask = e.ws.vmask[v];
    for (int d = lane; d < DP; d += 32) {
        double2 cv;
        cv.x = 0.0;
        cv.y = 1.0;
        if (d < D) {
            const double c = e.ws.vcen[(size_t)v * D + d];
            e.O.cf1[(size_t)slot * D + d] = ver_cf1(e.ws, v)[d];
            e.O.cf2[(size_t)slot * D + d] = ver_cf2(e.ws, v)[d];
            e.O.cen[(size_t)slot * D + d] = c;
            cv.x = c;
            cv.y = ((mask >> d) & 1ull) ? nm.wsel : 1.0;
        }
        e.O.cw[(size_t)slot * DP + d] = cv;
    }
    if (lane == 0) {
        e.O.w[slot] = ver_w(e.ws, v);
        e.O.mask[slot] = mask;
        if (created) {
            const int64_t id = e.ctl->outlier_last_id + rank;
            e.O.id[slot] = id;
            e.O.uid[slot] = (int32_t)id;
        }
    }
}

// The three steps of the commit in ONE launch: the first `rows_ctas` CTAs write the rows back (one warp per key), the
// others the per-cell results; the last CTA to finish (ticket) applies the upgrade (hddstream.py:397-430) and advances the
// list lengths, id counters and the block cursor.
__device__ __forceinline__ void bs_finish_block(const Eng &e, BsCtl *bc);

__global__ void __launch_bounds__(BS_THREADS) k_bs_commit(Eng e, int rows_ctas) {
    e.fetch();
    CCB_TS(17);
    CCB_PDL();
    __shared__ int s_last;
    BsCtl *bc = e.bc;
    if (!bc->active || bc->phase != 1) return;
    const int Mp = bc->Mp, Mo0 = bc->Mo0, KNEW = Mp + Mo0, m = bc->m_commit;
    if ((int)blockIdx.x < rows_ctas) {
        const Num nm = e.nm;
        const int kidx = blockIdx.x * (BS_THREADS / 32) + (threadIdx.x >> 5);
        commit_row(e, bc, nm, kidx, threadIdx.x & 31, Mp, Mo0, KNEW, m);
    } else {
        const int i = (blockIdx.x - rows_ctas) * BS_THREADS + threadIdx.x;
        if (i < m) {
            const int key = e.ws.eff[i];
            int32_t uid;
            uint8_t st;
            if (key < Mp) {
                uid = e.P.uid[key];
                st = 0;
            } else if (key < KNEW) {
                uid = e.O.uid[key - Mp];
                st = 1;
            } else {
                const int c = key - KNEW;
                uid = (int32_t)(e.ctl->outlier_last_id + e.ws.newrank[c]);
                st = c == i ? 3 : 1;
            }
            if (bc->upgrade && i == m - 1) st = 2;
            e.assign[bc->pos + i] = uid;
            if (e.stage) e.stage[bc->pos + i] = st;
        }
    }
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) s_last = atomicAdd(&bc->ticket_c, 1) == (int)gridDim.x - 1;
    __syncthreads();
    if (!s_last) return;
    __threadfence();
    bs_finish_block(e, bc);
}

// upgrade (hddstream.py:397-430), list lengths, id counters, next block length
__device__ __forceinline__ void bs_finish_block(const Eng &e, BsCtl *bc) {
    __shared__ int s_ncreated;
    Ctl *ctl = e.ctl;
    const Num nm = e.nm;
    const int D = nm.D, DP = nm.DP, tid = threadIdx.x;
    const int Mp = bc->Mp, Mo0 = bc->Mo0, KNEW = Mp + Mo0, m = bc->m_commit;
    const int nh = bc->nh, hnew0 = bc->hnew0;
    if (tid == 0) { // creations committed = created-in-block keys whose creator is < m (keys ascend with the creator)
        int lo = hnew0, hi = nh;
        while (lo < hi) {
            const int mid = (lo + hi) >> 1;
            if (e.ws.hkey[mid] - KNEW < m) lo = mid + 1;
            else hi = mid;
        }
        s_ncreated = e.ws.hrank[lo];
    }
    for (int h = tid; h < nh; h += BS_THREADS) { // forget the modified-flags of this block
        const int key = e.ws.hkey[h];
        if (key < KNEW) e.ws.firstmember[key - Mp] = INT_MAX;
    }
    __syncthreads();
    const int ncreated = s_ncreated;
    int slot = -1;
    if (bc->upgrade) {
        const int key = e.ws.eff[m - 1];
        slot = key < KNEW ? key - Mp : Mo0 + e.ws.newrank[key - KNEW];
        const int pj = Mp;
        for (int d = tid; d < D; d += BS_THREADS) {
            e.P.cf1[(size_t)pj * D + d] = e.O.cf1[(size_t)slot * D + d];
            e.P.cf2[(size_t)pj * D + d] = e.O.cf2[(size_t)slot * D + d];
            e.P.cen[(size_t)pj * D + d] = e.O.cen[(size_t)slot * D + d];
        }
    }
    __syncthreads();
    if (tid == 0) {
        if (slot >= 0) {
            const int pj = Mp;
            e.P.w[pj] = e.O.w[slot];
            e.P.mask[pj] = e.O.mask[slot];
            e.P.uid[pj] = e.O.uid[slot];
            e.P.id[pj] = ctl->pcore_last_id;
            ctl->pcore_last_id += 1;
            ctl->n_pcore = pj + 1;
            e.O.w[slot] = -1.0; // tombstone (a live weight is never negative); NaN keeps it out of kernel 1
            e.O.cw[(size_t)slot * DP].x = __longlong_as_double(0x7ff8000000000000LL);
            ctl->n_outlier_alive -= 1;
            ctl->upgrades += 1;
        }
        ctl->n_outlier = Mo0 + ncreated;
        ctl->n_outlier_alive += ncreated;
        ctl->outlier_last_id += ncreated;
        ctl->created += ncreated;
        bc->pos += m;
        bc->blocks += 1;
        if (m == bc->Bcur) bc->next_B = min(bc->next_B * 2, bc->Bmax);
        else if (!bc->upgrade) bc->next_B = max(bc->next_B / 2, bc->Bmin);
        CCB_DBG(bs_trace_round(bc, 2, m, ncreated, bc->nneed);)
        bc->nh = 0;
        bc->ticket_c = 0;
        bc->active = 0;
        if (bc->pos >= bc->N) bc->done = 1;
        if (e.h_outer) cudaGraphSetConditional(e.h_outer, bc->done ? 0u : 1u);
    }
}

} // namespace ccb
