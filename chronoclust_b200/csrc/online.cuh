// online.cuh -- device-side state of the ordered online phase and KERNEL 3 (decay / downgrade / compaction).
//
// The state replaces the two ordered lists of HDDStream (clustering/hddstream.py:56-64: pcore_MC, outlier_MC and the id
// counters) and the Microcluster objects in them (objects/microcluster.py:71-81) as structure-of-arrays stores whose
// physical order is the list order.  The ordered per-cell loop itself (hddstream.py:220-237) is KERNEL 2, the
// block-speculative versioned commit of engine.cuh; this file holds what it shares with the rest of the library
// (stores, control block, numeric parameters, the warp-held tentative absorb) and the timepoint-start maintenance:
//
// Kernel 3   k_maint_plan + k_maint_gather: fused decay x 2^(-lambda dt) (hddstream.py:247-286), downgrade with the
//            reference's skip-next-after-removal iteration and outlier deletion (hddstream.py:512-549), order-preserving
//            compaction.
// Input      k_stage_rows / k_colminmax: float32 / float64 rows (optionally a subset of their columns) widened to double,
//            optionally arcsinh(x / cofactor) transformed (asinh.h) and min-max transformed, and the fit
//            reductions (scaling/scaler.py:11-53).
#pragma once
#include "common.cuh"
#include "asinh.h"

namespace ccb {

// Device-resident control block shared by the host and the kernels.
struct Ctl {
    int32_t n_pcore, n_outlier; // physical list lengths (outlier list includes tombstones)
    int32_t n_outlier_alive, pad0;
    int64_t pcore_last_id, outlier_last_id;
    int64_t upgrades, created;
    int32_t new_n_pcore, new_n_outlier; // kernel 3 plan output
    int64_t downgraded, deleted;
};

struct Store { // one ordered MC list, physical order == list order
    double *cf1, *cf2, *cen; // [cap][D]
    double *w;               // [cap]
    uint64_t *mask;          // [cap]  bit d <=> preferred_dimension_vector[d] == k
    int64_t *id;             // [cap]
    int32_t *uid;            // [cap]  prev_outlier_id (unique per creation)
    double2 *cw;             // [cap][DP] packed (centroid, weight) rows for kernel 1 (outlier list only)
    int32_t cap;
};

struct Num { // numeric parameters common to the ordered kernels
    double delta2, k, wsel, eps2, beta_mu;
    int64_t pi;
    int32_t D, DP, div_mode, pi_active, cnt_gt1; // cnt_gt1: k > 1 (count(pref > 1) == popc(mask)) else 0
};

// ---------------------------------------------------------------------------------------------------
// An MC held by a warp: lane d owns dims d and d + 32.
struct LaneMc {
    double cf1[2], cf2[2], cen[2];
};
// 8-byte asynchronous global->shared copy (LDGSTS); used to prefetch the next wave's cells transposed
__device__ __forceinline__ void cp_async8(void *dst_smem, const void *src) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(smem_u32(dst_smem)), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async_commit_wait_all() {
    asm volatile("cp.async.commit_group;\ncp.async.wait_group 0;" ::: "memory");
}

// Tentative absorb held by one warp, lane d owns dims d and d+32; the D radius terms are summed in index
// order by every lane redundantly from warp-shuffle broadcasts (no shared memory, no barrier).
template <int DP>
__device__ __forceinline__ bool tentative_absorb_t(const LaneMc &m, double w, const double x[2], const Num &nm,
                                                   LaneMc &o, double &wn, uint64_t &nmask) {
    const int lane = threadIdx.x & 31;
    wn = dadd(w, 1.0);
    uint32_t bits[2] = {0u, 0u};
    double term[2] = {0.0, 0.0};
#pragma unroll
    for (int h = 0; h < 2; ++h) {
        if (h == 0 || DP > 32) {
            const int d = lane + 32 * h;
            // idle lanes (d >= D) carry CF = 1 so that their (discarded) quotients stay on the fast path of the
            // IEEE division; a zero dividend would drag the whole warp through the slow-path subroutine
            const bool act = d < nm.D;
            o.cf1[h] = dadd(m.cf1[h], x[h]);
            o.cf2[h] = dadd(m.cf2[h], dmul(x[h], x[h]));
            const double a = ddiv(o.cf2[h], wn);
            const double c = ddiv(o.cf1[h], wn);
            o.cen[h] = c;
            const double var = dsub(a, dmul(c, c));
            const bool bit = act && (var <= nm.delta2);
            term[h] = bit ? (nm.div_mode ? ddiv(var, nm.k) : dmul(var, nm.wsel)) : var;
            bits[h] = __ballot_sync(0xffffffffu, bit);
        }
    }
    nmask = (uint64_t)bits[0] | ((uint64_t)bits[1] << 32);
    double s = 0.0;
#pragma unroll
    for (int d = 0; d < DP; ++d) {
        if (d < nm.D) s = dadd(s, __shfl_sync(0xffffffffu, term[d >> 5], d & 31));
    }
    return s <= nm.eps2;
}

// ---------------------------------------------------------------------------------------------------
// Kernel 3.  Plan: one CTA decides, for the decayed weights, which pcore MCs are downgraded and which
// outlier MCs are deleted, reproducing Python's mutate-while-iterating behaviour: an element is examined
// iff the element before it (in the current list) was not just removed (hddstream.py:528-537, 545-549).
// removed[j] = cond[j] && !removed[j-1]  -- a two-state machine, composed across threads.
// Output: new position of every old pcore / outlier slot (-1 = gone; downgraded pcore MCs get a position in
// the NEW outlier list encoded as -2 - newpos).
struct MaintArgs {
    Store P, O, P2, O2; // old and new (ping-pong) stores
    Ctl *ctl;
    int32_t *p_new, *p_fin, *o_new; // [P.cap] phase-1 codes, [P.cap] final codes, [O.cap]
    double f, beta_mu, omicron;
    int64_t pi;
    int32_t D, DP, cnt_gt1;
    double wsel;
};

constexpr int MAINT_THREADS = 1024;

__global__ void __launch_bounds__(MAINT_THREADS, 1) k_maint_plan(MaintArgs a) {
    __shared__ int s_cnt[MAINT_THREADS];
    __shared__ unsigned char s_out0[MAINT_THREADS], s_out1[MAINT_THREADS], s_in[MAINT_THREADS];
    __shared__ int s_nmoved, s_np_new;
    const int tid = threadIdx.x;
    Ctl *ctl = a.ctl;
    const int np = ctl->n_pcore, no = ctl->n_outlier;
    // ---- pcore pass (short list): one thread walks it
    if (tid == 0) {
        int prev_removed = 0, keep = 0, moved = 0;
        for (int j = 0; j < np; ++j) {
            const double w = dmul(a.P.w[j], a.f);
            const int pd = a.cnt_gt1 ? popc64(a.P.mask[j]) : 0;
            const int cond = (w < a.beta_mu) || ((int64_t)pd > a.pi);
            const int rem = cond && !prev_removed;
            a.p_new[j] = rem ? (-2 - moved) : keep;
            a.p_fin[j] = keep; // overwritten below for downgraded MCs
            moved += rem;
            keep += !rem;
            prev_removed = rem;
        }
        s_nmoved = moved;
        s_np_new = keep;
    }
    __syncthreads();
    const int nmoved = s_nmoved;
    // ---- outlier pass over the sequence: live old outliers in order, then the downgraded pcores in order
    const int total = no + nmoved;
    const int per = (total + MAINT_THREADS - 1) / MAINT_THREADS;
    const int lo = min(total, tid * per), hi = min(total, lo + per);
    auto elem = [&](int e, bool &live, bool &cond) {
        if (e < no) {
            const double w0 = a.O.w[e];
            live = w0 >= 0.0; // tombstones carry -1
            cond = live && (dmul(w0, a.f) <= a.omicron);
        } else {
            // e - no-th downgraded pcore: find it (np is small)
            int k = e - no, jj = -1;
            for (int j = 0; j < np; ++j)
                if (a.p_new[j] == -2 - k) {
                    jj = j;
                    break;
                }
            live = true;
            cond = dmul(a.P.w[jj], a.f) <= a.omicron;
        }
    };
    {
        int st0 = 0, st1 = 1; // removed-state of the previous live element, for both possible inputs
        for (int e = lo; e < hi; ++e) {
            bool live, cond;
            elem(e, live, cond);
            if (!live) continue;
            st0 = cond && !st0;
            st1 = cond && !st1;
        }
        s_out0[tid] = (unsigned char)st0;
        s_out1[tid] = (unsigned char)st1;
    }
    __syncthreads();
    if (tid == 0) {
        int st = 0;
        for (int t = 0; t < MAINT_THREADS; ++t) {
            s_in[t] = (unsigned char)st;
            st = st ? s_out1[t] : s_out0[t];
        }
    }
    __syncthreads();
    int kept = 0;
    {
        int st = s_in[tid];
        for (int e = lo; e < hi; ++e) {
            bool live, cond;
            elem(e, live, cond);
            if (!live) continue;
            st = cond && !st;
            kept += !st;
        }
    }
    s_cnt[tid] = kept;
    __syncthreads();
    if (tid == 0) {
        int run = 0;
        for (int t = 0; t < MAINT_THREADS; ++t) {
            const int c = s_cnt[t];
            s_cnt[t] = run;
            run += c;
        }
        ctl->new_n_outlier = run;
        ctl->new_n_pcore = s_np_new;
        ctl->downgraded += nmoved;
    }
    __syncthreads();
    {
        int st = s_in[tid], posn = s_cnt[tid], ndel = 0;
        for (int e = lo; e < hi; ++e) {
            bool live, cond;
            elem(e, live, cond);
            int np_ = -1;
            if (live) {
                st = cond && !st;
                if (!st) np_ = posn++;
                else ++ndel;
            }
            if (e < no) {
                a.o_new[e] = np_;
            } else {
                const int k = e - no;
                for (int j = 0; j < np; ++j)
                    if (a.p_new[j] == -2 - k) {
                        // encode: moved and kept at outlier position np_  ->  -2 - np_ ; moved and deleted -> -1
                        a.p_fin[j] = np_ >= 0 ? (-2 - np_) : -1;
                        break;
                    }
            }
        }
        if (ndel) atomicAdd(reinterpret_cast<unsigned long long *>(&ctl->deleted), (unsigned long long)ndel);
    }
}

// Gather: writes the new (compacted, decayed) stores.  CF1, CF2, W are scaled by f; centroid and preference
// vector are NOT touched (hddstream.py:268-286, asserted by the reference's unittest_hddstream.py:90-121).
__global__ void k_maint_gather(MaintArgs a) {
    const Ctl *ctl = a.ctl;
    const int np = ctl->n_pcore, no = ctl->n_outlier;
    const int D = a.D, DP = a.DP;
    const int64_t total = (int64_t)(np + no) * DP;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        const int e = (int)(i / DP), d = (int)(i % DP);
        const bool from_p = e < np;
        const int j = from_p ? e : e - np;
        const Store &S = from_p ? a.P : a.O;
        const int code = from_p ? a.p_fin[j] : a.o_new[j];
        if (code == -1) continue;
        const bool to_p = from_p && code >= 0;
        const int nj = to_p ? code : (from_p ? (-2 - code) : code);
        const Store &T = to_p ? a.P2 : a.O2;
        if (d < D) {
            T.cf1[(size_t)nj * D + d] = dmul(S.cf1[(size_t)j * D + d], a.f);
            T.cf2[(size_t)nj * D + d] = dmul(S.cf2[(size_t)j * D + d], a.f);
            T.cen[(size_t)nj * D + d] = S.cen[(size_t)j * D + d];
        }
        if (!to_p) {
            double2 cv;
            cv.x = d < D ? S.cen[(size_t)j * D + d] : 0.0;
            cv.y = (d < D && ((S.mask[j] >> d) & 1ull)) ? a.wsel : 1.0;
            T.cw[(size_t)nj * DP + d] = cv;
        }
        if (d == 0) {
            T.w[nj] = dmul(S.w[j], a.f);
            T.mask[nj] = S.mask[j];
            T.uid[nj] = S.uid[j];
            T.id[nj] = (from_p && !to_p) ? (int64_t)S.uid[j] : S.id[j]; // downgrade: id <- [prev_outlier_id]
        }
    }
}

__global__ void k_maint_finish(Ctl *ctl) {
    ctl->n_pcore = ctl->new_n_pcore;
    ctl->n_outlier = ctl->new_n_outlier;
    ctl->n_outlier_alive = ctl->new_n_outlier;
}

// Rebuilds the packed (centroid, weight) rows of a store (after an import).
__global__ void k_repack_store(Store S, int n, int D, int DP, double wsel) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (int64_t)n * DP) return;
    const int j = (int)(i / DP), d = (int)(i % DP);
    double2 cv;
    cv.x = d < D ? S.cen[(size_t)j * D + d] : 0.0;
    cv.y = (d < D && ((S.mask[j] >> d) & 1ull)) ? wsel : 1.0;
    S.cw[i] = cv;
}

// ---- input staging and scaler (SURVEY 8f-3; scaling/scaler.py:11-53 -> sklearn MinMaxScaler) --------------------
// Rows of T (float or double, leading dimension ld_src in elements of T) -> double rows (leading dimension ld_dst).  Every
// element is widened to double first, which is exact; with a scaler the min-max transform follows as TWO roundings
// (sklearn: `X *= self.scale_; X += self.min_`), so results equal those of widening and scaling on the host.  src == dst
// (T = double, ld_src == ld_dst) scales the device copy of a timepoint in place: every element is read and written by
// the same thread, hence no __restrict__ on src / dst.  HBM-bound: 8 + 8 B (double) or 4 + 8 B (float) per element.
// cols (device [D], or null = the identity): output column d is source column cols[d].  The map sits in shared memory; a
// warp's 32 consecutive outputs still read from one or two source rows, so the reads of a row stay coalesced.
// k_stage_rows_tx: the same with the arcsinh transform.  cof (device, indexed by SOURCE column) holds the cofactors, and
// a column with cofactor c != 0 gets ccb_asinh(x / c) after the widening and before the scaler -- one IEEE division, then
// asinh.h's restatement of fdlibm, which gives the host's bits.  The cofactors of the D output columns sit in shared
// memory.  With no map and no scaler this is ccb_arcsinh's kernel.  (Two kernels over one body: the untransformed inputs
// keep a kernel of their own, with its own register allocation.)
template <typename T, bool TX>
__device__ __forceinline__ void stage_rows_body(const T *src, int64_t ld_src, double *dst, int64_t ld_dst, int64_t N, int D,
                                                const int32_t *__restrict__ cols, const double *__restrict__ cof,
                                                const double *__restrict__ scale, const double *__restrict__ shift) {
    __shared__ int32_t s_col[CCB_MAX_D];
    __shared__ double s_cof[TX ? CCB_MAX_D : 1];
    auto rows = [&](auto col_of) { // (one loop body, instantiated for the identity and for the map)
        const int64_t total = N * D;
        for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
            const int64_t r = e / D;
            const int d = (int)(e - r * D);
            double x = (double)src[r * ld_src + col_of(d)];
            if constexpr (TX) {
                const double c = s_cof[d];
                if (c != 0.0) x = ccb_asinh(ddiv(x, c));
            }
            if (scale) x = dadd(dmul(x, scale[d]), shift[d]);
            dst[r * ld_dst + d] = x;
        }
    };
    if constexpr (TX) {
        for (int d = threadIdx.x; d < D; d += blockDim.x) s_cof[d] = cof[cols ? cols[d] : d];
        if (!cols) __syncthreads();
    }
    if (cols) {
        for (int d = threadIdx.x; d < D; d += blockDim.x) s_col[d] = cols[d];
        __syncthreads();
        rows([&](int d) { return s_col[d]; });
    } else {
        rows([](int d) { return d; });
    }
}
template <typename T>
__global__ void k_stage_rows(const T *src, int64_t ld_src, double *dst, int64_t ld_dst, int64_t N, int D,
                             const int32_t *__restrict__ cols, const double *__restrict__ scale,
                             const double *__restrict__ shift) {
    stage_rows_body<T, false>(src, ld_src, dst, ld_dst, N, D, cols, nullptr, scale, shift);
}
template <typename T>
__global__ void k_stage_rows_tx(const T *src, int64_t ld_src, double *dst, int64_t ld_dst, int64_t N, int D,
                                const int32_t *__restrict__ cols, const double *__restrict__ cof,
                                const double *__restrict__ scale, const double *__restrict__ shift) {
    stage_rows_body<T, true>(src, ld_src, dst, ld_dst, N, D, cols, cof, scale, shift);
}

// fit: column-wise minimum / maximum ignoring NaN (np.nanmin / np.nanmax, what MinMaxScaler.partial_fit uses).
// Doubles are compared through the order-preserving map to unsigned integers, so that one atomicMin / atomicMax per
// column and CTA settles the result exactly.  okey[D] / okey[D + d]: running min / max keys (initialised by the caller).
__device__ __forceinline__ unsigned long long ordered_key(double v) {
    const unsigned long long b = (unsigned long long)__double_as_longlong(v);
    return (b >> 63) ? ~b : (b | 0x8000000000000000ull);
}
template <typename T>
__global__ void k_colminmax(const T *__restrict__ X, int64_t N, int64_t ld, int D, unsigned long long *okey) {
    __shared__ unsigned long long s_min[CCB_MAX_D], s_max[CCB_MAX_D];
    for (int d = threadIdx.x; d < D; d += blockDim.x) {
        s_min[d] = ~0ull;
        s_max[d] = 0ull;
    }
    __syncthreads();
    // a stride that is a multiple of D keeps every thread on one column: the first floor(threads / D) * D threads take
    // part (D <= 64 < 256, so that is never zero) and together cover every flat index exactly once per stride window
    const int64_t total = N * D;
    const int64_t stride = ((int64_t)gridDim.x * blockDim.x) / D * D;
    const int64_t e0 = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e0 < stride && e0 < total) {
        const int d = (int)(e0 % D);
        unsigned long long lo = ~0ull, hi = 0ull;
        for (int64_t e = e0; e < total; e += stride) {
            const double v = (double)X[(e / D) * ld + d]; // widened first (exact): the keys are those of the doubles
            if (v == v) { // not NaN
                const unsigned long long k = ordered_key(v);
                lo = k < lo ? k : lo;
                hi = k > hi ? k : hi;
            }
        }
        if (lo <= hi) {
            atomicMin(&s_min[d], lo);
            atomicMax(&s_max[d], hi);
        }
    }
    __syncthreads();
    for (int d = threadIdx.x; d < D; d += blockDim.x) {
        if (s_min[d] <= s_max[d]) {
            atomicMin(&okey[d], s_min[d]);
            atomicMax(&okey[D + d], s_max[d]);
        }
    }
}
__global__ void k_colminmax_finish(const unsigned long long *okey, int D, double *mn, double *mx) {
    const int d = blockIdx.x * blockDim.x + threadIdx.x;
    if (d >= D) return;
    auto back = [](unsigned long long k) {
        const unsigned long long b = (k >> 63) ? (k & 0x7fffffffffffffffull) : ~k;
        return __longlong_as_double((long long)b);
    };
    const bool any = okey[d] <= okey[D + d];
    mn[d] = any ? back(okey[d]) : __longlong_as_double(0x7ff8000000000000LL); // all-NaN column: NaN, like np.nanmin
    mx[d] = any ? back(okey[D + d]) : __longlong_as_double(0x7ff8000000000000LL);
}

} // namespace ccb
