// stats.cuh -- per-group cell counts, means, exact medians and linear quantiles of device-resident rows (sm_100a only).
//
// Pipeline (host side: group_stats_run in api.cu):
//   1. k_st_count           cells per group (shared-memory histogram for small G, warp-aggregated global atomics otherwise)
//   2. k_st_derive/k_st_scan group offsets, slices of at most ST_SLICE cells per group, the "large" groups (more than one
//                            slice) and their slices -- four exclusive scans in one launch
//   3. k_st_sort_hist/scatter stable LSD counting sort of the rows by group (8-bit digits): a deterministic permutation, so
//                            every later sum runs in the same order on every call
//   4. k_st_gather           the rows in group order, widened to double (and transformed per column) -> column-major order-preserving
//                            uint64 keys; per (slice, marker) partial sums and NaN counts, each summed in row order
//   5. k_st_small            groups of <= ST_SLICE cells: one CTA each, bitonic sort of each marker in shared memory
//      k_st_rsel_*           larger groups: radix select (8 passes x 8 bits) of every needed rank, the histograms of every
//                            slice of a group merged with integer atomics, so one big group is spread over all SMs
//   6. st_finish             numpy's median ((a + b) / 2), quantile (_lerp) and mean, with the NaN / empty-group rules
// Every reduction is either integer or in a fixed order: two calls give bit-identical results.
#pragma once
#include "common.cuh"
#include "asinh.h"

namespace ccb {

constexpr int ST_SLICE = 4096;  // cells of one group handled by one CTA (gather, small-group sort, radix histograms)
constexpr int ST_TILE = 4096;   // rows per CTA of the counting sort
constexpr int ST_THREADS = 256;
constexpr int ST_CHUNK = 64;    // rows staged in shared memory at a time by k_st_gather
constexpr uint64_t ST_SIGN = 0x8000000000000000ull;

// order-preserving map of a double onto uint64 (-0 sorts before +0; NaNs never reach a result)
__device__ __forceinline__ uint64_t st_key(double v) {
    const uint64_t u = (uint64_t)__double_as_longlong(v);
    return (u & ST_SIGN) ? ~u : (u | ST_SIGN);
}
__device__ __forceinline__ double st_val(uint64_t k) {
    return __longlong_as_double((long long)((k & ST_SIGN) ? (k ^ ST_SIGN) : ~k));
}

// one warp-aggregated shared/global atomic per distinct bin of the warp (bin < 0: no contribution); all lanes must call it
__device__ __forceinline__ void st_agg_add(unsigned *h, int bin) {
    const unsigned peers = __match_any_sync(0xffffffffu, bin);
    if (bin >= 0 && (int)(threadIdx.x & 31) == __ffs(peers) - 1) atomicAdd(h + bin, (unsigned)__popc(peers));
}

// Ranks a group of n cells needs: k = 0 / 1 the two middle order statistics of np.median, k = 2 + 2j / 3 + 2j the floor /
// floor + 1 neighbours of quantile j as numpy's _get_indexes picks them (both the last one when (n - 1) q >= n - 1).
__device__ __forceinline__ int64_t st_rank(int64_t n, int k, const double *q) {
    if (k == 0) return (n - 1) / 2;
    if (k == 1) return n / 2;
    const double v = dmul((double)(n - 1), q[(k - 2) >> 1]);
    if (v >= (double)(n - 1)) return n - 1;
    const int64_t lo = (int64_t)floor(v);
    return (k & 1) ? lo + 1 : lo;
}

// Outputs of one (group, marker) from its selected order statistics key(k) (k < 2 + 2 nq).
template <typename KeyAt>
__device__ __forceinline__ void st_finish(int64_t n, int64_t nan, double sum, KeyAt key, int nq, const double *q, size_t o,
                                          size_t qstride, double *mean, double *median, double *quant) {
    const double NaN = __longlong_as_double(0x7ff8000000000000ll);
    if (n == 0 || nan > 0) {
        mean[o] = median[o] = NaN;
        for (int j = 0; j < nq; ++j) quant[j * qstride + o] = NaN;
        return;
    }
    mean[o] = ddiv(sum, (double)n);
    const double a = st_val(key(0)), b = st_val(key(1));
    median[o] = (n & 1) ? a : ddiv(dadd(a, b), 2.0); // np.mean of the middle one / two
    for (int j = 0; j < nq; ++j) {
        const double v = dmul((double)(n - 1), q[j]);
        // numpy: gamma = v - previous index, the previous index being -1 when v >= n - 1
        const double g = v >= (double)(n - 1) ? dsub(v, -1.0) : dsub(v, floor(v));
        const double lo = st_val(key(2 + 2 * j)), hi = st_val(key(3 + 2 * j));
        const double diff = dsub(hi, lo);
        quant[j * qstride + o] = g >= 0.5 ? dsub(hi, dmul(diff, dsub(1.0, g))) : dadd(lo, dmul(diff, g));
    }
}

// ---- 1. cells per group -----------------------------------------------------------------------------------------------
// smem != 0: G <= ST_THREADS * 16 bins in shared memory, flushed once per CTA
__global__ void __launch_bounds__(ST_THREADS) k_st_count(const int32_t *group, int64_t N, int G, int smem, unsigned *cnt) {
    extern __shared__ unsigned st_h[];
    if (smem) {
        for (int i = threadIdx.x; i < G; i += blockDim.x) st_h[i] = 0;
        __syncthreads();
    }
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t base = (int64_t)blockIdx.x * blockDim.x; base < N; base += stride) {
        const int64_t r = base + threadIdx.x;
        int g = r < N ? group[r] : -1;
        if (g >= G) g = -1;
        st_agg_add(smem ? st_h : cnt, g);
    }
    if (smem) {
        __syncthreads();
        for (int i = threadIdx.x; i < G; i += blockDim.x)
            if (st_h[i]) atomicAdd(cnt + i, st_h[i]);
    }
}

// ---- 2. per-group derived counts and their scans ------------------------------------------------------------------------
// a[0] = cells, a[1] = slices, a[2] = 1 if the group takes the radix-select path, a[3] = its slices if so ([4][G])
__global__ void k_st_derive(const unsigned *cnt, int G, int32_t *a) {
    for (int g = blockIdx.x * blockDim.x + threadIdx.x; g < G; g += gridDim.x * blockDim.x) {
        const int n = (int)cnt[g];
        const int ns = (n + ST_SLICE - 1) / ST_SLICE;
        const int large = n > ST_SLICE;
        a[g] = n;
        a[G + g] = ns;
        a[2 * G + g] = large;
        a[3 * G + g] = large ? ns : 0;
    }
}

// Exclusive scan of n int32 per CTA: CTA b scans in + b * in_stride into out + b * (n + 1) (out[n] = total, also tot[b]).
// One CTA walks the whole array: the arrays scanned here have G or 256 x tiles entries.
__global__ void __launch_bounds__(1024) k_st_scan(const int32_t *in, int64_t in_stride, int32_t *out, int n, int32_t *tot) {
    __shared__ int32_t ws[32];
    __shared__ int32_t carry_s;
    in += blockIdx.x * in_stride;
    out += (int64_t)blockIdx.x * (n + 1);
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    int32_t carry = 0;
    for (int base = 0; base < n; base += 1024) {
        const int i = base + threadIdx.x;
        const int32_t v = i < n ? in[i] : 0;
        int32_t x = v;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int32_t y = __shfl_up_sync(0xffffffffu, x, o);
            if (lane >= o) x += y;
        }
        if (lane == 31) ws[w] = x;
        __syncthreads();
        if (w == 0) {
            int32_t s = ws[lane];
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const int32_t y = __shfl_up_sync(0xffffffffu, s, o);
                if (lane >= o) s += y;
            }
            ws[lane] = s; // inclusive over warps
        }
        __syncthreads();
        const int32_t incl = x + (w ? ws[w - 1] : 0);
        if (i < n) out[i] = carry + incl - v;
        if (threadIdx.x == 1023) carry_s = carry + incl;
        __syncthreads();
        carry = carry_s;
    }
    if (threadIdx.x == 0) {
        out[n] = carry;
        tot[blockIdx.x] = carry;
    }
}

// slice -> group; large group index -> group; large slice index -> (slice, large group index)  (sc: the scans of
// k_st_derive's arrays)
__global__ void k_st_slices(const int32_t *sc, int G, int32_t *slice_group, int32_t *large_group, int32_t *large_slice,
                            int32_t *large_slice_l) {
    const int32_t *soff = sc + (G + 1), *loff = sc + 2 * (G + 1), *lsoff = sc + 3 * (G + 1);
    for (int g = blockIdx.x * blockDim.x + threadIdx.x; g < G; g += gridDim.x * blockDim.x) {
        const int s0 = soff[g], ns = soff[g + 1] - s0;
        for (int j = 0; j < ns; ++j) slice_group[s0 + j] = g;
        if (loff[g + 1] > loff[g]) {
            large_group[loff[g]] = g;
            for (int j = 0; j < ns; ++j) {
                large_slice[lsoff[g] + j] = s0 + j;
                large_slice_l[lsoff[g] + j] = loff[g];
            }
        }
    }
}

// ---- 3. stable LSD counting sort of the rows by group -------------------------------------------------------------------
// FIRST: the keys are the caller's groups (out-of-range rows are dropped) and the values the row indices
template <bool FIRST>
__global__ void __launch_bounds__(ST_THREADS) k_st_sort_hist(const int32_t *key, int64_t n, int G, int shift, int32_t *th,
                                                             int ntiles) {
    __shared__ unsigned h[256];
    h[threadIdx.x] = 0;
    __syncthreads();
    const int64_t t0 = (int64_t)blockIdx.x * ST_TILE, t1 = min(n, t0 + ST_TILE);
    for (int64_t base = t0; base < t1; base += ST_THREADS) {
        const int64_t i = base + threadIdx.x;
        int d = -1;
        if (i < t1) {
            const int k = key[i];
            if (!FIRST || (k >= 0 && k < G)) d = (k >> shift) & 255;
        }
        st_agg_add(h, d);
    }
    __syncthreads();
    th[(int64_t)threadIdx.x * ntiles + blockIdx.x] = (int32_t)h[threadIdx.x];
}

// Scatter of one tile in rounds of ST_THREADS rows: a row's place = the scanned (digit, tile) offset + the rows of its
// digit in earlier rounds + those of earlier warps in this round + those of earlier lanes in its warp.
template <bool FIRST>
__global__ void __launch_bounds__(ST_THREADS) k_st_sort_scatter(const int32_t *key, const int32_t *val, int64_t n, int G,
                                                                int shift, const int32_t *toff, int ntiles, int32_t *key_out,
                                                                int32_t *val_out) {
    constexpr int NW = ST_THREADS / 32;
    __shared__ int32_t base[256];
    __shared__ int32_t wc[NW][256];
    const int t = threadIdx.x, lane = t & 31, w = t >> 5;
    base[t] = toff[(int64_t)t * ntiles + blockIdx.x];
    for (int j = 0; j < NW; ++j) wc[j][t] = 0;
    __syncthreads();
    const int64_t t0 = (int64_t)blockIdx.x * ST_TILE, t1 = min(n, t0 + ST_TILE);
    for (int64_t rb = t0; rb < t1; rb += ST_THREADS) {
        const int64_t i = rb + t;
        int k = -1, d = -1;
        if (i < t1) {
            k = key[i];
            if (!FIRST || (k >= 0 && k < G)) d = (k >> shift) & 255;
        }
        const unsigned peers = __match_any_sync(0xffffffffu, d);
        const int rank = __popc(peers & ((1u << lane) - 1));
        if (d >= 0 && rank == 0) wc[w][d] = __popc(peers);
        __syncthreads();
        int32_t acc = 0;
        for (int j = 0; j < NW; ++j) {
            const int32_t c = wc[j][t];
            wc[j][t] = acc;
            acc += c;
        }
        __syncthreads();
        if (d >= 0) {
            const int32_t pos = base[d] + wc[w][d] + rank;
            key_out[pos] = k;
            val_out[pos] = FIRST ? (int32_t)i : val[i];
        }
        __syncthreads();
        base[t] += acc;
        for (int j = 0; j < NW; ++j) wc[j][t] = 0;
        __syncthreads();
    }
}

// ---- 4. gather ---------------------------------------------------------------------------------------------------------
struct StGeom {
    const unsigned *cnt;       // [G]
    const int32_t *goff;       // [G + 1] first sorted position of each group
    const int32_t *soff;       // [G + 1] first slice of each group
    const int32_t *slice_group;
    const int32_t *perm;       // [Nv] row of every sorted position
    int64_t Nv;                // cells in some group (the column stride of keys)
    int D;
};

__device__ __forceinline__ void st_slice_range(const StGeom &g, int s, int &grp, int64_t &start, int &len) {
    grp = g.slice_group[s];
    const int j = s - g.soff[grp];
    start = (int64_t)g.goff[grp] + (int64_t)j * ST_SLICE;
    len = min(ST_SLICE, (int)g.cnt[grp] - j * ST_SLICE);
}

// Per-column transform of the values k_st_gather summarises.  A column m with bit m of `mask` set holds min-max scaled
// values, brought back by (x - shift[m]) / scale[m] (sklearn's inverse_transform); with `fwd` the rows hold the raw values
// and the forward transform x * scale[m] + shift[m] comes first (what the engine read after a column-subset ingest).
// Every other column is summarised as it is, widened to double.
struct StXf {
    const double *scale, *shift; // [CCB_MAX_D], indexed by column
    uint64_t mask;
    int fwd;
};

// One CTA per slice: rows staged ST_CHUNK at a time in shared memory (coalesced row reads, coalesced column writes).
// Thread m < D sums column m over the chunk in row order and adds the chunk to the slice's sum: a fixed order.
// k_st_gather_tx (the rows hold raw values of an ingest with arcsinh cofactors): a column m with cof[m] != 0 (device
// [CCB_MAX_D], indexed by column) is transformed to ccb_asinh(x / cof[m]) first, as k_stage_rows_tx transformed it for
// the engine.  (Two kernels over one body, as k_stage_rows / k_stage_rows_tx.)
template <typename T, bool TX>
__device__ __forceinline__ void st_gather_body(const StGeom &g, const T *X, int64_t ld, const StXf &xf, const double *cof,
                                               uint64_t *keys, double *psum, int32_t *pnan) {
    extern __shared__ double st_tile[]; // [ST_CHUNK][D + 1]
    const int D = g.D, P = D + 1, t = threadIdx.x;
    int grp, len;
    int64_t start;
    st_slice_range(g, blockIdx.x, grp, start, len);
    double sum = 0.0;
    int32_t nan = 0;
    for (int c0 = 0; c0 < len; c0 += ST_CHUNK) {
        const int rows = min(ST_CHUNK, len - c0);
        for (int e = t; e < rows * D; e += ST_THREADS) {
            const int r = e / D, m = e - r * D;
            double v = (double)X[(int64_t)g.perm[start + c0 + r] * ld + m];
            if constexpr (TX) {
                const double c = cof[m];
                if (c != 0.0) v = ccb_asinh(ddiv(v, c));
            }
            if ((xf.mask >> m) & 1ull) {
                if (xf.fwd) v = dadd(dmul(v, xf.scale[m]), xf.shift[m]);
                v = ddiv(dsub(v, xf.shift[m]), xf.scale[m]);
            }
            st_tile[r * P + m] = v;
        }
        __syncthreads();
        for (int e = t; e < rows * D; e += ST_THREADS) {
            const int m = e / rows, r = e - m * rows;
            keys[(int64_t)m * g.Nv + start + c0 + r] = st_key(st_tile[r * P + m]);
        }
        if (t < D) {
            double cs = 0.0;
            for (int r = 0; r < rows; ++r) {
                const double v = st_tile[r * P + t];
                cs = dadd(cs, v);
                nan += v != v;
            }
            sum = dadd(sum, cs);
        }
        __syncthreads();
    }
    if (t < D) {
        psum[(int64_t)blockIdx.x * D + t] = sum;
        pnan[(int64_t)blockIdx.x * D + t] = nan;
    }
}

template <typename T>
__global__ void __launch_bounds__(ST_THREADS) k_st_gather(StGeom g, const T *X, int64_t ld, StXf xf, uint64_t *keys,
                                                          double *psum, int32_t *pnan) {
    st_gather_body<T, false>(g, X, ld, xf, nullptr, keys, psum, pnan);
}
template <typename T>
__global__ void __launch_bounds__(ST_THREADS) k_st_gather_tx(StGeom g, const T *X, int64_t ld, StXf xf, const double *cof,
                                                             uint64_t *keys, double *psum, int32_t *pnan) {
    st_gather_body<T, true>(g, X, ld, xf, cof, keys, psum, pnan);
}

// sum / NaN count of (group, marker) over the group's slices, in slice order
__device__ __forceinline__ void st_group_sum(const StGeom &g, const double *psum, const int32_t *pnan, int grp, int m,
                                             double &sum, int64_t &nan) {
    sum = 0.0;
    nan = 0;
    for (int s = g.soff[grp]; s < g.soff[grp + 1]; ++s) {
        sum = dadd(sum, psum[(int64_t)s * g.D + m]);
        nan += pnan[(int64_t)s * g.D + m];
    }
}

struct StOut {
    const double *q; // [nq] device
    int nq, G;
    double *mean, *median, *quant; // [G][D], [G][D], [nq][G][D]
};

// ---- 5a. groups of at most ST_SLICE cells (and empty ones): one CTA each, every marker sorted in shared memory ----------
__global__ void __launch_bounds__(ST_THREADS) k_st_small(StGeom g, const uint64_t *keys, const double *psum,
                                                         const int32_t *pnan, StOut out) {
    __shared__ uint64_t s[ST_SLICE];
    const int grp = blockIdx.x, t = threadIdx.x, D = g.D;
    const int n = (int)g.cnt[grp];
    if (n > ST_SLICE) return;
    const size_t qstride = (size_t)out.G * D;
    int P = 1;
    while (P < n) P <<= 1;
    for (int m = 0; m < D; ++m) {
        const uint64_t *col = keys + (int64_t)m * g.Nv + (n ? g.goff[grp] : 0);
        for (int i = t; i < P; i += ST_THREADS) s[i] = i < n ? col[i] : ~0ull;
        __syncthreads();
        for (int k = 2; k <= P; k <<= 1)
            for (int j = k >> 1; j > 0; j >>= 1) {
                for (int i = t; i < P; i += ST_THREADS) {
                    const int p = i ^ j;
                    if (p > i) {
                        const uint64_t a = s[i], b = s[p];
                        if ((a > b) == ((i & k) == 0)) {
                            s[i] = b;
                            s[p] = a;
                        }
                    }
                }
                __syncthreads();
            }
        if (t == 0) {
            double sum = 0.0;
            int64_t nan = 0;
            if (n) st_group_sum(g, psum, pnan, grp, m, sum, nan);
            st_finish(n, nan, sum, [&](int k) { return s[st_rank(n, k, out.q)]; }, out.nq, out.q, (size_t)grp * D + m,
                      qstride, out.mean, out.median, out.quant);
        }
        __syncthreads();
    }
}

// ---- 5b. larger groups: radix select of every needed rank ---------------------------------------------------------------
// state per (large group l, marker m, rank k), index (l * D + m) * R + k: the key prefix fixed so far, the rank left
// within the keys that share it, and the 256-bin histogram of the current digit
struct StSel {
    const int32_t *large_group; // [L]
    const int32_t *large_slice;   // [NLS] slice of every slice of a large group
    const int32_t *large_slice_l; // [NLS] the index of that group among the large ones
    uint64_t *pre;
    int64_t *rem;
    unsigned *hist; // [L][D][R][256]
    int R;
};

__global__ void k_st_rsel_init(StGeom g, StSel sel, const double *q, int64_t items) {
    for (int64_t it = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; it < items; it += (int64_t)gridDim.x * blockDim.x) {
        const int k = (int)(it % sel.R);
        const int l = (int)(it / sel.R / g.D);
        sel.pre[it] = 0;
        sel.rem[it] = st_rank((int64_t)g.cnt[sel.large_group[l]], k, q);
    }
}

// one CTA per (slice of a large group, marker); R histograms of the keys whose bits above `shift + 8` match each prefix
__global__ void __launch_bounds__(ST_THREADS) k_st_rsel_hist(StGeom g, StSel sel, const uint64_t *keys, int shift) {
    extern __shared__ unsigned st_rh[]; // [R][256], then the R prefixes
    const int R = sel.R, t = threadIdx.x, m = blockIdx.y;
    uint64_t *pre = reinterpret_cast<uint64_t *>(st_rh + R * 256);
    int grp, len;
    int64_t start;
    st_slice_range(g, sel.large_slice[blockIdx.x], grp, start, len);
    const int64_t sbase = ((int64_t)sel.large_slice_l[blockIdx.x] * g.D + m) * R;
    for (int i = t; i < R * 256; i += ST_THREADS) st_rh[i] = 0;
    for (int k = t; k < R; k += ST_THREADS) pre[k] = sel.pre[sbase + k];
    __syncthreads();
    const uint64_t *col = keys + (int64_t)m * g.Nv + start;
    for (int b = 0; b < len; b += ST_THREADS) {
        const int i = b + t;
        const uint64_t key = i < len ? col[i] : 0;
        for (int k = 0; k < R; ++k) {
            const bool match = i < len && (shift == 56 || ((key ^ pre[k]) >> (shift + 8)) == 0);
            st_agg_add(st_rh + k * 256, match ? (int)((key >> shift) & 255) : -1);
        }
    }
    __syncthreads();
    for (int i = t; i < R * 256; i += ST_THREADS)
        if (st_rh[i]) atomicAdd(sel.hist + sbase * 256 + i, st_rh[i]);
}

// fixes the digit of every (l, m, k) and clears its histogram for the next pass
__global__ void k_st_rsel_fix(StSel sel, int64_t items, int shift) {
    for (int64_t it = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; it < items; it += (int64_t)gridDim.x * blockDim.x) {
        unsigned *h = sel.hist + it * 256;
        int64_t r = sel.rem[it], below = 0;
        int d = 0;
        for (; d < 255; ++d) {
            if (below + h[d] > r) break;
            below += h[d];
        }
        for (int b = 0; b < 256; ++b) h[b] = 0;
        sel.pre[it] |= (uint64_t)d << shift;
        sel.rem[it] = r - below;
    }
}

__global__ void k_st_large_finish(StGeom g, StSel sel, const double *psum, const int32_t *pnan, StOut out, int64_t items) {
    for (int64_t it = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; it < items; it += (int64_t)gridDim.x * blockDim.x) {
        const int m = (int)(it % g.D), l = (int)(it / g.D);
        const int grp = sel.large_group[l];
        double sum;
        int64_t nan;
        st_group_sum(g, psum, pnan, grp, m, sum, nan);
        const uint64_t *pre = sel.pre + it * sel.R;
        st_finish((int64_t)g.cnt[grp], nan, sum, [&](int k) { return pre[k]; }, out.nq, out.q, (size_t)grp * g.D + m,
                  (size_t)out.G * g.D, out.mean, out.median, out.quant);
    }
}

// ---- handle: cell -> group through the pcore list -----------------------------------------------------------------------
// lut [nlut] over MC uids: the group of every pcore MC, `none` for every other uid
__global__ void k_st_lut_fill(int32_t *lut, int64_t nlut, int32_t none) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < nlut; i += (int64_t)gridDim.x * blockDim.x)
        lut[i] = none;
}
__global__ void k_st_lut_pcore(const int32_t *uid, const int32_t *group_of_pcore, int n, int64_t nlut, int32_t none,
                               int32_t *lut) {
    for (int p = blockIdx.x * blockDim.x + threadIdx.x; p < n; p += gridDim.x * blockDim.x) {
        const int32_t u = uid[p];
        if (u >= 0 && u < nlut) lut[u] = group_of_pcore[p] >= 0 ? group_of_pcore[p] : none;
    }
}
__global__ void k_st_cell_group(const int32_t *assign, int64_t N, const int32_t *lut, int64_t nlut, int32_t none,
                                int32_t *group) {
    for (int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; r < N; r += (int64_t)gridDim.x * blockDim.x) {
        const int32_t a = assign[r];
        group[r] = a >= 0 && a < nlut ? lut[a] : none;
    }
}

} // namespace ccb
