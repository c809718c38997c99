// common.cuh -- shared device helpers for the ChronoClust B200 kernels (sm_100a only).
//
// Numerics contract (SURVEY.md Appendix C): the reference's arithmetic is sequential IEEE fp64 with
// no FMA contraction.  Every parity-critical operation below goes through the round-to-nearest
// intrinsics (__dadd_rn, __dmul_rn, __ddiv_rn), which nvcc never fuses, and the library is also built
// with -fmad=false.  Sums over dimensions are accumulated in index order by a single thread.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#define CCB_MAX_D 64
#define CCB_WAVE 32 // micro-batch width of the ordered-commit kernel (one ballot word)

namespace ccb {

// Per-call input reference read from device memory (CUDA-graph launches bake kernel arguments in; what changes
// from call to call is reached through this indirection instead).
struct XRef {
    const double *X;
    int64_t ld;
};

__device__ __forceinline__ double dadd(double a, double b) { return __dadd_rn(a, b); }
__device__ __forceinline__ double dsub(double a, double b) { return __dsub_rn(a, b); }
__device__ __forceinline__ double dmul(double a, double b) { return __dmul_rn(a, b); }
__device__ __forceinline__ double ddiv(double a, double b) { return __ddiv_rn(a, b); }

// ---- mbarrier + 1-D bulk TMA (cp.async.bulk, SASS: UBLKCP) -------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t *bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_fence_init() {
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t phase) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "WAIT_%=:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
        "@p bra DONE_%=;\n\t"
        "bra WAIT_%=;\n\t"
        "DONE_%=:\n\t"
        "}" ::"r"(smem_u32(bar)),
        "r"(phase)
        : "memory");
}
// global -> shared bulk copy; bytes must be a multiple of 16, both addresses 16-byte aligned
__device__ __forceinline__ void tma_load_1d(void *dst_smem, const void *src_gmem, uint32_t bytes, uint64_t *bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                     smem_u32(dst_smem)),
                 "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}

// ---- diagnostics build only: per-round timeline of the engine (csrc/debug.h: ccb_debug_trace) -------
#ifdef CCB_DEBUG
constexpr int CCB_TRACE_SLOTS = 40, CCB_TRACE_WORDS = 64, CCB_TRACE_MAX = 1 << 14;
__device__ long long g_trace_ts[CCB_TRACE_SLOTS];               // start of every kernel of the current round (globaltimer, ns)
__device__ long long g_trace[CCB_TRACE_MAX][CCB_TRACE_WORDS];   // one record per round (k_bs_decide) / block (k_bs_commit)
__device__ int g_trace_n;
__device__ unsigned long long g_dbg_cnt[16]; // free-form event / cycle counters of experiments (ccb_debug_counters)
__device__ __forceinline__ long long globaltimer_ns() {
    long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}
#define CCB_DBG(...) __VA_ARGS__
#define CCB_TS(slot)                                                                    \
    do {                                                                                \
        if (blockIdx.x == 0 && threadIdx.x == 0) g_trace_ts[slot] = globaltimer_ns();   \
    } while (0)
#define CCB_TS_ANY(slot)                                                                \
    do {                                                                                \
        if (threadIdx.x == 0) atomicMax((unsigned long long *)&g_trace_ts[slot], (unsigned long long)globaltimer_ns()); \
    } while (0)
#else
#define CCB_DBG(...)
#define CCB_TS(slot)
#define CCB_TS_ANY(slot)
#endif

// ---- programmatic dependent launch (sm_90+) -------------------------------------------------------
// Every kernel of the engine starts with CCB_PDL(): it lets the NEXT kernel of the stream be scheduled right away
// (launch_dependents) and then waits until the kernel BEFORE it has completed and flushed its writes (wait).  Launched with
// cudaLaunchAttributeProgrammaticStreamSerialization the launch latency of a kernel would hide behind its predecessor; the
// host no longer sets that attribute (measured neutral, DESIGN.md §6), so both instructions are no-ops.  They stay because
// removing them changes the kernels' code.  Nothing but launch constants may be read before CCB_PDL().
#define CCB_PDL()                                                      \
    do {                                                               \
        asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); \
        asm volatile("griddepcontrol.wait;" ::: "memory");             \
    } while (0)

// ---- small utilities ------------------------------------------------------------------------------
__device__ __forceinline__ int popc64(uint64_t m) { return __popcll(m); }

// lexicographic (dist, index) "better" test used by every argmin: strict < on the distance, ties go to
// the smaller list position -- identical to the reference's first-strictly-smaller-wins scan
// (hddstream.py:326-328, 373-375).  An index < 0 means "no candidate".
__device__ __forceinline__ bool better(double d, int i, double bd, int bi) {
    return i >= 0 && (bi < 0 || d < bd || (d == bd && i < bi));
}

__device__ __forceinline__ void warp_argmin(double &d, int &i) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        double od = __shfl_xor_sync(0xffffffffu, d, o);
        int oi = __shfl_xor_sync(0xffffffffu, i, o);
        if (better(od, oi, d, i)) {
            d = od;
            i = oi;
        }
    }
}

} // namespace ccb
