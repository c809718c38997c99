/*
 * debug.h -- diagnostics of the DEBUG build (python chronoclust_b200/build.py --debug -> libchronoclust_b200_debug.so,
 * compiled with -DCCB_DEBUG).  Not part of the product ABI: include/chronoclust_b200.h does not declare these symbols and
 * libchronoclust_b200.so does not export them.
 */
#ifndef CHRONOCLUST_B200_DEBUG_H
#define CHRONOCLUST_B200_DEBUG_H

#include "../../include/chronoclust_b200.h"

#ifdef __cplusplus
extern "C" {
#endif

/* Per pcore key of the last k_bs_chain_p launch: out[key][8] = {members, replay cycles, replay waiting for data, cycles in
 * stages with a CONTESTED cell or a ragged tail, CONTESTED cells, cycles at the head of the stages (flags), cycles at
 * their tail (proxy fence + arrive), clean full stages}.  The first call switches the counters on. */
int ccb_debug_chain(ccb_handle *h, int64_t *out, int32_t max_keys);
/* Timeline of the engine: one record of 48 int64 per refinement round (kind 0 / 1, written by k_bs_decide) and per block
 * (kind 2, k_bs_commit): control-block fields and the start time (globaltimer, ns) of every kernel of the round; layout in
 * tools/trace_rounds.py.  Returns the number of records written since the last call (at most max_records are copied) and
 * rewinds the ring. */
int64_t ccb_debug_trace(ccb_handle *h, int64_t *out, int64_t max_records);
/* 16 free-form event / cycle counters of the experiment at hand (see the CCB_DBG lines in csrc/engine.cuh). */
int ccb_debug_counters(ccb_handle *h, int64_t *out16, int32_t reset);

#ifdef __cplusplus
}
#endif
#endif
