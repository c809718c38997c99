/*
 * chronoclust_b200.h -- C ABI of the B200-native ChronoClust per-timepoint clustering hot path.
 *
 * One shared library (chronoclust_b200/libchronoclust_b200.so), plain pointers and sizes, no C++ or
 * torch types.  Every entry point returns 0 on success or a negative CCB_E* code; the message is
 * available from ccb_last_error().  No C++ exception crosses this boundary.  A handle is bound to
 * one CUDA device and one stream; the caller is single-threaded per handle; independent handles may
 * live on different devices (parameter sweeps).  There is NO CPU fallback: without a CUDA device
 * ccb_create fails with CCB_ECUDA.
 *
 * What each entry point replaces (file:line relative to the reference, ghar1821/Chronoclust):
 *
 *   ccb_create              HDDStream.__init__                      clustering/hddstream.py:30-67
 *   ccb_begin_timepoint     decay + downgrade + reset               clustering/hddstream.py:199-213,
 *                                                                    247-286, 512-549
 *   ccb_ingest[_device|_ex| the ordered per-point loop              clustering/hddstream.py:220-237,
 *              _cols|_tx]   (_add_to_pcore, _add_to_outlier,          288-343, 345-395, 397-430, 434-462
 *                            _upgrade_outlier_microcluster,          objects/microcluster.py:89-153,
 *                            _create_new_outlier_cluster)             167-197, 213-233
 *                                                                    utilities/mc_functions.py:14-62
 *   ccb_offline             HDDStream.offline_clustering            clustering/hddstream.py:464-510
 *                           + PreDeCon.run                          clustering/predecon.py:49-120,136-267
 *                                                                    objects/predecon_mc.py:50-80
 *                                                                    utilities/predeconmc_functions.py:4-62
 *                                                                    utilities/mc_functions.py:64-77
 *   ccb_export_list /       the Microcluster objects in             objects/microcluster.py:71-81
 *   ccb_import_list         HDDStream.pcore_MC / outlier_MC         (state for the Python facade, pickling)
 *   ccb_export_clusters     HDDStream.final_clusters                clustering/hddstream.py:508
 *   ccb_nearest             Microcluster.get_projected_dist_to_point objects/microcluster.py:167-181,
 *                           + the strict-< argmin of the scans       clustering/hddstream.py:311-328,371-375
 *   ccb_off_*               the row-sharded stages of PreDeCon      clustering/predecon.py:136-217
 *                           (multi-GPU offline path, config C4)
 *   ccb_cluster_stats /     (extension) per-cluster cell counts,    replaces grouping cluster_points_D{t}.csv
 *   ccb_group_stats         means, medians, quantiles of a timepoint  on the host after a run
 *   ccb_ingest_tx /         (extension) arcsinh(x / cofactor) of    replaces the caller's host pass (or
 *   ccb_arcsinh             cytometry intensities, one definition    torch.asinh) before clustering
 *                           for host and device (csrc/asinh.h)
 *
 * The derived constants (epsilon**2, upsilon*epsilon, delta**2, 2**(-lambda*dt), mu*N, omicron*N_prev,
 * round(pi)) are evaluated by the Python host with Python's own float semantics, exactly where the
 * reference evaluates them (hddstream.py:44-52, 107-126, 283), and passed in as doubles.
 */
#ifndef CHRONOCLUST_B200_H
#define CHRONOCLUST_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define CCB_OK 0
#define CCB_EINVAL (-1)  /* bad argument */
#define CCB_ECUDA (-2)   /* CUDA runtime error / no device */
#define CCB_ENOMEM (-3)  /* host or device allocation failed */
#define CCB_ESTATE (-4)  /* call sequence error */
#define CCB_ELIMIT (-5)  /* a documented limit was exceeded (D > 64, ids >= 2^31) */

#define CCB_MAX_D 64

typedef struct ccb_handle ccb_handle;

typedef struct {
    int32_t D;           /* markers per cell, 1..CCB_MAX_D */
    int32_t device;      /* CUDA device ordinal */
    double eps2;         /* epsilon ** 2                          hddstream.py:45 */
    double upsilon_eps;  /* float(upsilon) * epsilon              hddstream.py:47 */
    double upsilon_eps2; /* (upsilon * epsilon) ** 2              predecon.py:40 */
    double delta;        /*                                       hddstream.py:48 */
    double delta2;       /* delta ** 2                            hddstream.py:49 */
    double beta;         /*                                       hddstream.py:50 */
    double k;            /*                                       hddstream.py:51 */
    int32_t chunk;       /* max cells per block of the ordered engine (rounded up to a multiple of 32); 0 = default 32768 */
    int32_t bsv_bmin;    /* smallest block length; 0 = default (1024) */
    int32_t bsv_iters;   /* refinement rounds per block before the exact prefix is committed;
                            0 = default (3 with stream launches, 8 inside the CUDA graph) */
    int32_t bsv_stream;  /* 1 = plain stream launches instead of the CUDA graph with device-driven WHILE nodes (the graph
                            is also bypassed while ccb_enable_timing is on) */
    int32_t off_csr_min_m; /* offline cluster growth: number of potential microclusters from which the CSR formulation
                              (isolated microclusters in parallel, lists instead of bit rows) replaces the single-CTA
                              bit-row scan; 0 = default (2048).  Both give identical results. */
    int32_t reserved0;   /* must be 0 */
} ccb_params;

/* Counters since ccb_create (monotonic); all int64.  None of the engine knobs above ever changes a result; the
 * bsv_* counters describe how the ordered engine got there. */
typedef struct {
    int64_t points;          /* cells ingested */
    int64_t nearest_pairs;   /* (cell x outlier MC) distances evaluated by kernel 1 */
    int64_t upgrades, created, downgraded, deleted;
    int64_t kernel_launches; /* every kernel this library launched */
    int64_t borderline_pairs; /* offline pairs resolved on the host through dnrm2 */
    /* block-speculative engine */
    int64_t bsv_blocks;        /* blocks committed */
    int64_t bsv_rounds;        /* speculate / verify rounds executed */
    int64_t bsv_mismatches;    /* rounds whose verification found a cell decided differently than speculated */
    int64_t bsv_cuts_unknown;  /* blocks cut because every listed snapshot candidate of a cell was stale */
    int64_t bsv_cuts_rounds;   /* blocks cut because the enqueued rounds ran out */
    int64_t bsv_cuts_capacity; /* blocks cut because the outlier-stage list of the block was full */
    int64_t bsv_late_topk;     /* cells whose top-K list had to be fetched in a refinement round */
    int64_t bsv_outlier_stage_cells; /* cells given a top-K list up front (not SAFE) */
    int64_t bsv_replayed_cells;      /* cells replayed by the chain kernels, summed over rounds */
    int64_t bsv_light_rounds;        /* refinement rounds that re-ran the outlier side only (pcore side unchanged) */
    int64_t bsv_serial_cells;        /* sum over the pcore replays of the longest chain's member count: x one dependent-add
                                        latency = the serial floor of kernel 2 (what the reference's ordering forces) */
    int64_t bsv_pdl;                 /* always 0: the engine no longer uses programmatic dependent launch (field kept for the ABI) */
} ccb_stats;

int ccb_create(const ccb_params *params, ccb_handle **out);
void ccb_destroy(ccb_handle *h);
/* h == NULL returns the message of the last failed ccb_create / stateless call of this thread. */
const char *ccb_last_error(const ccb_handle *h);
/* cudaStream_t the handle launches on (for CUDA-event timing by the caller). */
void *ccb_stream(ccb_handle *h);
int ccb_get_stats(const ccb_handle *h, ccb_stats *out);
/* Forgets every microcluster and both id counters (a new run on the same device / stream). */
int ccb_reset(ccb_handle *h);

/* Optional GPU timing per kernel category, taken with CUDA events on the handle's stream (this is
 * what bench.py reads for the live roofline).  ms / launches: arrays of CCB_NCAT. */
#define CCB_CAT_PCORE 0   /* kernel 2   ordered replay of the pcore keys (k_bs_chain_p) */
#define CCB_CAT_NEAREST 1 /* kernel 1   k_nearest (+ merge) on the cells that may reach the outlier stage */
#define CCB_CAT_RESOLVE 2 /* kernel 2   exact verification (k_bs_verify_p/o) */
#define CCB_CAT_MAINT 3   /* kernel 3   k_maint_plan + k_maint_gather */
#define CCB_CAT_OFFLINE 4 /* kernel 4   offline pipeline (device part) */
#define CCB_CAT_MISC 5    /* small helpers */
#define CCB_CAT_COPY 6    /* host<->device copies of ccb_ingest */
#define CCB_CAT_SPEC 7    /* kernel 2   speculation from the snapshot (k_bs_begin/spec/need/spec_o) */
#define CCB_CAT_LISTS 8   /* kernel 2   candidate lists + addend records (k_bs_tilecnt/pscan/pscatter) */
#define CCB_CAT_CHAIN_O 9 /* kernel 2   ordered replay of the outlier-side keys (k_bs_chain_o) */
#define CCB_CAT_OLIST 10  /* kernel 2   outlier-side member lists (k_bs_olist) */
#define CCB_CAT_DERIVE 11 /* kernel 2   centroid / preference mask / radius of every version (k_bs_derive) */
#define CCB_CAT_DECIDE 12 /* kernel 2   exact-prefix decision / refinement (k_bs_decide) */
#define CCB_CAT_COMMIT 13 /* kernel 2   write-back of the exact prefix (k_bs_commit) */
#define CCB_NCAT 16
int ccb_enable_timing(ccb_handle *h, int32_t on);
int ccb_get_timing(ccb_handle *h, double ms[CCB_NCAT], int64_t launches[CCB_NCAT], int32_t reset);

/* The BLAS dnrm2 the reference reaches through numba (predeconmc_functions.py:16-17):
 * double fn(int *n, double *x, int *incx).  Used only for offline pairs whose squared distance is
 * within a guard band of (upsilon*epsilon)^2; NULL restores the built-in restatement. */
int ccb_set_dnrm2(ccb_handle *h, void *fn);

/* Timepoint start.  decay != 0 iff t != last_data_timestamp (hddstream.py:199); decay_factor is
 * 2 ** (-lambda * interval).  mu = float(config mu) * N, omicron = config omicron * N_prev,
 * pi = D if config pi <= 0 else round(pi)  (hddstream.py:107-126). */
int ccb_begin_timepoint(ccb_handle *h, double mu, double omicron, int64_t pi, int32_t decay, double decay_factor);

/* The ordered loop over N cells.  X: host, row-major, leading dimension ld (doubles).
 * assign_uid[r] (host, N) receives the unique creation id (= prev_outlier_id, microcluster.py:83-84)
 * of the MC that absorbed row r; stage[r] (host, N, may be NULL): 0 pcore absorb, 1 outlier absorb,
 * 2 outlier absorb + upgrade, 3 new outlier MC. */
int ccb_ingest(ccb_handle *h, const double *X, int64_t N, int64_t ld, int32_t *assign_uid, uint8_t *stage);
/* The same for RAW rows: every row is min-max scaled on the device first, x * scale[d] + min_[d] as two roundings --
 * exactly sklearn's MinMaxScaler.transform with its fitted scale_ / min_ (scaling/scaler.py:43-47) -- so the host never
 * makes the scaled pass over the data (SURVEY 8f-3).  scale, min_: host arrays [D]. */
int ccb_ingest_scaled(ccb_handle *h, const double *X_raw, int64_t N, int64_t ld, const double *scale, const double *min_,
                      int32_t *assign_uid, uint8_t *stage);
/* Same with X, assign_uid and stage already resident on the handle's device (stage may be NULL). */
int ccb_ingest_device(ccb_handle *h, const double *X_dev, int64_t N, int64_t ld, int32_t *assign_uid_dev,
                      uint8_t *stage_dev);
/* Element types of the rows handed to ccb_ingest_ex / ccb_colminmax_ex. */
#define CCB_DTYPE_F64 0
#define CCB_DTYPE_F32 1
/* The ordered loop over N cells (clustering/hddstream.py:220-237, as ccb_ingest) for rows of either element type.
 * X: row-major, leading dimension ld in ELEMENTS of dtype.  on_device != 0: X, assign_uid and stage are device pointers
 * on the handle's device (as ccb_ingest_device), else host pointers (as ccb_ingest).  scale, min_: host [D], both NULL or
 * both set (the transform of ccb_ingest_scaled, scaling/scaler.py:43-47).  Every element is widened to double first
 * (exact): results are those of ccb_ingest[_scaled] on the widened rows, bit for bit.  X is never written.  Device-resident
 * float64 rows without a scaler go to the engine as they are; any other device input is widened / scaled by one launch
 * into a handle-owned buffer first; float32 host rows travel as float32 and are widened on the device.
 * An unknown dtype, only one of scale / min_, or ld < D: CCB_EINVAL. */
int ccb_ingest_ex(ccb_handle *h, const void *X, int32_t dtype, int32_t on_device, int64_t N, int64_t ld,
                  const double *scale, const double *min_, int32_t *assign_uid, uint8_t *stage);
/* ccb_ingest_ex on a subset of the columns of wider rows (extension): X holds rows of W >= D columns (leading dimension
 * ld >= W) and the engine clusters the columns cols [D] (host, distinct, each in [0, W)) in that order.  Results are those
 * of ccb_ingest_ex on the gathered rows X[:, cols], bit for bit; scale / min_ have D entries and belong to the clustering
 * columns.  X is never written.  Host rows travel W wide through the segmented copy into a handle-owned staging buffer
 * and are gathered, widened and scaled behind each segment's copy; device rows take one staging launch.
 * Afterwards ccb_cluster_stats reports all W columns: a clustering column is reported as the engine read it brought back
 * to the input scale (under a scaler: MinMaxScaler.inverse_transform(transform(x))), every other column as the raw value
 * widened to double.  CCB_EINVAL: W outside [D, 64], ld < W, a null cols, an entry of cols outside [0, W), a repeated
 * entry, or anything ccb_ingest_ex rejects. */
int ccb_ingest_cols(ccb_handle *h, const void *X, int32_t dtype, int32_t on_device, int64_t N, int64_t ld, int32_t W,
                    const int32_t *cols, const double *scale, const double *min_, int32_t *assign_uid, uint8_t *stage);
/* ccb_ingest_cols with the arcsinh transform of cytometry intensities (extension).  cols: as ccb_ingest_cols, or NULL for
 * the identity (then W must be D).  cofactor: host [W] by SOURCE column, or NULL for none; a column with cofactor c != 0
 * is read as asinh((double)x / c) (csrc/asinh.h's ccb_asinh: widened first, one IEEE division, then a restatement of fdlibm's
 * asinh that gives the same bits on host and device), a column with c == 0 stays linear.  The order is: widen, gather,
 * asinh, scaler.  Results are those of ccb_ingest_ex on ccbio_arcsinh_host's output (gathered), bit for bit.  X is never
 * written: host float64 rows are transformed in their device copy, every other input by the staging launch.
 * Afterwards ccb_cluster_stats reports the transformed columns in transformed space (clustering columns under a scaler
 * brought back through it as after the other ingests).  CCB_EINVAL: a cofactor that is NaN, negative or infinite, W != D
 * without cols, or anything ccb_ingest_cols rejects; with cols and cofactor NULL this is ccb_ingest_cols, without both
 * ccb_ingest_ex. */
int ccb_ingest_tx(ccb_handle *h, const void *X, int32_t dtype, int32_t on_device, int64_t N, int64_t ld, int32_t W,
                  const int32_t *cols, const double *cofactor, const double *scale, const double *min_, int32_t *assign_uid,
                  uint8_t *stage);

/* Offline phase over the current pcore list; returns the number of clusters. */
int ccb_offline(ccb_handle *h, int64_t *n_clusters);

/* out[0] = pcore MCs, out[1] = outlier MCs, out[2] = pcore_MC_last_id, out[3] = outlier_MC_last_id */
int ccb_counts(ccb_handle *h, int64_t out[4]);
/* which: 0 pcore, 1 outlier.  Arrays in list order: ids/uids [n], w [n], cf1/cf2/cen/pref [n][D]. */
int ccb_export_list(ccb_handle *h, int32_t which, int64_t *ids, int64_t *uids, double *w, double *cf1, double *cf2,
                    double *cen, double *pref);
/* Replaces a list (restore / white-box tests).  pref entries equal to k become "preferred". */
int ccb_import_list(ccb_handle *h, int32_t which, int64_t n, const int64_t *ids, const int64_t *uids,
                    const double *w, const double *cf1, const double *cf2, const double *cen, const double *pref);
int ccb_set_counters(ccb_handle *h, int64_t pcore_last_id, int64_t outlier_last_id);

/* Result of the last ccb_offline.  out[0] = clusters, out[1] = total members, out[2] = pcore MCs seen. */
int ccb_cluster_sizes(ccb_handle *h, int64_t out[3]);
/* off [nc+1], members [out[1]] = pcore ids in claim order (insert into a Python set in this order),
 * w [nc], cf1/cf2/cen/pref [nc][D]; label [out[2]] = cluster index of every pcore MC in list order, -1 none. */
int ccb_export_clusters(ccb_handle *h, int64_t *off, int64_t *members, double *w, double *cf1, double *cf2,
                        double *cen, double *pref, int32_t *label);
/* White-box: core flags [M], neighbour / weighted-neighbour matrices [M*M] bytes, subspace weights [M][D]. */
int ccb_export_offline(ccb_handle *h, uint8_t *core, uint8_t *nbr, uint8_t *wnbr, double *subw);

/* Per-cluster statistics of the cells of the LAST ingest call (extension): the cells are grouped through
 * group_of_pcore [n_pcore] (host, pcore list order as ccb_export_list(0) returns it, -1 = in no group, else < G): a cell
 * whose assigned MC sits in the pcore list at position p belongs to group group_of_pcore[p]; every other cell (absorbed by
 * an outlier MC, or by a pcore MC in no group) to the extra last row G.  Outputs as ccb_group_stats with G + 1 rows.
 * The values are the rows the engine read widened to double; after a scaled ingest they are (x - min_) / scale_ (two
 * roundings: sklearn's MinMaxScaler.inverse_transform), i.e. the values app.run writes to cluster_points_D{t}.csv.
 * The rows and assignments are read where the ingest left them: the handle's own buffers, or, for device input
 * (ccb_ingest_ex with on_device, ccb_ingest_device), the CALLER's device rows and assignment buffer, which must still hold
 * what they held at the ingest.  Reads only: nothing later computed by the handle changes.
 * After ccb_ingest_cols the outputs cover all W columns of the rows ([G + 1][W], quantiles [nq][G + 1][W]); otherwise
 * they have D columns.
 * CCB_ESTATE unless an ingest happened since the last ccb_begin_timepoint / ccb_reset / ccb_import_list; CCB_EINVAL if
 * n_pcore != the pcore count, G < 0, a group_of_pcore entry >= G, or a q outside [0, 1].  Synchronises the handle's stream. */
int ccb_cluster_stats(ccb_handle *h, const int32_t *group_of_pcore, int64_t n_pcore, int32_t G, int32_t nq, const double *q,
                      int64_t *count, double *mean, double *median, double *quant);

/* ---------------------------------------------------------------------------------------------
 * Stateless device-pointer entry points (all pointers are device memory on `device`; stream is a
 * cudaStream_t or NULL).  These are what bench.py times for the roofline and what the multi-GPU
 * offline path calls between its NCCL all-gathers.
 * ------------------------------------------------------------------------------------------- */

/* Kernel 1: for every row of X [N][ld] the nearest of M microclusters under the preference-weighted
 * projected distance sum_d ((x_d - c_d)^2) / pref_d, strict-< first-wins.  cen [M][D]; prefmask [M]
 * (bit d set <=> pref_d == k, else 1.0).  slot [N] (-1 if M == 0), dist [N]. */
int ccb_nearest(int32_t device, void *stream, const double *X, int64_t N, int64_t ld, int32_t D, const double *cen,
                const uint64_t *prefmask, int64_t M, double k, int32_t *slot, double *dist);

/* Scaler (SURVEY 8f-3; scaling/scaler.py:11-53 -> sklearn MinMaxScaler).  ccb_colminmax: column-wise minimum / maximum of
 * a device-resident X [N][ld] ignoring NaN (np.nanmin / np.nanmax of partial_fit); min_dev / max_dev [D] on the device.
 * The transform itself is part of ccb_ingest_scaled (below the handle API). */
int ccb_colminmax(int32_t device, void *stream, const double *X_dev, int64_t N, int64_t ld, int32_t D, double *min_dev,
                  double *max_dev);
/* The same for rows of either element type (CCB_DTYPE_*; ld in elements of dtype): the results are np.nanmin / np.nanmax
 * of the rows widened to double.  An unknown dtype: CCB_EINVAL. */
int ccb_colminmax_ex(int32_t device, void *stream, const void *X_dev, int32_t dtype, int64_t N, int64_t ld, int32_t D,
                     double *min_dev, double *max_dev);
/* The arcsinh transform of ccb_ingest_tx on its own (extension): out_dev [N][D] (float64, contiguous) = X_dev [N][ld]
 * (CCB_DTYPE_*, ld in elements) widened to double, every column d with cofactor[d] != 0 as asinh(x / cofactor[d]) (ccb_asinh).
 * cofactor: host [D].  The values the engine clusters, for plots or for fitting the scaler with ccb_colminmax_ex; the
 * host library's ccbio_arcsinh_host (chronoclust_b200/csrc/hostio.c) gives the same bits.  Asynchronous on `stream`.
 * CCB_EINVAL: an unknown dtype, D outside [1, 64], ld < D, N < 0, null pointers, or a cofactor that is NaN, negative or
 * infinite. */
int ccb_arcsinh(int32_t device, void *stream, const void *X_dev, int32_t dtype, int64_t N, int64_t ld, int32_t D,
                const double *cofactor, double *out_dev);

/* Association scan (SURVEY 8f-1; replaces the inner loops of TrackByHistoricalAssociation.track_cluster_history,
 * tracking/cluster_tracker.py:127-144): for every CURRENT pcore microcluster q the index of the previous-timepoint
 * pcore microcluster j, in scan order, that minimises q.get_projected_dist_to_point(prev_cen[j]) =
 * sum_d ((prev_cen[j][d] - cur_cen[q][d])^2) / pref_q[d] (microcluster.py:167-181), first strictly smaller wins.
 * cur_cen [Q][D], cur_prefmask [Q] (bit d set <=> pref_q[d] == k), prev_cen [P][D]; best [Q] (-1 if P == 0), dist [Q]. */
int ccb_assoc_nearest(int32_t device, void *stream, const double *cur_cen, const uint64_t *cur_prefmask, int64_t Q,
                      const double *prev_cen, int64_t P, int32_t D, double k, int32_t *best, double *dist);
/* The same scan, also returning the runner-up distance dist2 [Q] (+inf if P < 2).  Used for the gating label of every
 * cluster (SURVEY 8f-4; replaces the loop of find_closest_gating, app.py:497-512, over Cluster.get_projected_dist_to_point,
 * objects/cluster.py:94-104): that reference expression squares with Python's float `** 2` (libm pow), which may differ
 * from the IEEE product in the last bit, so the caller accepts the device's argmin only when dist2 - dist clears a guard
 * band and re-evaluates the few near-ties with the reference expression itself. */
int ccb_assoc_nearest2(int32_t device, void *stream, const double *cur_cen, const uint64_t *cur_prefmask, int64_t Q,
                       const double *prev_cen, int64_t P, int32_t D, double k, int32_t *best, double *dist, double *dist2);

/* Per-group statistics of device rows (extension).  X [N][ld] (CCB_DTYPE_*, ld in elements) on `device`, group [N] int32
 * on the device: -1 (or any value outside [0, G)) = skip the row, else its group.  q: host [nq], each in [0, 1].
 * Outputs (host): count [G]; mean / median [G][D]; quant [nq][G][D] (may be NULL when nq == 0).
 *   median = np.median of the group's values, bit for bit ((a + b) / 2 of the middle two for an even count);
 *   quant  = np.quantile(values, q, method="linear"), bit for bit (numpy's index rule and _lerp);
 *   mean   = np.mean up to rounding, summed in a fixed order: identical from call to call.
 * A group without cells: count 0, NaN elsewhere; a NaN among a marker's values: NaN mean / median / quantiles there.
 * CCB_EINVAL: bad shapes, G < 1, an unknown dtype, a q outside [0, 1] (or NaN); CCB_ELIMIT: N >= 2^31 or nq > 64.
 * Scratch from the stream-ordered pool, about N * (8 D + 24) bytes.  Synchronises `stream`. */
int ccb_group_stats(int32_t device, void *stream, const void *X, int32_t dtype, int64_t N, int64_t ld, int32_t D,
                    const int32_t *group, int32_t G, int32_t nq, const double *q, int64_t *count, double *mean, double *median,
                    double *quant);

/* FP64 pipe microbenchmark for the roofline denominators: mode 0 = DFMA stream (2 flop/instr), mode 1 =
 * separate DMUL + DADD (1 flop/instr, the only form the parity contract allows).  Launches `blocks` CTAs of
 * 256 threads x 8 independent chains x iters; *flops_out = flops executed.  Time it with CUDA events. */
int ccb_fp64_peak(int32_t device, void *stream, int32_t mode, int32_t iters, int32_t blocks, double *sink,
                  double *flops_out);

/* Offline stage 1 for rows [r0, r1) of M pcore MCs: neighbourhood bit rows nbr [(r1-r0)][words]
 * (words = ceil(M/32), uint32) and neighbour counts cnt [(r1-r0)] of the test dnrm2(c_q - c_p) <= E.  The device decides
 * every pair whose squared distance is outside a guard band around E2 = E^2; the pairs inside it are settled on the host
 * with dnrm2 (as for ccb_set_dnrm2; NULL = the built-in restatement).  *n_border (host) = the number of such pairs.
 * Synchronises the stream. */
int ccb_off_neighbours(int32_t device, void *stream, const double *cen, int64_t M, int32_t D, int64_t r0, int64_t r1,
                       double E, double E2, void *dnrm2, uint32_t *nbr, int32_t *cnt, int64_t *n_border);
/* Offline stage 2: subspace preference masks submask [(r1-r0)] from the neighbour rows (delta, not delta^2). */
int ccb_off_subspace(int32_t device, void *stream, const double *cen, int64_t M, int32_t D, int64_t r0, int64_t r1,
                     const uint32_t *nbr, const int32_t *cnt, double delta, uint64_t *submask);
/* Offline stage 3: weighted-neighbour bit rows for rows [r0, r1); submask_all [M] is the gathered mask of all rows. */
int ccb_off_weighted(int32_t device, void *stream, const double *cen, int64_t M, int32_t D, int64_t r0, int64_t r1,
                     const uint32_t *nbr, const uint64_t *submask_all, double k, double E2, uint32_t *wnbr);
/* Offline stage 4: ordered cluster growth over the full weighted-neighbour matrix wnbr [M][words].
 * label [M] (-1 none), order [M] = MC indices in claim order grouped by cluster, cl_off [M+1], n_cl [1].
 * csr_min_m: as ccb_params.off_csr_min_m (0 = default).
 * Clusters whose accumulated weight is not > 0 are dropped by the caller (predecon.py:83). */
int ccb_off_clusters(int32_t device, void *stream, int64_t M, const uint32_t *wnbr, const uint8_t *core,
                     const uint64_t *submask_all, double k, int64_t pi, int32_t csr_min_m, int32_t *label, int32_t *order,
                     int32_t *cl_off, int32_t *n_cl);

/* Offline stage 4, sharded form (config C4): instead of all-gathering the weighted-neighbour BIT ROWS (M^2 / 8 bytes), every
 * rank turns its own rows [r0, r1) into CSR form and only the lists travel.
 * ccb_offc_rowinfo: per own row the isolated flag (WN(p) = {p}) and the number of CSR entries it needs (0 if isolated);
 *   wnbr_rows [(r1-r0)][words], iso / nnz [(r1-r0)].
 * ccb_offc_fill: column indices of the own non-isolated rows into the GLOBAL CSR col at off_all[row] (iso_all [M], off_all
 *   [M + 1] = exclusive prefix of the gathered nnz; the caller merges the ranks' disjoint segments, e.g. by an all-reduce).
 * ccb_off_clusters_csr: the ordered cluster growth of ccb_off_clusters over that CSR (same outputs). */
int ccb_offc_rowinfo(int32_t device, void *stream, const uint32_t *wnbr_rows, int64_t M, int64_t r0, int64_t r1, uint8_t *iso,
                     int32_t *nnz);
int ccb_offc_fill(int32_t device, void *stream, const uint32_t *wnbr_rows, int64_t M, int64_t r0, int64_t r1,
                  const uint8_t *iso_all, const int64_t *off_all, int32_t *col);
int ccb_off_clusters_csr(int32_t device, void *stream, int64_t M, const int64_t *off, const int32_t *col, const uint8_t *iso,
                         const uint8_t *core, const uint64_t *submask_all, double k, int64_t pi, int32_t *label, int32_t *order,
                         int32_t *cl_off, int32_t *n_cl);

#ifdef __cplusplus
}
#endif
#endif /* CHRONOCLUST_B200_H */
