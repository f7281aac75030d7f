/*
 * rr_b200.h -- C ABI of librr_b200.so, the B200 (sm_100a) replacement for the routing hot
 * path of rileyhales/river-route.  Plain pointers and sizes only; no torch / numpy types.
 *
 * Every entry point names the reference interface it replaces (paths relative to the
 * reference repository root).  All functions return 0 on success, non-zero on failure;
 * rr_last_error() returns a thread-local description of the last failure.
 *
 * Conventions
 *   - fp64 arithmetic everywhere; index arrays are int32 (scipy's run-time dtype for the
 *     reference's CSC arrays), reach counts are int64.
 *   - 2-D arrays are time-major with an explicit leading dimension in ELEMENTS:
 *     a[t * ld + reach], exactly the reference's C-contiguous (T, n) layout when ld == n.
 *   - "host" entry points take host pointers (pageable or pinned) and stream chunks of
 *     time steps through pinned double buffers; "dev" entry points take device pointers
 *     (e.g. torch.Tensor.data_ptr()) and a cudaStream_t passed as void*.
 *   - There is no CPU fallback: without a CUDA device every compute call fails.
 */
#ifndef RR_B200_H
#define RR_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct rr_plan rr_plan;

/* Router variants (the three numba kernels of river_route/routers/_numba_kernels.py). */
enum {
    RR_MODE_MUSKINGUM = 0, /* muskingum_route, _numba_kernels.py:9-46   */
    RR_MODE_RAPID     = 1, /* rapid_route,     _numba_kernels.py:49-84  */
    RR_MODE_UNIT      = 2  /* unit_route,      _numba_kernels.py:88-171 */
};

/* Tunables of the wavefront solve; zero / negative fields mean "choose for me". */
typedef struct rr_plan_opts {
    int32_t time_tile;      /* routing substeps advanced per work item (default 64)          */
    int32_t tile_stride;    /* ticket-key distance between consecutive tiles of one block;
                               0 = smallest power of two whose exchange rings fit the budget */
    int32_t device;         /* CUDA device ordinal (default: current device)                 */
    int32_t threads_per_cta;/* persistent CTA size, multiple of 32 (default 256)             */
    int64_t raw_budget_bytes;/* cap for the exchange buffer (default 16 GiB)                 */
    int32_t renumber;       /* 0 auto, 1 keep the params_file order, 2 always work on reaches sorted
                               by topological level (inputs/outputs stay in params_file order; the
                               library permutes them on the device)                             */
    int32_t staging;        /* renumbered plans: 0 auto: the direct pipeline (rr_direct.cu: staging kernels + direct-exchange
                               wavefront; headwater blocks routed while staging when the network has >= 2^18 reaches)
                               whenever it applies (one substep per row, RapidMuskingum / Muskingum, time_tile a multiple
                               of 16), else as 2.  6: direct pipeline, headwaters always routed while staging; 7: never.
                               Experiments kept for comparison: 1 register path on row-major working arrays, 2 register
                               path on tile-major working arrays with exchange rings, 3 bulk-async-copy (TMA) staged
                               kernel, 4 as 2 with reach-major discharge tiles, 5 as 2 with [row group][lane][4]
                               lateral tiles                                                                   */
} rr_plan_opts;

/* Host-visible description of a built plan (for tests, DESIGN.md numbers and bench.py). */
typedef struct rr_plan_info {
    int64_t n;               /* reaches                                                     */
    int64_t n_edges;         /* reaches with a downstream reach                              */
    int64_t n_blocks;        /* 32-reach blocks                                              */
    int64_t n_export;        /* reaches whose downstream lives in another block              */
    int64_t n_internal_edges;/* edges served by in-warp shuffles                             */
    int32_t max_skew;        /* largest in-block systolic delay                              */
    int32_t max_indegree;    /* largest number of upstream reaches of one reach              */
    int32_t max_block_level; /* depth of the block dependency DAG                            */
    int32_t n_outlets_lo;    /* number of outlets (low 32 bits)                              */
    int64_t n_dep_edges;     /* distinct (block -> upstream block) dependencies              */
    int64_t device_bytes;    /* bytes of plan-owned device memory (after first upload)       */
    int32_t renumbered;      /* 1 when the plan works on level-sorted reaches                */
    int32_t reach_depth;     /* longest upstream-to-outlet path, in reaches                  */
    int32_t all_fast;        /* 1 when every block is fast-path eligible (no in-block edge, in-degree <= 4) */
    int32_t narrow_blocks;   /* blocks in levels narrower than 4096 blocks (progress published per 16 rows) */
    int64_t n_headwaters;    /* reaches without upstream (level 0)                                          */
    int64_t n_work;          /* working slots: n, or more when every level is padded to whole 32-reach blocks */
} rr_plan_info;

const char *rr_last_error(void);
int  rr_version(void);
/* 1 when a CUDA device is usable from this process, else 0 (never falls back to CPU). */
int  rr_cuda_available(void);

/* ---- topology --------------------------------------------------------------------------
 * Replaces river_route.tools.adjacency_matrix (tools.py:75-109) and the pre-checks of
 * Muskingum._set_network_dependent_vectors (routers/Muskingum.py:153-167).
 * Writes down_idx[i] = index of the reach downstream of i, or -1 for outlets
 * (downstream_id < 0, tools.py:98-99).  Status codes mirror the reference's ValueErrors:
 *   1 duplicate river id (Muskingum.py:153-154)        -> *bad = the id
 *   2 unknown downstream id (tools.py:101-102)         -> *bad = the id
 *   3 not topologically sorted (tools.py:103-104)      -> *bad = the upstream index
 * The first offending row in file order is reported, as the reference's loop does. */
int rr_downstream_index(int64_t n, const int64_t *river_ids, const int64_t *downstream_ids,
                        int32_t *down_idx, int64_t *bad);

/* Basin (connected component) label of every reach = index of its terminal outlet, and
 * optional LPT bin-packing of basins over n_parts devices by reach count
 * (docs/references/parallelism.md:67-75 names watersheds as the unit of parallelism).
 * basin[i] in [0, n_basins); part[i] in [0, n_parts) (part may be NULL). */
int rr_label_basins(int64_t n, const int32_t *down_idx, int32_t *basin, int64_t *n_basins,
                    int32_t n_parts, int32_t *part);

/* ---- plan -------------------------------------------------------------------------------
 * A plan owns everything derived from the network alone: the upstream-CSR in ascending
 * upstream order, 32-reach blocks, in-block systolic delays, block dependency lists, the
 * wavefront ticket order and (lazily) their device copies and the exchange buffer.
 * It plays the role of the reference's cached CSC arrays
 * (Muskingum._set_muskingum_coefficients, routers/Muskingum.py:187-193). Host only; needs
 * no GPU until the first route call. */
int  rr_plan_create(int64_t n, const int32_t *down_idx, const rr_plan_opts *opts, rr_plan **out);
void rr_plan_destroy(rr_plan *p);
int  rr_plan_get_info(const rr_plan *p, rr_plan_info *info);

/* Coefficients c1,c2,c3 (Muskingum.py:176-179) and c4_dt = (c1+c2)/dt_runoff
 * (TransformMuskingum.py:104, RapidMuskingum.py:25); host pointers, length n, computed by
 * the caller with the reference's exact numpy expressions so they are bit-identical.
 * c4_dt may be NULL for RR_MODE_MUSKINGUM / RR_MODE_UNIT. */
int rr_plan_set_coefficients(rr_plan *p, const double *c1, const double *c2, const double *c3,
                             const double *c4_dt);

/* ---- routing ----------------------------------------------------------------------------
 * One call == one call of the reference kernel:
 *   RR_MODE_RAPID     rapid_route(csc..., c2, c3, c4_dt, q_t, qlateral, discharge_array,
 *                                 num_substeps)                       _numba_kernels.py:50-55
 *   RR_MODE_MUSKINGUM muskingum_route(csc..., c2, c3, q_t, discharge_array,
 *                                 num_output_steps, num_routing_per_output)        :9-14
 *                     (T = num_output_steps, substeps = num_routing_per_output, lateral NULL)
 *   RR_MODE_UNIT      unit_route(...)                                              :89-99
 *                     lateral = convolved lateral over ALL reaches; q_state = full-length
 *                     channel state; headwater/inner split is derived inside the plan
 *                     (UnitMuskingum._hook_before_route, routers/UnitMuskingum.py:39-46) and
 *                     the returned state is the recombined vector of :94-98.
 * q_state [n] is read as the initial state and overwritten with the final state (the
 * reference mutates q_t in place).  out is [T][ldo] and fully overwritten.
 * q_full is used by RR_MODE_UNIT only and may be NULL:
 *   NULL      router-level semantics: q_ch = q_full = q_state on entry
 *             (UnitMuskingum.py:78-79), q_state = recombined final vector on exit (:94-98);
 *   non-NULL  kernel-level semantics of unit_route's q_ch / q_full argument pair, both
 *             full length n: q_state is q_ch, q_full is q_full, both read and both updated
 *             (entries of headwater reaches are ignored and left untouched).
 * Device variant: all pointers are device pointers on the plan's device; the call is
 * asynchronous on `stream`. */
int rr_route_dev(rr_plan *p, int mode, double *q_state, double *q_full, const double *lateral,
                 int64_t ldl, double *out, int64_t ldo, int64_t T, int64_t substeps, void *stream);

/* Host variant: host pointers; time is cut into chunks that are copied through pinned
 * double buffers (cudaMemcpyAsync) overlapping H2D, compute and D2H.  Synchronous. */
int rr_route_host(rr_plan *p, int mode, double *q_state, double *q_full, const double *lateral,
                  int64_t ldl, double *out, int64_t ldo, int64_t T, int64_t substeps);

/* Host variant with the output tail of the reference's router loop done on the device before the copy back:
 * `resample` >= 1 consecutive rows are averaged (q_array.reshape(T/k, k, n).mean(axis=1),
 * routers/TransformMuskingum.py:128-139; rows added in order, then divided by k) and, with out_f32 != 0, the result
 * is cast to float32 exactly as the reference's `astype(np.float32)` before the writer (:146, Muskingum.py:259).
 * out is [T / resample][ldo] of float64 or float32; T must be a multiple of resample.  Halves (or more) the
 * device-to-host traffic of a run; results are bit-identical to doing both steps in numpy on the fp64 array. */
int rr_route_host_ex(rr_plan *p, int mode, double *q_state, double *q_full, const double *lateral,
                     int64_t ldl, void *out, int64_t ldo, int64_t T, int64_t substeps, int out_f32,
                     int64_t resample);

/* As rr_route_host_ex with lateral inflows stored as float32 (lateral_f32 != 0; ldl in float32 elements): the rows
 * cross PCIe as they are stored and are upcast on the device.  The reference upcasts a float32 qlateral variable on the
 * host with astype(float64) (routers/TransformMuskingum.py:36); the conversion is exact, so results are bit-identical
 * while the host-to-device traffic halves. */
int rr_route_host_typed(rr_plan *p, int mode, double *q_state, double *q_full, const void *lateral, int lateral_f32,
                        int64_t ldl, void *out, int64_t ldo, int64_t T, int64_t substeps, int out_f32, int64_t resample);

/* Restrict what the host streaming calls (rr_route_host, rr_route_host_ex, rr_runoff_route_host) copy back to a
 * subset of river segments -- the device-side form of the reference's "save a subset of the routed flows" writer
 * pattern (docs/tutorial/advanced.md:147-170), e.g. gauges or basin outlets only.  idx are params-file indices in
 * any order; out then is [T / resample][ldo >= n_sub] with column s = segment idx[s].  All segments are still
 * routed and q_state is still the full final state.  n_sub = 0 restores the full output. */
int rr_plan_set_output_subset(rr_plan *p, int64_t n_sub, const int32_t *idx);

/* Ensemble: n_members independent lateral arrays routed from the SAME initial state in one
 * launch (TransformMuskingum._execute_routing 'ensemble' mode, TransformMuskingum.py:121-126).
 * lateral[m], out[m], q_final[m] are device pointers per member; q_init [n] is shared. */
int rr_route_ensemble_dev(rr_plan *p, int mode, const double *q_init, int32_t n_members,
                          const double *const *lateral, int64_t ldl, double *const *out, int64_t ldo,
                          double *const *q_final, int64_t T, int64_t substeps, void *stream);

/* Output rows one work item of the wavefront kernel covers in a call of T rows x substeps (the time tile the
 * per-call cost model picks; bench.py's roofline arithmetic: coefficients and topology are read once per tile). */
int64_t rr_plan_tile_rows(const rr_plan *p, int64_t T, int64_t substeps);

/* Ensemble from host arrays (pinned for full PCIe rate): lateral[m] / out[m] are host pointers per member, float64 or
 * float32 as flagged; time is cut into chunks, and the members of a chunk are routed by one launch.  q_init is the
 * shared initial state [n] (ld_init = 0) or, for a later time slab of the same members, one state per member
 * [n_members][ld_init]; q_final (optional, [n_members][ldq]) receives every member's final state and q_mean (optional,
 * [n]) their mean, accumulated in member order and divided by the count exactly as np.array(states).mean(axis=0) does
 * (TransformMuskingum.py:145-146).  out_f32 / resample as rr_route_host_ex.  RR_MODE_RAPID / RR_MODE_MUSKINGUM. */
int rr_route_ensemble_host(rr_plan *p, int mode, const double *q_init, int64_t ld_init, int32_t n_members, const void *const *lateral,
                           int lateral_f32, int64_t ldl, void *const *out, int64_t ldo, int out_f32, double *q_final,
                           int64_t ldq, double *q_mean, int64_t T, int64_t substeps, int64_t resample);

/* ---- ensemble statistics ---------------------------------------------------------------------
 * Per-time-step statistics across ensemble members, computed on the device so that only the statistics cross PCIe
 * (S rows instead of M member rows per time step).  Every statistic is bit-identical to numpy on the stacked
 * (members, rows, n) fp64 array:
 *   RR_STAT_MEAN        np.mean(axis=0): members added in member order, then divided by M
 *   RR_STAT_STD         np.std(axis=0) (ddof = 0): d = x - mean, d*d added in member order, / M, sqrt
 *   RR_STAT_MIN / MAX   np.min / np.max
 *   RR_STAT_PERCENTILE  np.percentile(axis=0, q) with numpy's default 'linear' method, q an integer in [0, 100]
 *   RR_STAT_EXCEED      np.mean(x > thr[q], axis=0): the fraction of members strictly above the reach's threshold in
 *                       row q of the thresholds (x == thr does not count; a NaN threshold is never exceeded: 0.0)
 * Input contract: no NaN (routed discharge is clamped to >= +0 and never NaN; resample means keep that).
 * Horizon peaks (the _ex forms): per statistic and column, the maximum over the output rows and the first row where
 * it occurs, i.e. rows.max(axis=0) and rows.argmax(axis=0) of the fp64 statistic rows (ties: the earliest row). */
#define RR_MAX_STATS 16
enum { RR_STAT_MEAN = 0, RR_STAT_STD = 1, RR_STAT_MIN = 2, RR_STAT_MAX = 3, RR_STAT_PERCENTILE = 4, RR_STAT_EXCEED = 5 };
typedef struct rr_stats_spec {
    int32_t n_stats;             /* 1 .. RR_MAX_STATS                                                            */
    int32_t kind[RR_MAX_STATS];  /* RR_STAT_*                                                                    */
    int32_t q[RR_MAX_STATS];     /* percentile in [0, 100] of RR_STAT_PERCENTILE entries; threshold row of EXCEED */
} rr_stats_spec;

/* Per-river thresholds (e.g. return-period flows) for RR_STAT_EXCEED in params-file (user) order: host [n_thr][ldt],
 * ldt >= n, copied; uploaded to the plan's device lazily and versioned like the output subset.  n_thr = 0 clears. */
int rr_plan_set_thresholds(rr_plan *p, int32_t n_thr, const double *thr, int64_t ldt);

/* The statistics kernel alone, on device pointers: member m, row t, reach i is x[m * member_stride + t * ld + i]
 * (1 <= n_members <= 64).  out[s] (device pointers, one per statistic) is [rows][ldo], float32 (out_f32 != 0) or
 * float64; column c shows reach subset[c] (device int32 array; NULL: reach c).  Asynchronous on `stream`. */
int rr_ensemble_stats_dev(const rr_stats_spec *stats, int32_t n_members, const double *x, int64_t member_stride,
                          int64_t ld, int64_t rows, int64_t n_out, const int32_t *subset, void *const *out, int64_t ldo,
                          int out_f32, void *stream);

/* rr_ensemble_stats_dev plus thresholds and running peaks.  thr: device [n_thr][ldt], indexed by reach (column c reads
 * thr[q * ldt + subset[c]]); needed by RR_STAT_EXCEED entries, NULL otherwise.  peak / peak_row: device [n_stats][ldk]
 * fp64 / int32, read and updated: where a statistic's value at row t is strictly greater than peak[s][c], peak[s][c]
 * becomes that value and peak_row[s][c] becomes row0 + t.  Start peak at -inf; launches over consecutive rows with
 * row0 = the global index of each launch's first row then give the maximum over all of them and its first row.  out
 * may be NULL (no per-step rows) when peak is given; peak needs peak_row.  No atomics: the result is deterministic. */
int rr_ensemble_stats_dev_ex(const rr_stats_spec *stats, int32_t n_members, const double *x, int64_t member_stride,
                             int64_t ld, int64_t rows, int64_t n_out, const int32_t *subset, const double *thr,
                             int64_t ldt, void *const *out, int64_t ldo, int out_f32, double *peak, int32_t *peak_row,
                             int64_t ldk, int64_t row0, void *stream);

/* rr_route_ensemble_host with the member outputs reduced on the device: per time chunk, all members are routed into an
 * fp64 device scratch, averaged over `resample` rows, reduced to the statistics of `stats`, and only those are copied
 * back: out[s] is a host array [T / resample][ldo] (float32 or float64).  Honours the plan's output subset
 * (rr_plan_set_output_subset).  Inputs, q_init / ld_init, q_final and q_mean as rr_route_ensemble_host.  The chunk
 * length follows the free device memory; a call fails when not even one output row of all members fits. */
int rr_route_ensemble_stats_host(rr_plan *p, int mode, const double *q_init, int64_t ld_init, int32_t n_members,
                                 const void *const *lateral, int lateral_f32, int64_t ldl, const rr_stats_spec *stats,
                                 void *const *out, int64_t ldo, int out_f32, double *q_final, int64_t ldq, double *q_mean,
                                 int64_t T, int64_t substeps, int64_t resample);

/* rr_route_ensemble_stats_host with the plan's thresholds (rr_plan_set_thresholds; RR_STAT_EXCEED reads the threshold
 * of reach subset[c] for column c) and optional horizon peaks: peak / peak_row are host [n_stats][ldk], fp64 value and
 * int32 output row relative to this call, over the call's T / resample rows (the library initialises them).  out may be
 * NULL when peak is given: then no per-step rows are kept on the device or copied back. */
int rr_route_ensemble_stats_host_ex(rr_plan *p, int mode, const double *q_init, int64_t ld_init, int32_t n_members,
                                    const void *const *lateral, int lateral_f32, int64_t ldl, const rr_stats_spec *stats,
                                    void *const *out, int64_t ldo, int out_f32, double *q_final, int64_t ldq,
                                    double *q_mean, int64_t T, int64_t substeps, int64_t resample, double *peak,
                                    int32_t *peak_row, int64_t ldk);

/* Kernel launches issued by this library on this thread since the last reset (bench.py's
 * gpu_launches claim). */
int64_t rr_launch_count(int reset);
/* Optional device timing of this library's kernels with CUDA events on the launching stream:
 * ms[0] routing kernel, ms[1] permute to working order, ms[2] permute to params order, ms[3] other;
 * counts[] = launches per class.  rr_timing_read synchronises on the recorded events. */
int rr_timing_enable(int on);
int rr_timing_read(double *ms, int64_t *counts, int reset);

/* ---- unit hydrograph ----------------------------------------------------------------------
 * Replaces UnitHydrograph.convolve (river_route/uhkernels/UnitHydrograph.py:77-107):
 * out[t,b] = carry-in + sum_tau kernel[tau,b] * lateral[t-tau,b], accumulated oldest
 * contribution first (the order of convolve_incrementally, :64-75); state [n_ks][lds] is
 * updated in place with the tail that spills past T (:100-105).  Device pointers. */
int rr_uh_convolve_dev(int64_t n, int64_t n_ks, int64_t T,
                       const double *lateral, int64_t ldl, const double *kernel, int64_t ldk,
                       double *state, int64_t lds, double *out, int64_t ldo, void *stream);
int rr_uh_convolve_host(int64_t n, int64_t n_ks, int64_t T,
                        const double *lateral, int64_t ldl, const double *kernel, int64_t ldk,
                        double *state, int64_t lds, double *out, int64_t ldo);

/* ---- grid weights -------------------------------------------------------------------------
 * Replaces the SpMM core and in-place tail of runoff_to_qlateral (river_route/runoff.py:292-337):
 * y[t,r] = sum_j w[j] * x[t, col[j]] over CSR row r in stored order, then
 * cumulative->incremental, optional clip at 0, NaN->0, optional multiply by area[r].
 * x is the gathered grid runoff [T][ldx], float32 (x_is_f32 != 0) or float64; the product
 * is formed in fp64 as the reference's scipy call does.  Device pointers.
 * force_positive: bit 0 = clip at zero (force_positive_runoff, :313-314); bit 1 = leave NaN in place -- for the
 * rare irregular-time-axis path, where the reference resamples the series (:316-329) BEFORE it zeroes NaN. */
int rr_weights_transform_dev(int64_t n_rivers, int64_t n_points, int64_t T, const int32_t *indptr,
                             const int32_t *indices, const double *w, const void *x, int x_is_f32,
                             int64_t ldx, double *y, int64_t ldy, int cumulative, int force_positive,
                             const double *area, void *stream);
int rr_weights_transform_host(int64_t n_rivers, int64_t n_points, int64_t T, const int32_t *indptr,
                              const int32_t *indices, const double *w, const void *x, int x_is_f32,
                              int64_t ldx, double *y, int64_t ldy, int cumulative, int force_positive,
                              const double *area);

/* ---- gridded runoff -> discharge in one residency -----------------------------------------------
 * The whole per-file chain of TransformMuskingum.route() with grid inputs (routers/TransformMuskingum.py:38-51,
 * :108-148) without the lateral inflows ever leaving the device:
 *   gathered grid runoff (host, float32 or float64, [T][ldx] in unique-cell order, runoff.py:267-280)
 *   -> weight SpMM + tail (runoff.py:292-337)  [-> UnitHydrograph.convolve, RR_MODE_UNIT, UnitMuskingum.py:75]
 *   -> route -> optional resample / float32 (as rr_route_host_ex) -> host.
 * An rr_transform is the device-resident weight table in CSR form over the plan's river order (row r = river r of
 * the params file; the reference assumes, runoff.py:265, that the table lists rivers in that order), built on the
 * host exactly as scipy builds W (duplicates summed, columns ascending); area may be NULL when as_volumes is never
 * used.  rr_transform_set_uh attaches the (n_ks, n) unit-hydrograph kernel and carry-over state
 * (uhkernels/UnitHydrograph.py:27-62); the state lives on the device across calls like UnitHydrograph.state does
 * across files and is read back with rr_transform_get_uh_state. */
typedef struct rr_transform rr_transform;
int  rr_transform_create(int64_t n_rivers, int64_t n_points, const int32_t *indptr, const int32_t *indices,
                         const double *w, const double *area, int32_t device, rr_transform **out);
int  rr_transform_set_uh(rr_transform *t, int64_t n_ks, const double *kernel, int64_t ldk,
                         const double *state /* NULL = zeros */, int64_t lds);
int  rr_transform_get_uh_state(rr_transform *t, double *state, int64_t lds);
void rr_transform_destroy(rr_transform *t);
/* mode: RR_MODE_RAPID (as_volumes as RapidMuskingum sets it) or RR_MODE_UNIT (depths -> unit hydrograph).
 * cumulative / force_positive are runoff_to_qlateral's options (runoff.py:309-314). */
int rr_runoff_route_host(rr_plan *p, rr_transform *t, int mode, double *q_state, const void *runoff,
                         int x_is_f32, int64_t ldx, int64_t T, int cumulative, int force_positive,
                         int as_volumes, void *out, int64_t ldo, int64_t substeps, int out_f32,
                         int64_t resample);

/* Diagnostic cycle counters of the routing kernel (builds with -DRR_PROFILE; zeros otherwise), summed over warps:
 * [0] ticket + decode, [1] per-item constants + dependency waits, [2] item body, [3] publish.  Resets on read. */
int rr_plan_read_profile(rr_plan *p, uint64_t *out8);

/* ---- pinned host memory for the streaming path ---------------------------------------------- */
int rr_host_alloc(void **ptr, int64_t bytes);
int rr_host_free(void *ptr);

/* ---- synthetic networks (SURVEY.md section 8d; used by tests and bench.py) -------------------
 * Forest grown upstream from outlets; final index = reverse growth order, so down[i] > i.
 * basin sizes ~ lognormal(sigma) normalised to n.  main_stem > 0 pre-seeds a chain of that
 * length in the first basin.  Deterministic for a given seed on every platform. */
int rr_synth_forest(int64_t n, int64_t n_basins, uint64_t seed, double depth_bias,
                    int64_t main_stem, double sigma, int32_t *down_idx);

/* ---- plan introspection for tests (host copies; pointers valid until rr_plan_destroy) -------- */
int rr_plan_get_arrays(const rr_plan *p,
                       const int32_t **up_ptr,   /* [n+1]   upstream-CSR row pointers            */
                       const int32_t **up_idx,   /* [edges] upstream reach indices, ascending    */
                       const uint8_t **skew,     /* [n]     in-block systolic delay              */
                       const int32_t **slot_src, /* [edges] >=0 export id of an external upstream,
                                                            <0: -(lane+1) of an in-block upstream */
                       const int32_t **export_id,/* [n]     compact id in the exchange buffer or -1 */
                       const int32_t **blk_level,/* [n_blocks] level in the block DAG            */
                       const int32_t **dep_ptr,  /* [n_blocks+1]                                 */
                       const int32_t **dep_idx,  /* distinct upstream blocks                     */
                       const int32_t **exp_span, /* [n_export] block-level distance producer -> consumer */
                       const int32_t **perm      /* [n_work] user index of each working slot (-1: padding), NULL if not renumbered */);
/* Ticket -> (block, tile) decode used by the kernel, for schedule-validity tests. */
int rr_plan_schedule(const rr_plan *p, int64_t n_tiles, int32_t tile_stride, int64_t *n_items,
                     int32_t *item_block /* [n_blocks*n_tiles] or NULL */,
                     int32_t *item_tile  /* same */);

#ifdef __cplusplus
}
#endif
#endif /* RR_B200_H */
