// rr_stats.cu -- per-time-step statistics across ensemble members (mean, std, min, max, percentiles, threshold
// exceedance) and their running peaks over the time rows, for sm_100a.
//
// One thread per (output row, output column): it loads the M member values of its reach into registers (averaging
// `k` consecutive rows first when the output is resampled), forms mean / std in member order, and, when a percentile
// is asked for, sorts the values with a fully unrolled bitonic network over M padded with +inf to 8 / 16 / 32 / 64.
// Every value is read once and every statistic written once: M * k * 8 B in, S * (4 or 8) B out per (row, column).
//
// The results are bit-identical to numpy on the stacked (M, rows, n) fp64 array, so every product, sum and quotient
// is rounded on its own (__dmul_rn / __dadd_rn / __dsub_rn / __ddiv_rn: nvcc would otherwise contract to FMAs):
//   mean  np.mean(axis=0)      sum in member order, / M
//   std   np.std(axis=0)       d = x - mean; d*d summed in member order; / M; sqrt (ddof = 0)
//   pQ    np.percentile        'linear': v = (M-1) * (Q/100), lo = floor(v), hi = min(lo+1, M-1), g = v - lo;
//                              a + (b-a)*g for g < 0.5, else b - (b-a)*(1-g)  (numpy's _lerp); v, lo, g on the host
//   exceed np.mean(x > thr[q])  members strictly above the reach's threshold, counted over the M real slots (the count
//                              does not depend on their order, so it holds after the sort too), / M; NaN never exceeds
//
// Peak mode (PEAK): statistic s also keeps a running maximum over the output rows, peak[s][c] (fp64) and its first row
// peak_row[s][c] = row0 + t: updated on a strict '>' against the stored value (the caller starts it at -inf), which is
// rows.max(axis=0) / rows.argmax(axis=0) of the fp64 statistic rows, ties to the first row, and carries across launches.
// The grid then has one row of CTAs: the thread of column c walks every row in order and is the only one to touch the
// column's peak, so there are no atomics and the result is deterministic.  The peak is kept in global memory, 12 B read
// and written per (row, column, statistic) next to the M * 8 B of member values the thread reads anyway, because
// registers are the kernel's limit (the P = 64 sorting instantiation).
// Inputs are routed discharge, never NaN (the output clamp maps NaN and negatives to +0), so plain compares order them.
#include <cuda_runtime.h>
#include <math_constants.h>

#include <algorithm>
#include <climits>
#include <cmath>
#include <string>

#include "rr_internal.h"

void rr_count_launch(int64_t k);

#define CK(call)                                                                \
    do {                                                                        \
        cudaError_t e_ = (call);                                                \
        if (e_ != cudaSuccess) {                                                \
            rr_set_error(std::string(#call) + ": " + cudaGetErrorString(e_));   \
            return 200;                                                         \
        }                                                                       \
    } while (0)

namespace {

constexpr int kThreads = 128;

struct stats_args {
    int32_t n_stats, n_exceed;
    int32_t kind[RR_MAX_STATS], lo[RR_MAX_STATS], hi[RR_MAX_STATS];   // exceed: lo = threshold row
    double g[RR_MAX_STATS];
    void *out[RR_MAX_STATS];   // NULL: no per-step rows of that statistic
    const double *thr;         // [n_thr][ldt] by reach
    int64_t ldt;
    double *peak;              // PEAK: [n_stats][ldk]
    int32_t *peak_row;
    int64_t ldk, row0;
};

// v[idx] for an index that is the same in every thread: selects keep the array in registers (a dynamic index would
// move it to local memory)
template <int P>
__device__ __forceinline__ double pick(const double (&v)[P], int idx) {
    double r = v[0];
#pragma unroll
    for (int j = 1; j < P; ++j) r = (j == idx) ? v[j] : r;
    return r;
}

template <int P, bool SORT, bool PEAK, typename OT>
__global__ void __launch_bounds__(kThreads) ensemble_stats_kernel(const __grid_constant__ stats_args a, const double *__restrict__ x, int M,
                                                                  int64_t mstride, int64_t ld, int k, int64_t rows,
                                                                  int64_t n_out, const int32_t *__restrict__ subset,
                                                                  int64_t ldo) {
    const int64_t c = (int64_t)blockIdx.x * kThreads + threadIdx.x;
    if (c >= n_out) return;
    const int64_t i = subset ? (int64_t)__ldg(subset + c) : c;
    for (int64_t t = blockIdx.y; t < rows; t += gridDim.y) {
        const double *p = x + t * k * ld + i;
        double v[P];
        // all loads of a row are issued before any is used (no branch per member: slots past M re-read member M-1, an
        // L1 hit, and become +inf); finish_output's resample: rows added in order, then / k
#pragma unroll
        for (int m = 0; m < P; ++m) v[m] = __ldg(p + (int64_t)min(m, M - 1) * mstride);
#pragma unroll 1
        for (int r = 1; r < k; ++r) {
#pragma unroll
            for (int m = 0; m < P; ++m) v[m] = __dadd_rn(v[m], __ldg(p + (int64_t)min(m, M - 1) * mstride + (int64_t)r * ld));
        }
#pragma unroll
        for (int m = 0; m < P; ++m) {
            if (k > 1) v[m] = __ddiv_rn(v[m], (double)k);
            if (m >= M) v[m] = CUDART_INF;
        }
        double sum = v[0];
#pragma unroll
        for (int m = 1; m < P; ++m)
            if (m < M) sum = __dadd_rn(sum, v[m]);
        const double mean = __ddiv_rn(sum, (double)M);
        double ss = 0.0;
        bool want_std = false;
#pragma unroll
        for (int s = 0; s < RR_MAX_STATS; ++s) want_std |= s < a.n_stats && a.kind[s] == RR_STAT_STD;
        if (want_std) {
            const double d0 = __dsub_rn(v[0], mean);
            ss = __dmul_rn(d0, d0);
#pragma unroll
            for (int m = 1; m < P; ++m) {
                if (m < M) {
                    const double d = __dsub_rn(v[m], mean);
                    ss = __dadd_rn(ss, __dmul_rn(d, d));
                }
            }
        }
        const double sd = __dsqrt_rn(__ddiv_rn(ss, (double)M));
        // statistic s of this row: its per-step value and its running peak
        auto emit = [&](int s, double r) {
            if (a.out[s]) ((OT *)a.out[s])[t * ldo + c] = (OT)r;
            if (PEAK) {
                const int64_t o = (int64_t)s * a.ldk + c;
                if (r > a.peak[o]) { a.peak[o] = r; a.peak_row[o] = (int32_t)(a.row0 + t); }
            }
        };
        double lo_v, hi_v;
        if (SORT) {
#pragma unroll
            for (int size = 2; size <= P; size <<= 1) {
#pragma unroll
                for (int stride = size >> 1; stride > 0; stride >>= 1) {
#pragma unroll
                    for (int j = 0; j < P; ++j) {
                        const int l = j ^ stride;
                        if (l > j) {
                            // one compare, two selects: no NaN to order (fmin / fmax would test for it)
                            const double e = v[j], f = v[l];
                            const bool swap = ((j & size) == 0) ? (f < e) : (e < f);
                            v[j] = swap ? f : e;
                            v[l] = swap ? e : f;
                        }
                    }
                }
            }
            lo_v = v[0];
            hi_v = pick(v, M - 1);
        } else {
            lo_v = hi_v = v[0];
#pragma unroll
            for (int m = 1; m < P; ++m) {
                if (m < M) { lo_v = v[m] < lo_v ? v[m] : lo_v; hi_v = v[m] > hi_v ? v[m] : hi_v; }
            }
        }
#pragma unroll
        for (int s = 0; s < RR_MAX_STATS; ++s) {
            if (s >= a.n_stats) break;
            double r;
            switch (a.kind[s]) {
                case RR_STAT_MEAN: r = mean; break;
                case RR_STAT_STD: r = sd; break;
                case RR_STAT_MIN: r = lo_v; break;
                case RR_STAT_MAX: r = hi_v; break;
                case RR_STAT_EXCEED: continue;   // below
                default: {
                    if (!SORT) { r = 0.0; break; }   // unreachable: percentiles launch the sorting instantiation
                    const double va = pick(v, a.lo[s]), vb = pick(v, a.hi[s]);
                    const double diff = __dsub_rn(vb, va), g = a.g[s];
                    r = g < 0.5 ? __dadd_rn(va, __dmul_rn(diff, g)) : __dsub_rn(vb, __dmul_rn(diff, __dsub_rn(1.0, g)));
                }
            }
            emit(s, r);
        }
        // exceedance in a loop of its own, not unrolled: the member values stay in registers (fixed indices), and the
        // count code exists once instead of once per statistic slot (which would cost registers in every launch)
        if (a.n_exceed) {
#pragma unroll 1
            for (int s = 0; s < a.n_stats; ++s) {
                if (a.kind[s] != RR_STAT_EXCEED) continue;
                const double th = __ldg(a.thr + (int64_t)a.lo[s] * a.ldt + i);
                int cnt = 0;
#pragma unroll
                for (int m = 0; m < P; ++m) cnt += (m < M && v[m] > th) ? 1 : 0;
                emit(s, __ddiv_rn((double)cnt, (double)M));
            }
        }
    }
}

template <int P, bool SORT, bool PEAK>
cudaError_t launch_p(const stats_args &a, int out_f32, dim3 grid, cudaStream_t stream, const double *x, int M, int64_t mstride,
                     int64_t ld, int k, int64_t rows, int64_t n_out, const int32_t *subset, int64_t ldo) {
    if (out_f32) ensemble_stats_kernel<P, SORT, PEAK, float><<<grid, kThreads, 0, stream>>>(a, x, M, mstride, ld, k, rows, n_out, subset, ldo);
    else ensemble_stats_kernel<P, SORT, PEAK, double><<<grid, kThreads, 0, stream>>>(a, x, M, mstride, ld, k, rows, n_out, subset, ldo);
    return cudaGetLastError();
}

template <bool SORT, bool PEAK>
cudaError_t launch_sort(const stats_args &a, int out_f32, dim3 grid, cudaStream_t stream, const double *x, int M, int64_t mstride,
                        int64_t ld, int k, int64_t rows, int64_t n_out, const int32_t *subset, int64_t ldo) {
    if (M <= 8) return launch_p<8, SORT, PEAK>(a, out_f32, grid, stream, x, M, mstride, ld, k, rows, n_out, subset, ldo);
    if (M <= 16) return launch_p<16, SORT, PEAK>(a, out_f32, grid, stream, x, M, mstride, ld, k, rows, n_out, subset, ldo);
    if (M <= 32) return launch_p<32, SORT, PEAK>(a, out_f32, grid, stream, x, M, mstride, ld, k, rows, n_out, subset, ldo);
    return launch_p<64, SORT, PEAK>(a, out_f32, grid, stream, x, M, mstride, ld, k, rows, n_out, subset, ldo);
}

__global__ void __launch_bounds__(256) peak_init_kernel(double *__restrict__ peak, int32_t *__restrict__ peak_row, int64_t count) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < count) { peak[i] = -CUDART_INF; peak_row[i] = 0; }
}

}  // namespace

int rr_stats_prepare(const rr_stats_spec *spec, int32_t n_members, int64_t n_thr, rr_stats_plan *out) {
    if (!spec || !out) { rr_set_error("null argument"); return 100; }
    if (n_members < 1 || n_members > 64) { rr_set_error("ensemble statistics need 1 to 64 members"); return 100; }
    if (spec->n_stats < 1 || spec->n_stats > RR_MAX_STATS) { rr_set_error("between 1 and 16 statistics per call"); return 100; }
    rr_stats_plan sp;
    sp.n_stats = spec->n_stats;
    sp.n_members = n_members;
    for (int s = 0; s < spec->n_stats; ++s) {
        const int kind = spec->kind[s];
        if (kind < RR_STAT_MEAN || kind > RR_STAT_EXCEED) { rr_set_error("unknown statistic kind"); return 100; }
        sp.kind[s] = kind;
        if (kind == RR_STAT_EXCEED) {
            const int q = spec->q[s];
            if (n_thr == 0) { rr_set_error("RR_STAT_EXCEED needs thresholds (rr_plan_set_thresholds)"); return 100; }
            if (q < 0 || q >= n_thr) {
                rr_set_error("threshold index " + std::to_string(q) + " outside the " + std::to_string((long long)n_thr) +
                             " threshold rows set");
                return 100;
            }
            sp.lo[s] = q;
            sp.exceed = 1;
            continue;
        }
        if (kind != RR_STAT_PERCENTILE) continue;
        const int q = spec->q[s];
        if (q < 0 || q > 100) { rr_set_error("percentiles must lie in [0, 100]"); return 100; }
        // np.percentile: quantile = q / 100, virtual index = (n - 1) * quantile, two IEEE operations as in numpy
        const double v = (double)(n_members - 1) * ((double)q / 100.0);
        const double lo = std::floor(v);
        sp.lo[s] = (int32_t)lo;
        sp.hi[s] = std::min<int32_t>(sp.lo[s] + 1, n_members - 1);
        sp.g[s] = v - lo;
        sp.sort = 1;
    }
    *out = sp;
    return 0;
}

int rr_stats_launch(const rr_stats_plan &sp, const double *x, int64_t member_stride, int64_t ld, int k, int64_t rows_out,
                    int64_t n_out, const int32_t *subset, void *const *out, int64_t ldo, int out_f32, const rr_stats_ext &ex,
                    void *stream) {
    if (rows_out <= 0 || n_out <= 0) return 0;
    stats_args a{};
    a.n_stats = sp.n_stats;
    for (int s = 0; s < sp.n_stats; ++s) {
        a.n_exceed += sp.kind[s] == RR_STAT_EXCEED;
        a.kind[s] = sp.kind[s]; a.lo[s] = sp.lo[s]; a.hi[s] = sp.hi[s]; a.g[s] = sp.g[s]; a.out[s] = out ? out[s] : nullptr;
    }
    a.thr = ex.thr; a.ldt = ex.ldt; a.peak = ex.peak; a.peak_row = ex.peak_row; a.ldk = ex.ldk; a.row0 = ex.row0;
    const bool peak = ex.peak != nullptr;
    // peak mode: one thread owns a column across all rows of the launch (grid.y = 1)
    const dim3 grid((unsigned)((n_out + kThreads - 1) / kThreads), peak ? 1u : (unsigned)std::min<int64_t>(rows_out, 65535));
    const cudaStream_t st = (cudaStream_t)stream;
    const int M = sp.n_members;
    cudaError_t e;
    if (sp.sort) e = peak ? launch_sort<true, true>(a, out_f32, grid, st, x, M, member_stride, ld, k, rows_out, n_out, subset, ldo)
                          : launch_sort<true, false>(a, out_f32, grid, st, x, M, member_stride, ld, k, rows_out, n_out, subset, ldo);
    else e = peak ? launch_sort<false, true>(a, out_f32, grid, st, x, M, member_stride, ld, k, rows_out, n_out, subset, ldo)
                  : launch_sort<false, false>(a, out_f32, grid, st, x, M, member_stride, ld, k, rows_out, n_out, subset, ldo);
    CK(e);
    rr_count_launch(1);
    return 0;
}

int rr_stats_peak_init(double *peak, int32_t *peak_row, int64_t count, void *stream) {
    if (count <= 0) return 0;
    peak_init_kernel<<<(unsigned)((count + 255) / 256), 256, 0, (cudaStream_t)stream>>>(peak, peak_row, count);
    CK(cudaGetLastError());
    rr_count_launch(1);
    return 0;
}

extern "C" int rr_ensemble_stats_dev_ex(const rr_stats_spec *stats, int32_t n_members, const double *x, int64_t member_stride,
                                        int64_t ld, int64_t rows, int64_t n_out, const int32_t *subset, const double *thr,
                                        int64_t ldt, void *const *out, int64_t ldo, int out_f32, double *peak, int32_t *peak_row,
                                        int64_t ldk, int64_t row0, void *stream) {
    rr_stats_plan sp;
    // a caller's device threshold array: its row count is not known here, any index >= 0 is taken
    int rc = rr_stats_prepare(stats, n_members, thr ? INT32_MAX : 0, &sp);
    if (rc) return rc;
    if (!x || rows < 0 || n_out < 0) { rr_set_error("bad argument"); return 100; }
    if (!out && !peak) { rr_set_error("no output: give per-step arrays (out), peaks (peak / peak_row) or both"); return 100; }
    if (peak && !peak_row) { rr_set_error("peak needs peak_row"); return 100; }
    if ((out && ldo < n_out) || (!subset && ld < n_out) || (peak && ldk < n_out) || (thr && !subset && ldt < n_out)) {
        rr_set_error("leading dimension smaller than the number of columns");
        return 100;
    }
    if (peak && (row0 < 0 || row0 + rows > INT32_MAX)) { rr_set_error("peak rows must lie in [0, 2^31)"); return 100; }
    for (int s = 0; out && s < sp.n_stats; ++s)
        if (!out[s]) { rr_set_error("null output array"); return 100; }
    rr_stats_ext ex;
    ex.thr = thr; ex.ldt = ldt; ex.peak = peak; ex.peak_row = peak_row; ex.ldk = ldk; ex.row0 = row0;
    return rr_stats_launch(sp, x, member_stride, ld, 1, rows, n_out, subset, out, ldo, out_f32, ex, stream);
}

extern "C" int rr_ensemble_stats_dev(const rr_stats_spec *stats, int32_t n_members, const double *x, int64_t member_stride,
                                     int64_t ld, int64_t rows, int64_t n_out, const int32_t *subset, void *const *out, int64_t ldo,
                                     int out_f32, void *stream) {
    if (!out) { rr_set_error("bad argument"); return 100; }
    return rr_ensemble_stats_dev_ex(stats, n_members, x, member_stride, ld, rows, n_out, subset, nullptr, 0, out, ldo, out_f32,
                                    nullptr, nullptr, 0, 0, stream);
}
