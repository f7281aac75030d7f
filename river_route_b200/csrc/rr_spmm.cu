// rr_spmm.cu -- grid-runoff -> catchment lateral inflow for sm_100a.
//
// Replaces the SpMM core and the in-place tail of runoff_to_qlateral
// (river_route/runoff.py:292-337): y[t,r] = sum_j w[j] * x[t, col[j]] over CSR row r in stored
// (ascending column) order -- scipy's csr_matvecs row-wise axpy order -- then cumulative ->
// incremental, optional clip at zero, NaN -> 0 and optional multiplication by catchment area.
// Memory-bound CSR SpMM with time as the dense dimension: one thread per river so the (T, n)
// output rows are written as coalesced 256-byte segments; the runoff is first re-laid as
// [time block][cell][8 steps] so that each weight entry reads one full 32-byte sector and the CTAs of one
// time block gather from an L2-resident slab.
#include <cuda_runtime.h>

#include <algorithm>
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

constexpr int TB = 8;   // time steps per register block == one 32-byte sector of float32 runoff

// Gathered grid runoff arrives time-major (T, n_points); a catchment touches a handful of scattered
// cells, so reading it in place wastes 7/8 of every sector.  It is re-laid once per call as
// [time block][cell][TB steps]: the TB time steps of one cell are one 32-byte sector (float32), and all the
// sectors of one time block are contiguous -- n_points x 32 bytes, small enough to stay in L2 while one
// launch gathers from it (each cell is read by several catchments, in no particular order).
// One thread per cell and time block: TB coalesced 4- or 8-byte reads down the rows of the time-major array (a warp reads
// 128 / 256 contiguous bytes per row), one whole 32-byte sector (float32; two for float64) written per thread, 1 KB
// contiguous per warp.  (Round 1 went through a 32 x 33 shared-memory tile: 3.0 TB/s under ncu; no tile is needed when the
// block of TB steps is what a thread owns.)
template <typename XT, bool STRIDE>
__global__ void __launch_bounds__(256) transpose_kernel(const XT *__restrict__ x, int64_t ldx, XT *__restrict__ xt,
                                                        int64_t Tp, int64_t T, int64_t n_points) {
    const int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= n_points) return;
    // grid.y is capped at 65535: with more time blocks a CTA strides over them (STRIDE), else it handles one
    int64_t t0 = (int64_t)blockIdx.y * TB;
    do {
        XT v[TB];
#pragma unroll
        for (int u = 0; u < TB; ++u) v[u] = (t0 + u < T) ? __ldg(x + (t0 + u) * ldx + c) : XT(0);
        XT *dst = xt + ((t0 / TB) * n_points + c) * TB;
        if (sizeof(XT) == 4) {
            asm volatile("st.global.v8.f32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"l"(dst), "f"((float)v[0]), "f"((float)v[1]), "f"((float)v[2]),
                         "f"((float)v[3]), "f"((float)v[4]), "f"((float)v[5]), "f"((float)v[6]), "f"((float)v[7]) : "memory");
        } else {
            asm volatile("st.global.v4.f64 [%0], {%1, %2, %3, %4};" ::"l"(dst), "d"((double)v[0]), "d"((double)v[1]), "d"((double)v[2]), "d"((double)v[3]) : "memory");
            asm volatile("st.global.v4.f64 [%0], {%1, %2, %3, %4};" ::"l"(dst + 4), "d"((double)v[4]), "d"((double)v[5]), "d"((double)v[6]), "d"((double)v[7]) : "memory");
        }
    } while (STRIDE && (t0 += (int64_t)gridDim.y * TB) < Tp);
}

template <typename XT> struct vec8;
// 8 consecutive time steps of one cell: one 256-bit load (float) or two (double)
template <> struct vec8<float> {
    float v[8];
    __device__ __forceinline__ void load(const float *p) {
        asm volatile("ld.global.nc.v8.f32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
                     : "=f"(v[0]), "=f"(v[1]), "=f"(v[2]), "=f"(v[3]), "=f"(v[4]), "=f"(v[5]), "=f"(v[6]), "=f"(v[7]) : "l"(p));
    }
};
template <> struct vec8<double> {
    double v[8];
    __device__ __forceinline__ void load(const double *p) {
        asm volatile("ld.global.nc.v4.f64 {%0, %1, %2, %3}, [%4];" : "=d"(v[0]), "=d"(v[1]), "=d"(v[2]), "=d"(v[3]) : "l"(p));
        asm volatile("ld.global.nc.v4.f64 {%0, %1, %2, %3}, [%4];" : "=d"(v[4]), "=d"(v[5]), "=d"(v[6]), "=d"(v[7]) : "l"(p + 4));
    }
};

// One thread per river, TB outputs in registers; row entries are walked in stored (ascending column)
// order so every output accumulates in scipy's csr_matvecs order; the tail of runoff.py:309-337 is fused.
// A CTA handles time block blockIdx.y and, with STRIDE (more than 65535 time blocks: grid.y is capped there), every
// gridDim.y-th block after it.
template <typename XT, bool STRIDE>
__global__ void __launch_bounds__(128) weights_kernel(int64_t n_rivers, int64_t n_points, int64_t T,
                                                      const int32_t *__restrict__ indptr,
                                                      const int32_t *__restrict__ indices,
                                                      const double *__restrict__ w, const XT *__restrict__ xt,
                                                      double *__restrict__ y, int64_t ldy,
                                                      int cumulative, int force_positive,
                                                      const double *__restrict__ area, int64_t t_skip) {
    const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= n_rivers) return;
    const int p0 = __ldg(indptr + r);
    const int p1 = __ldg(indptr + r + 1);
    const double a = area ? __ldg(area + r) : 1.0;
    int64_t t0 = (int64_t)blockIdx.y * TB;
    do {
        double prev = 0.0;   // aggregated value of the step before this block (cumulative input, runoff.py:310-312)
        if (cumulative && t0 > 0)
            for (int j = p0; j < p1; ++j)
                prev = fma(__ldg(w + j), (double)__ldg(xt + (((t0 - 1) / TB) * n_points + __ldg(indices + j)) * TB + (t0 - 1) % TB), prev);
        double acc[TB];
#pragma unroll
        for (int u = 0; u < TB; ++u) acc[u] = 0.0;
        const XT *blk = xt + (t0 / TB) * n_points * TB;
        // (batching the row's gathers for more loads in flight was measured slower: the registers cost occupancy)
        for (int j = p0; j < p1; ++j) {
            const double wj = __ldg(w + j);
            vec8<XT> xv;
            xv.load(blk + (int64_t)__ldg(indices + j) * TB);
#pragma unroll
            for (int u = 0; u < TB; ++u) acc[u] = fma(wj, (double)xv.v[u], acc[u]);
        }
#pragma unroll
        for (int u = 0; u < TB; ++u) {
            if (t0 + u < T && t0 + u >= t_skip) {   // rows before t_skip only seed `prev` (streamed chunks)
                double q = acc[u];
                if (cumulative) { if (t0 + u > 0) q = acc[u] - prev; prev = acc[u]; }
                if ((force_positive & 1) && q < 0.0) q = 0.0;        // :313-314
                if (!(force_positive & 2) && q != q) q = 0.0;        // :331-333 (bit 1: the caller resamples first, :316-329)
                if (area) q *= a;                         // :335-336
                y[(t0 + u - t_skip) * ldy + r] = q;
            } else if (cumulative && t0 + u < T) prev = acc[u];
        }
    } while (STRIDE && (t0 += (int64_t)gridDim.y * TB) < T);
}

template <typename XT>
int run_weights(int64_t n_rivers, int64_t n_points, int64_t T, const int32_t *indptr, const int32_t *indices,
                const double *w, const XT *x, int64_t ldx, double *y, int64_t ldy, int cumulative, int force_positive,
                const double *area, int64_t t_skip, cudaStream_t stream) {
    const int64_t Tp = ((T + TB - 1) / TB) * TB;
    XT *xt = nullptr;
    {   // keep the stream-ordered pool's memory between calls (the default trims it at every sync)
        static thread_local int tuned_device = -1;
        int dev = 0;
        cudaGetDevice(&dev);
        if (tuned_device != dev) {
            cudaMemPool_t pool;
            if (cudaDeviceGetDefaultMemPool(&pool, dev) == cudaSuccess) {
                uint64_t keep = ~0ull;
                cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &keep);
            }
            tuned_device = dev;
        }
    }
    CK(cudaMallocAsync((void **)&xt, sizeof(XT) * (size_t)n_points * Tp, stream));
    // one grid row per time block of TB steps, at most 65535: past that the CTAs stride over the rest (the striding
    // instantiations are separate so that shorter calls keep the registers, and the occupancy, of one block per CTA)
    const bool stride = Tp / TB > 65535;
    const unsigned gy = (unsigned)std::min<int64_t>(Tp / TB, 65535);
    dim3 tg((unsigned)((n_points + 255) / 256), gy);
    if (stride) transpose_kernel<XT, true><<<tg, 256, 0, stream>>>(x, ldx, xt, Tp, T, n_points);
    else transpose_kernel<XT, false><<<tg, 256, 0, stream>>>(x, ldx, xt, Tp, T, n_points);
    CK(cudaGetLastError());
    const int threads = 128;
    const unsigned gx = (unsigned)((n_rivers + threads - 1) / threads);
    // ONE launch, grid.y = time blocks of TB steps: CTAs are dispatched x-fastest, so the launch sweeps all rivers of one time
    // block before the next and the cells of the block in flight (n_points x 32 B, 33 MB at C3) stay in L2 while they are
    // gathered -- each cell is read by several catchments in no particular order.  (A thread that swept all time steps
    // itself cost 13x the algorithmic DRAM reads; one launch per 32 MB of cells, the round-1 scheme, cost 93 launches of 64 us
    // with their ramps and tails at C3.)  Cumulative inputs: a block recomputes the aggregate of the step before it from xt,
    // which holds every row of the call.
    dim3 grid(gx, gy);
    if (stride)
        weights_kernel<XT, true><<<grid, threads, 0, stream>>>(n_rivers, n_points, T, indptr, indices, w, xt, y, ldy, cumulative,
                                                               force_positive, area, t_skip);
    else
        weights_kernel<XT, false><<<grid, threads, 0, stream>>>(n_rivers, n_points, T, indptr, indices, w, xt, y, ldy, cumulative,
                                                                force_positive, area, t_skip);
    CK(cudaGetLastError());
    CK(cudaFreeAsync(xt, stream));
    rr_count_launch(2);
    return 0;
}

}  // namespace

// Internal form used by the streaming pipeline (rr_api.cu): x has T rows of which the first t_skip (0 or 1) only
// provide the previous cumulative value of a streamed time chunk; y receives T - t_skip rows.
int rr_weights_run(int64_t n_rivers, int64_t n_points, int64_t T, const int32_t *indptr, const int32_t *indices,
                   const double *w, const void *x, int x_is_f32, int64_t ldx, double *y, int64_t ldy, int cumulative,
                   int force_positive, const double *area, int64_t t_skip, cudaStream_t stream) {
    if (n_rivers <= 0 || T <= t_skip || n_points <= 0) { rr_set_error("n_rivers, n_points and T must be positive"); return 100; }
    if (!indptr || !indices || !w || !x || !y) { rr_set_error("null argument"); return 100; }
    if (ldx < n_points || ldy < n_rivers) { rr_set_error("leading dimension too small"); return 100; }
    if (x_is_f32)
        return run_weights<float>(n_rivers, n_points, T, indptr, indices, w, (const float *)x, ldx, y, ldy, cumulative,
                                  force_positive, area, t_skip, stream);
    return run_weights<double>(n_rivers, n_points, T, indptr, indices, w, (const double *)x, ldx, y, ldy, cumulative,
                               force_positive, area, t_skip, stream);
}

extern "C" int rr_weights_transform_dev(int64_t n_rivers, int64_t n_points, int64_t T, const int32_t *indptr,
                                        const int32_t *indices, const double *w, const void *x, int x_is_f32,
                                        int64_t ldx, double *y, int64_t ldy, int cumulative, int force_positive,
                                        const double *area, void *stream_) {
    return rr_weights_run(n_rivers, n_points, T, indptr, indices, w, x, x_is_f32, ldx, y, ldy, cumulative, force_positive,
                          area, 0, (cudaStream_t)stream_);
}

extern "C" int rr_weights_transform_host(int64_t n_rivers, int64_t n_points, int64_t T, const int32_t *indptr,
                                         const int32_t *indices, const double *w, const void *x, int x_is_f32,
                                         int64_t ldx, double *y, int64_t ldy, int cumulative, int force_positive,
                                         const double *area) {
    if (n_rivers <= 0 || T <= 0 || n_points <= 0) { rr_set_error("sizes must be positive"); return 100; }
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
        cudaGetLastError();
        rr_set_error("no CUDA device available: librr_b200 has no CPU fallback");
        return 201;
    }
    const size_t es = x_is_f32 ? 4 : 8;
    const int64_t nnz = indptr[n_rivers];
    const int64_t ldyd = ((n_rivers + 31) / 32) * 32;
    int32_t *d_ptr = nullptr, *d_idx = nullptr;
    double *d_w = nullptr, *d_y = nullptr, *d_area = nullptr;
    void *d_x = nullptr;
    CK(cudaMalloc((void **)&d_ptr, sizeof(int32_t) * (size_t)(n_rivers + 1)));
    CK(cudaMalloc((void **)&d_idx, sizeof(int32_t) * (size_t)std::max<int64_t>(nnz, 1)));
    CK(cudaMalloc((void **)&d_w, sizeof(double) * (size_t)std::max<int64_t>(nnz, 1)));
    CK(cudaMalloc((void **)&d_x, es * (size_t)T * n_points));
    CK(cudaMalloc((void **)&d_y, sizeof(double) * (size_t)T * ldyd));
    if (area) CK(cudaMalloc((void **)&d_area, sizeof(double) * (size_t)n_rivers));
    int rc = 0;
    auto fail = [&](cudaError_t e, const char *what) {
        if (e != cudaSuccess && !rc) { rr_set_error(std::string(what) + ": " + cudaGetErrorString(e)); rc = 200; }
    };
    fail(cudaMemcpy(d_ptr, indptr, sizeof(int32_t) * (size_t)(n_rivers + 1), cudaMemcpyHostToDevice), "H2D indptr");
    fail(cudaMemcpy(d_idx, indices, sizeof(int32_t) * (size_t)nnz, cudaMemcpyHostToDevice), "H2D indices");
    fail(cudaMemcpy(d_w, w, sizeof(double) * (size_t)nnz, cudaMemcpyHostToDevice), "H2D weights");
    fail(cudaMemcpy2D(d_x, n_points * es, x, ldx * es, n_points * es, T, cudaMemcpyHostToDevice), "H2D runoff");
    if (area) fail(cudaMemcpy(d_area, area, sizeof(double) * (size_t)n_rivers, cudaMemcpyHostToDevice), "H2D area");
    if (!rc)
        rc = rr_weights_transform_dev(n_rivers, n_points, T, d_ptr, d_idx, d_w, d_x, x_is_f32, n_points, d_y, ldyd,
                                      cumulative, force_positive, d_area, nullptr);
    if (!rc) fail(cudaStreamSynchronize(nullptr), "weights kernel");
    if (!rc) fail(cudaMemcpy2D(y, ldy * 8, d_y, ldyd * 8, n_rivers * 8, T, cudaMemcpyDeviceToHost), "D2H qlateral");
    cudaFree(d_ptr); cudaFree(d_idx); cudaFree(d_w); cudaFree(d_x); cudaFree(d_y);
    if (d_area) cudaFree(d_area);
    return rc;
}
