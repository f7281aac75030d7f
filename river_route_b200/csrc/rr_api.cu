// rr_api.cu -- C-ABI entry points that touch the GPU: plan upload, route launches (device and
// host-streaming variants), ensembles, pinned host memory.  Interfaces are documented in
// include/rr_b200.h together with the reference functions they replace.
#include <cuda_runtime.h>

#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <functional>
#include <string>
#include <thread>
#include <vector>

#include "rr_route.cuh"

cudaError_t rr_launch_wavefront(int mode, const rr_route_params &P, int grid, int block, cudaStream_t stream);
int rr_wavefront_occupancy(int mode, int block);
// rr_direct.cu: the pipeline of level-sorted plans with one substep per row
cudaError_t rr_launch_direct(int mode, int max_deg, const rr_route_params &P, int grid, cudaStream_t stream, int sentinel);
int rr_direct_occupancy(int mode, int max_deg);
int rr_stage_in(const void *src, int src_f32, int64_t lds, double *lat_w, double *out_w, const int32_t *inv, int64_t n, int64_t T,
                int64_t tile_rows, int64_t n_blocks, int64_t hw_cut, const double *c3, const double *c4,
                const double *q_init, double *q_final, int sm_count, cudaStream_t stream);
int rr_stage_out_unit(const double *out_w, const double *lat, int64_t ldl, void *dst, int dst_f32, int64_t ldd, const int32_t *inv,
                      const int32_t *subset, int64_t n_out, int64_t T, int64_t tile_rows, int64_t n_blocks, int64_t hw_slots,
                      cudaStream_t stream);
int rr_unit_state_to_user(const double *qs_w, const double *qf_w, const int32_t *inv, int64_t n, int64_t hw_slots, int last,
                          const double *lat_last, double *q_state, double *q_full, cudaStream_t stream);
int rr_fill_sentinel(double *out_w, const int32_t *narrow_blocks, int64_t n_narrow, int64_t first_block, int64_t n_blocks,
                     int64_t n_tiles, int64_t pitch, cudaStream_t stream);
int rr_stage_out_sub(const double *out_w, void *dst, int dst_f32, int64_t ldd, const int32_t *inv, const int32_t *subset,
                     int64_t n_out, int64_t T, int64_t tile_rows, int64_t pitch, int64_t n_blocks, int K, cudaStream_t stream);
int rr_stage_out(const double *out_w, void *dst, int dst_f32, int64_t ldd, const int32_t *inv, const int32_t *subset,
                 int64_t n_out, int64_t T, int64_t tile_rows, int64_t n_blocks, cudaStream_t stream);

static thread_local int64_t g_launches = 0;
extern "C" int64_t rr_launch_count(int reset) {
    const int64_t v = g_launches;
    if (reset) g_launches = 0;
    return v;
}
void rr_count_launch(int64_t k) { g_launches += k; }

// Optional per-kernel timing with CUDA events on the launching stream (bench.py's roofline numbers).
struct rr_timed { int cls; cudaEvent_t a, b; };
static thread_local bool g_timing = false;
static thread_local std::vector<rr_timed> g_timed;
extern "C" int rr_timing_enable(int on) { g_timing = on != 0; return 0; }
struct rr_timer {
    rr_timed t{};
    bool on;
    cudaStream_t s;
    rr_timer(int cls, cudaStream_t stream) : on(g_timing), s(stream) {
        if (!on) return;
        t.cls = cls;
        cudaEventCreate(&t.a);
        cudaEventCreate(&t.b);
        cudaEventRecord(t.a, s);
    }
    ~rr_timer() {
        if (!on) return;
        cudaEventRecord(t.b, s);
        g_timed.push_back(t);
    }
};
extern "C" int rr_timing_read(double *ms, int64_t *counts, int reset) {
    for (int k = 0; k < 4; ++k) { ms[k] = 0.0; counts[k] = 0; }
    for (auto &t : g_timed) {
        cudaEventSynchronize(t.b);
        float e = 0.f;
        cudaEventElapsedTime(&e, t.a, t.b);
        ms[t.cls & 3] += e;
        counts[t.cls & 3]++;
    }
    if (reset) {
        for (auto &t : g_timed) { cudaEventDestroy(t.a); cudaEventDestroy(t.b); }
        g_timed.clear();
    }
    return 0;
}

#define CK(call)                                                                                   \
    do {                                                                                           \
        cudaError_t e_ = (call);                                                                   \
        if (e_ != cudaSuccess) {                                                                   \
            rr_set_error(std::string(#call) + ": " + cudaGetErrorString(e_));                      \
            return 200;                                                                            \
        }                                                                                          \
    } while (0)

extern "C" int rr_cuda_available(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
    return n > 0 ? 1 : 0;
}

struct rr_device_state {
    int device = 0, sm_count = 0;
    // plan arrays
    int32_t *up_ptr = nullptr, *up_idx = nullptr, *slot_src = nullptr, *export_id = nullptr;
    int32_t *dep_ptr = nullptr, *dep_idx = nullptr, *down = nullptr, *exp_ro = nullptr, *edge_ro = nullptr;
    uint8_t *skew = nullptr;
    rr_blk_meta *meta = nullptr;
    int32_t *narrow_blocks = nullptr;   // ids of the blocks of narrow levels (RR_META_NARROW)
    int64_t n_narrow = 0;
    double *coef = nullptr;  // c1|c2|c3|c4, each n
    uint64_t coeff_version = 0;
    // launch scratch
    int64_t sched_budget_rows = -1;
    rr_schedule sched;
    struct key_table { int64_t n_tiles = -1, first_block = 0, n_items = 0; int32_t delta = 0; int32_t *dev = nullptr; size_t cap = 0; uint64_t used = 0; };   // ticket -> (block, tile)
    key_table keys[4];
    uint64_t key_clock = 0;
    double *raw = nullptr;
    size_t raw_bytes = 0;
    int32_t *done = nullptr;
    size_t done_bytes = 0;
    unsigned long long *ticket = nullptr, *prof = nullptr;
    int occ[3] = {0, 0, 0}, occ_direct[3] = {0, 0, 0};
    // host streaming path
    cudaStream_t s_comp = nullptr, s_in = nullptr, s_out = nullptr;
    cudaEvent_t ev_in[2] = {nullptr, nullptr}, ev_comp[2] = {nullptr, nullptr}, ev_out[2] = {nullptr, nullptr};
    void *s_inb[2] = {nullptr, nullptr}, *s_outb[2] = {nullptr, nullptr};   // double-buffered chunk input / output
    size_t s_inb_cap[2] = {0, 0}, s_outb_cap[2] = {0, 0};                     // bytes
    int32_t *out_subset = nullptr;                                            // device copy of rr_plan::out_subset
    uint64_t out_subset_version = 0;
    void *h_inb[2] = {nullptr, nullptr}, *h_outb[2] = {nullptr, nullptr};   // pinned bounce buffers for pageable callers
    size_t h_inb_cap[2] = {0, 0}, h_outb_cap[2] = {0, 0};
    double *s_lat = nullptr, *s_conv = nullptr, *s_route = nullptr;           // compute-stream scratch of one chunk
    size_t s_lat_cap = 0, s_conv_cap = 0, s_route_cap = 0;
    double *d_q = nullptr, *d_qfull = nullptr;
    double *ens_q = nullptr;                                                   // ensemble calls: [q_init][mean][member states]
    size_t ens_q_cap = 0;
    void *ens_peak = nullptr;                                                  // ensemble statistics: running peaks, [S][ld] fp64 | [S][ld] int32
    size_t ens_peak_cap = 0;
    double *thr = nullptr;                                                     // device copy of rr_plan::thr
    uint64_t thr_version = 0;
    // renumbered plans: user -> working index and scratch in the working order
    int32_t *inv = nullptr;
    double *p_lat = nullptr, *p_out = nullptr, *p_q = nullptr;
    size_t p_lat_cap = 0, p_out_cap = 0, p_q_cap = 0;   // bytes
    size_t bytes = 0;
};

template <typename T>
static int upload(T **dst, const std::vector<T> &src, size_t &bytes) {
    const size_t nb = std::max<size_t>(src.size(), 1) * sizeof(T);
    CK(cudaMalloc((void **)dst, nb));
    if (!src.empty()) CK(cudaMemcpy(*dst, src.data(), src.size() * sizeof(T), cudaMemcpyHostToDevice));
    bytes += nb;
    return 0;
}

// Device / pinned host buffers that only grow (`cap` and `need` in bytes); growing waits for the device first, since
// earlier work may still use the old buffer.
static int grow_device(void **buf, size_t *cap, size_t need, bool zero = false) {
    if (need <= *cap) return 0;
    CK(cudaDeviceSynchronize());
    if (*buf) CK(cudaFree(*buf));
    *buf = nullptr; *cap = 0;
    CK(cudaMalloc(buf, need));
    if (zero) CK(cudaMemset(*buf, 0, need));
    *cap = need;
    return 0;
}
static int grow_pinned(void **buf, size_t *cap, size_t need) {
    if (need <= *cap) return 0;
    CK(cudaDeviceSynchronize());
    if (*buf) CK(cudaFreeHost(*buf));
    *buf = nullptr; *cap = 0;
    CK(cudaHostAlloc(buf, need, cudaHostAllocDefault));
    *cap = need;
    return 0;
}

static int ensure_device(rr_plan *p) {
    if (!rr_cuda_available()) {
        rr_set_error("no CUDA device available: librr_b200 has no CPU fallback");
        return 201;
    }
    if (p->dev) { CK(cudaSetDevice(p->dev->device)); }
    else {
        rr_device_state *d = new rr_device_state();
        p->dev = d;
        if (p->opts.device >= 0) CK(cudaSetDevice(p->opts.device));
        CK(cudaGetDevice(&d->device));
        CK(cudaDeviceGetAttribute(&d->sm_count, cudaDevAttrMultiProcessorCount, d->device));
        int rc = 0;
        rc |= upload(&d->up_ptr, p->up_ptr, d->bytes);
        rc |= upload(&d->up_idx, p->up_idx, d->bytes);
        rc |= upload(&d->slot_src, p->slot_src, d->bytes);
        rc |= upload(&d->export_id, p->export_id, d->bytes);
        rc |= upload(&d->dep_ptr, p->dep_ptr, d->bytes);
        rc |= upload(&d->dep_idx, p->dep_idx, d->bytes);
        rc |= upload(&d->down, p->down, d->bytes);
        rc |= upload(&d->skew, p->skew, d->bytes);
        rc |= upload(&d->meta, p->meta, d->bytes);
        if (!p->inv.empty()) rc |= upload(&d->inv, p->inv, d->bytes);
        {
            std::vector<int32_t> nb;
            for (int64_t b = 0; b < p->n_blocks; ++b) if (p->meta[b].int_mask & RR_META_NARROW) nb.push_back((int32_t)b);
            d->n_narrow = (int64_t)nb.size();
            rc |= upload(&d->narrow_blocks, nb, d->bytes);
        }
        if (rc) return rc;
        CK(cudaMalloc((void **)&d->coef, sizeof(double) * 4 * (size_t)p->n_work));
        d->bytes += sizeof(double) * 4 * (size_t)p->n_work;
        CK(cudaMalloc((void **)&d->ticket, sizeof(unsigned long long)));
        CK(cudaMalloc((void **)&d->prof, 8 * sizeof(unsigned long long)));
        CK(cudaMemset(d->prof, 0, 8 * sizeof(unsigned long long)));
        CK(cudaStreamCreateWithFlags(&d->s_comp, cudaStreamNonBlocking));
        CK(cudaStreamCreateWithFlags(&d->s_in, cudaStreamNonBlocking));
        CK(cudaStreamCreateWithFlags(&d->s_out, cudaStreamNonBlocking));
        for (int k = 0; k < 2; ++k) {
            CK(cudaEventCreateWithFlags(&d->ev_in[k], cudaEventDisableTiming));
            CK(cudaEventCreateWithFlags(&d->ev_comp[k], cudaEventDisableTiming));
            CK(cudaEventCreateWithFlags(&d->ev_out[k], cudaEventDisableTiming));
        }
    }
    rr_device_state *d = p->dev;
    if (d->coeff_version != p->coeff_version) {
        if (p->c1.empty()) { rr_set_error("coefficients not set: call rr_plan_set_coefficients first"); return 100; }
        const size_t nb = sizeof(double) * (size_t)p->n_work;
        CK(cudaMemcpy(d->coef, p->c1.data(), nb, cudaMemcpyHostToDevice));
        CK(cudaMemcpy(d->coef + p->n_work, p->c2.data(), nb, cudaMemcpyHostToDevice));
        CK(cudaMemcpy(d->coef + 2 * p->n_work, p->c3.data(), nb, cudaMemcpyHostToDevice));
        CK(cudaMemcpy(d->coef + 3 * p->n_work, p->c4.data(), nb, cudaMemcpyHostToDevice));
        d->coeff_version = p->coeff_version;
    }
    return 0;
}

void rr_device_release(rr_plan *p) {
    rr_device_state *d = p->dev;
    if (!d) return;
    cudaSetDevice(d->device);
    cudaDeviceSynchronize();
    void *ptrs[] = {d->up_ptr, d->up_idx, d->slot_src, d->export_id, d->dep_ptr, d->dep_idx, d->down, d->exp_ro, d->edge_ro,
                    d->skew, d->meta, d->narrow_blocks, d->coef, d->raw, d->done, d->ticket, d->prof,
                    d->s_inb[0], d->s_inb[1], d->s_outb[0], d->s_outb[1], d->s_lat, d->s_conv, d->s_route, d->d_q, d->d_qfull,
                    d->inv, d->p_lat, d->p_out, d->p_q, d->out_subset, d->ens_q, d->ens_peak, d->thr};
    for (void *q : ptrs)
        if (q) cudaFree(q);
    for (auto &k : d->keys) if (k.dev) cudaFree(k.dev);
    for (int k = 0; k < 2; ++k) {
        if (d->h_inb[k]) cudaFreeHost(d->h_inb[k]);
        if (d->h_outb[k]) cudaFreeHost(d->h_outb[k]);
    }
    if (d->s_comp) cudaStreamDestroy(d->s_comp);
    if (d->s_in) cudaStreamDestroy(d->s_in);
    if (d->s_out) cudaStreamDestroy(d->s_out);
    for (int k = 0; k < 2; ++k) {
        if (d->ev_in[k]) cudaEventDestroy(d->ev_in[k]);
        if (d->ev_comp[k]) cudaEventDestroy(d->ev_comp[k]);
        if (d->ev_out[k]) cudaEventDestroy(d->ev_out[k]);
    }
    delete d;
    p->dev = nullptr;
}

// One kernel launch == one reference call (or one time chunk of it).
// Rows of one work item for a call of T rows with K substeps per row (aims at `time_tile` substeps per item).
// With an automatic tile the length is chosen per call from a two-term cost model: streaming time of the call
// (longer tiles amortise the per-item setup) against the dependency critical path of one launch,
// (block levels + tiles) x item latency (shorter tiles shorten every hop).  Small per-GPU networks -- strong
// scaling over many GPUs -- are latency bound and get shorter tiles.
static int64_t tile_rows_for(const rr_plan *p, int64_t T, int64_t K) {
    int64_t tile = p->opts.time_tile;
    if (p->auto_tile) {
        double best = 1e300;
        for (int64_t cand : {64, 32, 16}) {
            const double overhead = cand == 64 ? 1.0 : (cand == 32 ? 1.18 : 1.6);
            const double stream_us = (double)p->n * (double)T * (double)K * 33.0 / 4.6e6 * overhead;   // bytes / (B/us)
            const double rows = (double)std::max<int64_t>(1, cand / K);
            const double n_tiles = std::ceil((double)T / rows);
            // measured with the kernel's cycle counters: ~12 us of per-item setup + ~0.35 us per substep
            const double critical_us = ((double)p->max_level + n_tiles) * (12.0 + 0.35 * rows * (double)K);
            const double est = std::max(stream_us, critical_us) + 0.3 * std::min(stream_us, critical_us);
            if (est < best) { best = est; tile = cand; }
        }
    }
    return std::max<int64_t>(1, std::min<int64_t>(T, tile / K));
}

#ifdef RR_TRACE
// tools/trace_chain.py: device buffer [block][group][event][2] the direct kernel stamps (trace builds only)
static unsigned long long *g_rr_trace = nullptr;
extern "C" void rr_trace_set(void *dev_buffer) { g_rr_trace = (unsigned long long *)dev_buffer; }
#endif
static bool pipeline_ok(const rr_plan *p, int mode, int64_t K);
extern "C" int64_t rr_plan_tile_rows(const rr_plan *p, int64_t T, int64_t substeps) {
    if (!p || T <= 0 || substeps <= 0) return 0;
    if (pipeline_ok(p, RR_MODE_RAPID, substeps)) {
        if (substeps > 1) return std::max<int64_t>(1, std::min<int64_t>(p->opts.time_tile / substeps, T));
        return std::min<int64_t>(p->opts.time_tile / RR_FLAG_ROWS * RR_FLAG_ROWS, (T + RR_FLAG_ROWS - 1) / RR_FLAG_ROWS * RR_FLAG_ROWS);
    }
    return tile_rows_for(p, T, substeps);
}

static int launch_route(rr_plan *p, int mode, int n_members, const double *q_init, const double *const *lateral,
                        int64_t ldl, double *const *out, int64_t ldo, double *const *q_state, double *const *q_full,
                        int64_t T, int64_t K, int first_call, int last_call, cudaStream_t stream, int tile_major = 0,
                        int out_layout = 0, int direct = 0, int64_t rows_in = 0, int64_t first_block = 0, int pipeline = 0,
                        int64_t q_init_stride = 0, const double *qf_init = nullptr, int64_t hw_slots = 0) {
    if (mode < 0 || mode > 2) { rr_set_error("unknown router mode"); return 100; }
    if (T <= 0 || K <= 0 || T > 0x7fffffff || K > 0x7fffffff) { rr_set_error("T and substeps must be positive"); return 100; }
    if (n_members < 1 || n_members > RR_MAX_MEMBERS) { rr_set_error("n_members must be in [1, 64]"); return 100; }
    if (mode == RR_MODE_RAPID && !p->have_c4) { rr_set_error("RapidMuskingum needs c4_dt coefficients"); return 100; }
    if (!tile_major && mode != RR_MODE_MUSKINGUM && ldl < p->n) { rr_set_error("lateral leading dimension smaller than n"); return 100; }
    if (!tile_major && ldo < p->n) { rr_set_error("output leading dimension smaller than n"); return 100; }
    int rc = ensure_device(p);
    if (rc) return rc;
    rr_device_state *d = p->dev;

    // tile geometry: aim for `time_tile` routing substeps per work item
    const int64_t rows = rows_in > 0 ? rows_in : tile_rows_for(p, T, K);
    const int64_t n_tiles = (T + rows - 1) / rows;
    // row pitch of the exchange buffer: [14] q_full carry, [15] carry, [16+s] substeps (rr_route.cu); sized for the
    // plan's nominal tile so that short calls (the last chunk of a stream) reuse the same rings
    const int64_t nominal = std::max<int64_t>(std::max<int64_t>(1, p->opts.time_tile / K) * K, rows * K);
    const int64_t pitch = 16 + ((nominal + 15) / 16) * 16;
    const int64_t budget_rows = std::max<int64_t>(1, p->opts.raw_budget_bytes / (int64_t)(pitch * sizeof(double) * n_members));
    if ((double)n_tiles * (double)(p->max_level + 1) > 2e9) {
        rr_set_error("network too deep for the ticket scheduler at this tile size; raise time_tile");
        return 100;
    }
    if (d->sched_budget_rows != budget_rows) {
        // exchange rings depend on the network and the budget only; built once and kept on the device
        rr_build_rings(*p, p->opts.tile_stride, budget_rows, d->sched);
        CK(cudaDeviceSynchronize());   // an earlier launch may still be reading the old tables
        if (!d->exp_ro) {
            CK(cudaMalloc((void **)&d->exp_ro, std::max<size_t>(d->sched.exp_ro.size(), 2) * sizeof(int32_t)));
            CK(cudaMalloc((void **)&d->edge_ro, std::max<size_t>(d->sched.edge_ro.size(), 2) * sizeof(int32_t)));
        }
        if (!d->sched.exp_ro.empty())
            CK(cudaMemcpy(d->exp_ro, d->sched.exp_ro.data(), d->sched.exp_ro.size() * sizeof(int32_t), cudaMemcpyHostToDevice));
        if (!d->sched.edge_ro.empty())
            CK(cudaMemcpy(d->edge_ro, d->sched.edge_ro.data(), d->sched.edge_ro.size() * sizeof(int32_t), cudaMemcpyHostToDevice));
        d->sched_budget_rows = budget_rows;
        for (auto &k : d->keys) k.n_tiles = -1;
    }
    // ticket keys per call length: a few tables are cached (the streaming path alternates between the
    // full chunk and the last, shorter one)
    // Ticket-key distance between consecutive tiles of a block.  Ring-exchange launches take it from the ring sizing.
    // The pipeline has no rings; its natural value is the number of levels a dependency chain advances while one block
    // works through a tile: narrow levels pass results on every 16-row group, so one level costs about one group and a
    // tile about gpt of them.  With that stride the fronts of all tiles in flight share a ticket key and fit the
    // resident warps; with stride 1 they spread over 3 x n_tiles keys and most of them wait for a warp (C2: the 3000-level
    // stem ran 23 tiles in batches of ~7).
    const int32_t delta_use = pipeline ? (p->opts.tile_stride > 0 ? p->opts.tile_stride : (int32_t)((rows * K + RR_FLAG_ROWS - 1) / RR_FLAG_ROWS))
                                       : d->sched.delta;
    rr_device_state::key_table *kt = nullptr;
    for (auto &k : d->keys) if (k.n_tiles == n_tiles && k.first_block == first_block && k.delta == delta_use) kt = &k;
    if (!kt) {
        kt = &d->keys[0];
        for (auto &k : d->keys) if (k.used < kt->used) kt = &k;
        rr_schedule tmp;
        tmp.delta = delta_use;
        rr_build_keys(*p, n_tiles, tmp, first_block);
        std::vector<int32_t> items;
        rr_build_items(*p, n_tiles, tmp, items, first_block);
        CK(cudaDeviceSynchronize());
        if (items.size() > kt->cap) {
            if (kt->dev) CK(cudaFree(kt->dev));
            kt->dev = nullptr; kt->cap = 0;
            CK(cudaMalloc((void **)&kt->dev, std::max<size_t>(items.size(), 4) * sizeof(int32_t)));
            kt->cap = items.size();
        }
        CK(cudaMemcpy(kt->dev, items.data(), items.size() * sizeof(int32_t), cudaMemcpyHostToDevice));
        kt->n_tiles = n_tiles; kt->first_block = first_block; kt->delta = delta_use; kt->n_items = tmp.n_items;
    }
    kt->used = ++d->key_clock;
    // one spare row: the kernel prefetches a few lines past the row it is reading
    // direct exchange needs no rings: the working discharge array is the exchange buffer
    const size_t raw_need = direct ? (size_t)pitch * sizeof(double)
                                   : ((size_t)n_members * (size_t)d->sched.raw_rows + 1) * pitch * sizeof(double);
    if ((rc = grow_device((void **)&d->raw, &d->raw_bytes, raw_need))) return rc;
    const size_t done_need = (size_t)n_members * p->n_blocks;
    if ((rc = grow_device((void **)&d->done, &d->done_bytes, done_need * sizeof(int32_t)))) return rc;

    rr_route_params P;
    std::memset(&P, 0, sizeof(P));
    P.n = p->n_work; P.n_blocks = (int32_t)p->n_blocks; P.max_level = p->max_level;
    P.up_ptr = d->up_ptr; P.up_idx = d->up_idx; P.slot_src = d->slot_src; P.skew = d->skew;
    P.export_id = d->export_id; P.meta = d->meta;
    P.dep_ptr = d->dep_ptr; P.dep_idx = d->dep_idx; P.down = d->down;
    P.exp_ro = d->exp_ro; P.edge_ro = d->edge_ro; P.raw_rows = d->sched.raw_rows;
    P.c1 = d->coef; P.c2 = d->coef + p->n_work; P.c3 = d->coef + 2 * p->n_work; P.c4 = d->coef + 3 * p->n_work;
    P.items = reinterpret_cast<const int4 *>(kt->dev); P.n_items = kt->n_items;
    P.delta = delta_use; P.n_tiles = (int32_t)n_tiles;
    P.T = (int32_t)T; P.K = (int32_t)K; P.tile_rows = (int32_t)rows;
    P.raw_pitch = (int32_t)pitch; P.n_members = n_members; P.first_call = first_call; P.last_call = last_call;
    P.ldl = ldl; P.ldo = ldo;
    P.raw = d->raw; P.done = d->done; P.ticket = d->ticket; P.prof = d->prof;
#ifdef RR_TRACE
    P.prof = g_rr_trace;
#endif
 P.q_init = q_init; P.q_init_stride = q_init_stride;
    P.qf_init = qf_init; P.hw_slots = hw_slots;
    for (int m = 0; m < n_members; ++m) {
        P.lateral[m] = lateral ? lateral[m] : nullptr;
        P.out[m] = out[m];
        P.q_state[m] = q_state[m];
        P.q_full[m] = q_full ? q_full[m] : nullptr;
    }
    P.ticket_batch = 1;   // larger batches were measured slower: neighbouring blocks should run concurrently
    CK(cudaMemsetAsync(d->done, 0, done_need * sizeof(int32_t), stream));
    // blocks the staging kernel has routed already (whole-headwater blocks) count as finished for every tile
    for (int m = 0; m < n_members && first_block > 0; ++m)
        CK(cudaMemsetAsync(d->done + (size_t)m * p->n_blocks, 0x3f, (size_t)first_block * sizeof(int32_t), stream));
    CK(cudaMemsetAsync(d->ticket, 0, sizeof(unsigned long long), stream));
    int block = p->opts.threads_per_cta;
    P.tile_major = tile_major;
    P.out_layout = out_layout;
    P.direct = direct;
    P.tile_pitch = (int32_t)((rows + 3) & ~(int64_t)3);
    P.gpt = (int32_t)((rows + RR_FLAG_ROWS - 1) / RR_FLAG_ROWS);
    P.lat_pitch = P.tile_pitch;
    if (pipeline) {   // tiles hold rows x K routing substeps, padded to whole 16-entry groups
        P.gpt = (int32_t)((rows * K + RR_FLAG_ROWS - 1) / RR_FLAG_ROWS);
        P.tile_pitch = P.gpt * RR_FLAG_ROWS;
        if (K == 1) P.lat_pitch = P.tile_pitch;
    }
    // stress-test hooks (tests/test_gpu_stress.py): fewer persistent CTAs than the device holds, and pseudo-random delays
    // around the flag operations -- any grid size and any timing must give the same bits
    int64_t grid_cap = 0;
    if (const char *env = getenv("RR_GRID_CTAS")) grid_cap = std::max(1, atoi(env));
    if (const char *env = getenv("RR_JITTER")) P.jitter = std::max(0, atoi(env));
    P.spin_ns = 32;
    if (const char *env = getenv("RR_PROG_SPIN_NS")) P.spin_ns = std::max(0, atoi(env));
    if (pipeline) {
        // Small networks (at most RR_SENTINEL_MAX_BLOCKS blocks: every level is narrow and the launch is bound by the latency of
        // the dependency chain) hand results over through the "not written yet" pattern (rr_direct.cu, narrow_item): arm the
        // tiles.  Larger networks keep per-group progress flags on their narrow levels: there the pattern costs bandwidth --
        // the fill, and DRAM reads of armed lines by consumers that arrive early -- which the bandwidth-bound part of the
        // launch pays for (C4: wavefront 6.45 ms with flags, 6.85 - 7.6 ms with the pattern on levels below 256 - 4096
        // blocks; the N = 8 shard shape 6.7 vs 7.2 - 8.3 ms), while C1 (1674 blocks) runs in 3.55 ms instead of 4.2 ms.
        int sentinel = (mode != RR_MODE_UNIT && p->n_blocks <= RR_SENTINEL_MAX_BLOCKS) ? 1 : 0;
        if (const char *env = getenv("RR_SENTINEL")) sentinel = (mode != RR_MODE_UNIT && atoi(env) != 0) ? 1 : 0;   // tests, measurements
        P.poll_lo = (int32_t)first_block;
        P.spin_ns = sentinel ? 0 : 32;   // the pattern is watched through one word per warp: no need to sleep between polls
        if (const char *env = getenv("RR_PROG_SPIN_NS")) P.spin_ns = std::max(0, atoi(env));
        if (sentinel)
            for (int m = 0; m < n_members; ++m) {
                rr_timer tm(3, stream);
                if ((rc = rr_fill_sentinel(out[m], d->narrow_blocks, d->n_narrow, first_block, p->n_blocks, n_tiles, P.tile_pitch, stream))) return rc;
            }
        // rr_direct.cu: done[] counts 16-row groups; 8 warps per CTA share 32 KB of output staging
        if (!d->occ_direct[mode]) {
            d->occ_direct[mode] = rr_direct_occupancy(mode, p->max_deg);
            if (d->occ_direct[mode] <= 0) { rr_set_error("occupancy query failed for the direct wavefront kernel"); return 200; }
        }
        const int64_t total = kt->n_items * n_members;
        int64_t g = (int64_t)d->sm_count * d->occ_direct[mode];
        g = std::max<int64_t>(1, std::min<int64_t>(g, (total + 7) / 8));
        if (grid_cap) g = std::min<int64_t>(g, grid_cap);
        {
            rr_timer tm(0, stream);
            CK(rr_launch_direct(mode, p->max_deg, P, (int)g, stream, sentinel));
        }
        rr_count_launch(1);
        return 0;
    }
    if (tile_major == 1 && K == 1 && mode != RR_MODE_UNIT) {
        // TMA-staged kernel: 4 warps per CTA, each with [tile | upstream row slots | mbarrier] in shared memory
        int max_smem = 0;
        CK(cudaDeviceGetAttribute(&max_smem, cudaDevAttrMaxSharedMemoryPerBlockOptin, d->device));
        const int64_t tile_bytes = rows * RR_BLOCK * 8, row_bytes = pitch * 8 + 16;
        const int64_t slots = std::min<int64_t>(64, ((int64_t)max_smem / 4 - tile_bytes - 16 - 128) / row_bytes);
        if (slots >= 32) {
            P.row_slots = (int32_t)slots;
            P.smem_region = (int32_t)(((tile_bytes + slots * row_bytes + 16 + 127) / 128) * 128);
            block = 128;
        }
    }
    if (!d->occ[mode]) {
        d->occ[mode] = rr_wavefront_occupancy(mode, block);
        if (d->occ[mode] <= 0) { rr_set_error("occupancy query failed for the wavefront kernel"); return 200; }
    }
    const int64_t warps_per_cta = block / 32;
    const int64_t total_items = kt->n_items * n_members;
    int64_t grid = (int64_t)d->sm_count * (P.smem_region > 0 ? 1 : d->occ[mode]);
    grid = std::max<int64_t>(1, std::min<int64_t>(grid, (total_items + warps_per_cta - 1) / warps_per_cta));
    if (grid_cap) grid = std::min<int64_t>(grid, grid_cap);
    {
        rr_timer tm(0, stream);
        CK(rr_launch_wavefront(mode, P, (int)grid, block, stream));
    }
    rr_count_launch(1);
    return 0;
}

// ---------------------------------------------------------------------------------------------------
// Renumbered plans: the caller's arrays stay in params_file order; the router works on reaches sorted
// by level.  Both permutations walk the USER index (coalesced on the caller's side); reaches that are
// neighbours in the working order are same-level reaches with nearby user indices, so the scattered
// side of each copy completes whole 32-byte sectors while they are still in L2.
// ---------------------------------------------------------------------------------------------------
#define PERM_ROWS 8
// Address of working element (row t, working reach k).  tile_rows == 0: row-major with leading dimension ld;
// otherwise the tile-major layout [tile][block][row in tile][lane] the TMA-staged kernel reads with bulk copies.
__device__ __forceinline__ int64_t working_index(int64_t t, int64_t k, int64_t ld, int64_t tile_rows, int64_t n_blocks,
                                                 int layout) {
    if (layout == 0) return t * ld + k;
    const int64_t j = t / tile_rows, r = t - j * tile_rows;
    if (layout == 1) return ((j * n_blocks + (k >> 5)) * tile_rows + r) * RR_BLOCK + (k & 31);
    const int64_t pitch = (tile_rows + 3) & ~(int64_t)3;
    if (layout == 3) return (((j * n_blocks + (k >> 5)) * (pitch >> 2) + (r >> 2)) * RR_BLOCK + (k & 31)) * 4 + (r & 3);
    return ((j * n_blocks + (k >> 5)) * RR_BLOCK + (k & 31)) * pitch + r;
}
__device__ __forceinline__ void st256(double *p, double a, double b, double c, double d) {
    asm volatile("st.global.v4.f64 [%0], {%1, %2, %3, %4};" ::"l"(p), "d"(a), "d"(b), "d"(c), "d"(d) : "memory");
}
__device__ __forceinline__ void ld256(const double *p, double &a, double &b, double &c, double &d) {
    asm volatile("ld.global.v4.f64 {%0, %1, %2, %3}, [%4];" : "=d"(a), "=d"(b), "=d"(c), "=d"(d) : "l"(p) : "memory");
}
template <int ROWS>
__global__ void __launch_bounds__(256) permute_to_working(const double *__restrict__ src, int64_t lds, double *__restrict__ dst,
                                                          int64_t ldd, const int32_t *__restrict__ inv, int64_t n, int64_t T,
                                                          int64_t tile_rows, int64_t n_blocks, int layout) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const int64_t k = __ldg(inv + i);
    const int64_t t0 = (int64_t)blockIdx.y * ROWS;
    double v[ROWS];
#pragma unroll
    for (int r = 0; r < ROWS; ++r) v[r] = (t0 + r < T) ? __ldg(src + (t0 + r) * lds + i) : 0.0;
    if (layout == 2 && (tile_rows % ROWS) == 0) {
        // the ROWS rows of this reach are contiguous in its tile: whole-sector (ROWS = 16: whole-line) stores
        double *q = dst + working_index(t0, k, ldd, tile_rows, n_blocks, 2);
#pragma unroll
        for (int r = 0; r < ROWS; r += 4) st256(q + r, v[r], v[r + 1], v[r + 2], v[r + 3]);
        return;
    }
    if (layout == 3 && (tile_rows % ROWS) == 0) {
        // groups of 4 rows are one sector each, 1 KB apart (the 32 lanes of the block sit in between)
        double *q = dst + working_index(t0, k, ldd, tile_rows, n_blocks, 3);
#pragma unroll
        for (int r = 0; r < ROWS; r += 4) st256(q + (size_t)(r >> 2) * (RR_BLOCK * 4), v[r], v[r + 1], v[r + 2], v[r + 3]);
        return;
    }
#pragma unroll
    for (int r = 0; r < ROWS; ++r)
        if (t0 + r < T) dst[working_index(t0 + r, k, ldd, tile_rows, n_blocks, layout)] = v[r];
}
template <int ROWS>
__global__ void __launch_bounds__(256) permute_to_user(const double *__restrict__ src, int64_t lds, double *__restrict__ dst,
                                                       int64_t ldd, const int32_t *__restrict__ inv, int64_t n, int64_t T,
                                                       int64_t tile_rows, int64_t n_blocks, int layout, int clamp) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const int64_t k = __ldg(inv + i);
    const int64_t t0 = (int64_t)blockIdx.y * ROWS;
    double v[ROWS];
    if (layout == 2 && (tile_rows % ROWS) == 0) {
        const double *q = src + working_index(t0, k, lds, tile_rows, n_blocks, 2);
#pragma unroll
        for (int r = 0; r < ROWS; r += 4) ld256(q + r, v[r], v[r + 1], v[r + 2], v[r + 3]);
    } else {
#pragma unroll
        for (int r = 0; r < ROWS; ++r)
            v[r] = (t0 + r < T) ? src[working_index(t0 + r, k, lds, tile_rows, n_blocks, layout)] : 0.0;
    }
    if (clamp) {   // direct exchange: the working array holds the raw series; the reference's clamp (_numba_kernels.py:44-46, :82-84)
#pragma unroll
        for (int r = 0; r < ROWS; ++r) v[r] = v[r] > 0.0 ? v[r] : 0.0;
    }
#pragma unroll
    for (int r = 0; r < ROWS; ++r)
        if (t0 + r < T) dst[(t0 + r) * ldd + i] = v[r];
}
static int permute(bool to_working, const double *src, int64_t lds, double *dst, int64_t ldd, const int32_t *inv,
                   int64_t n, int64_t T, cudaStream_t stream, int64_t tile_rows = 0, int64_t n_blocks = 0, int layout = 0,
                   int clamp = 0) {
    rr_timer tm(to_working ? 1 : 2, stream);
    const unsigned gx = (unsigned)((n + 255) / 256);
    if (to_working && (layout == 2 || layout == 3) && (tile_rows % 16) == 0) {
        dim3 grid(gx, (unsigned)((T + 15) / 16));
        permute_to_working<16><<<grid, 256, 0, stream>>>(src, lds, dst, ldd, inv, n, T, tile_rows, n_blocks, layout);
    } else if (to_working) {
        dim3 grid(gx, (unsigned)((T + PERM_ROWS - 1) / PERM_ROWS));
        permute_to_working<PERM_ROWS><<<grid, 256, 0, stream>>>(src, lds, dst, ldd, inv, n, T, tile_rows, n_blocks, layout);
    } else if (layout == 2 && (tile_rows % 16) == 0) {
        dim3 grid(gx, (unsigned)((T + 15) / 16));
        permute_to_user<16><<<grid, 256, 0, stream>>>(src, lds, dst, ldd, inv, n, T, tile_rows, n_blocks, layout, clamp);
    } else {
        dim3 grid(gx, (unsigned)((T + PERM_ROWS - 1) / PERM_ROWS));
        permute_to_user<PERM_ROWS><<<grid, 256, 0, stream>>>(src, lds, dst, ldd, inv, n, T, tile_rows, n_blocks, layout, clamp);
    }
    CK(cudaGetLastError());
    rr_count_launch(1);
    return 0;
}
// Where a call's discharge goes when the caller wants the router loop's tail fused into the last device pass:
// float32 cast (TransformMuskingum.py:146) and / or an output subset, written straight from the working tiles.
struct rr_out_spec {
    void *dst = nullptr;
    int f32 = 0;
    int64_t ld = 0;
    const int32_t *subset = nullptr;   // device pointer; nullptr = all segments
    int64_t n_out = 0;
};

// The rr_direct.cu pipeline serves level-sorted plans whose blocks are all fast-path eligible, one substep per row,
// tile lengths that are whole 16-row groups (all three routers).
static bool pipeline_ok(const rr_plan *p, int mode, int64_t K) {
    const int st = p->opts.staging;
    // several routing substeps per row: RapidMuskingum / Muskingum, at least one whole row per tile.  Opt-in
    // (staging='direct' / 'direct-nohw'): on C1 with 12 substeps the substep-tile pipeline measured 38.4 ms against 30.8 ms
    // for the ring path (stage_out_sub re-reads all K substeps of every row; the wavefront itself takes the same time)
    if (K > 1 && (mode == RR_MODE_UNIT || K > p->opts.time_tile || !(st == 6 || st == 7))) return false;
    return !p->perm.empty() && p->all_fast && (st == 0 || st == 6 || st == 7) && (p->opts.time_tile % RR_FLAG_ROWS) == 0;
}

// Route with all arrays in the caller's (params_file) order, whatever order the plan works in.
static int route_any(rr_plan *p, int mode, int n_members, const double *q_init, const double *const *lateral,
                     int64_t ldl, double *const *out, int64_t ldo, double *const *q_state, double *const *q_full,
                     int64_t T, int64_t K, int first_call, int last_call, cudaStream_t stream,
                     const rr_out_spec *spec = nullptr /* one per member */, int lat_f32 = 0) {
    if (lat_f32 && !(pipeline_ok(p, mode, K) && K == 1 && !p->perm.empty())) { rr_set_error("internal: float32 lateral inflows need the direct pipeline"); return 101; }
    if (p->perm.empty()) {
        if (spec) { rr_set_error("internal: fused output needs a level-sorted plan"); return 101; }
        return launch_route(p, mode, n_members, q_init, lateral, ldl, out, ldo, q_state, q_full, T, K, first_call,
                            last_call, stream);
    }
    int rc = ensure_device(p);
    if (rc) return rc;
    rr_device_state *d = p->dev;
    const int64_t n = p->n, ldp = ((p->n_work + 31) / 32) * 32;   // user segments; slots per working row
    const bool has_lat = mode != RR_MODE_MUSKINGUM;
    const bool unit = mode == RR_MODE_UNIT;
    if (n_members < 1 || n_members > RR_MAX_MEMBERS) { rr_set_error("n_members must be in [1, 64]"); return 100; }
    if (T <= 0 || K <= 0) { rr_set_error("T and substeps must be positive"); return 100; }
    const bool pipeline = pipeline_ok(p, mode, K);
    if (spec && !pipeline) { rr_set_error("internal: fused output is a feature of the direct pipeline"); return 101; }
    // working arrays: row-major (staging 1, substeps), [tile][block][row][lane] for the TMA-staged
    // kernel (3), [tile][block][lane][row] otherwise (register path: whole-sector accesses everywhere)
    const bool tiled = pipeline || (K == 1 && p->opts.staging != 1 && !(unit && p->opts.staging == 3));
    // lateral: reach-major tiles (whole-sector scatter in the permute, 256-bit loads in the kernel); discharge:
    // row-major tiles (coalesced row stores in the kernel, sector-sharing gathers in the permute) -- measured best
    const int layout = !tiled ? 0 : (p->opts.staging == 3 ? 1 : (p->opts.staging == 5 ? 3 : 2));
    // "direct exchange": the working discharge array (reach-major tiles, raw values) is the exchange buffer
    // (default for level-sorted plans with one substep per row; staging 2 / 4 / 5 keep the exchange rings)
    const bool direct = tiled && (!unit || pipeline) && (p->opts.staging == 6 || p->opts.staging == 0 || p->opts.staging == 7);
    const int out_layout = !tiled ? 0 : ((p->opts.staging == 4 || direct) ? 2 : 1);
    int64_t trows = tiled ? tile_rows_for(p, T, K) : 0;
    // the pipeline's tiles are whole 16-row groups (short calls get one padded tile)
    // (the per-call tile model of tile_rows_for does not apply: narrow levels hand results on every 16 rows whatever
    // the tile length, so long tiles cost no latency and save per-item setup)
    if (pipeline) trows = std::min<int64_t>(p->opts.time_tile / RR_FLAG_ROWS * RR_FLAG_ROWS, (T + RR_FLAG_ROWS - 1) / RR_FLAG_ROWS * RR_FLAG_ROWS);
    // several substeps per row: a tile is as many whole rows as fit time_tile substeps; the discharge tiles hold substeps
    if (pipeline && K > 1) trows = std::max<int64_t>(1, std::min<int64_t>(p->opts.time_tile / K, T));
    const int64_t lpitch = ((trows + 3) & ~(int64_t)3);                                                  // lateral tile: rows
    const int64_t tpitch = pipeline ? (trows * K + RR_FLAG_ROWS - 1) / RR_FLAG_ROWS * RR_FLAG_ROWS : lpitch;   // discharge tile
    const int64_t n_tiles = tiled ? (T + trows - 1) / trows : 0;
    const size_t member_elems = tiled ? (size_t)n_tiles * p->n_blocks * tpitch * RR_BLOCK : (size_t)T * ldp;
    const size_t lat_elems = (pipeline && K > 1) ? (size_t)n_tiles * p->n_blocks * lpitch * RR_BLOCK : member_elems;
    // zero-filled: padding slots of level-sorted plans are routed along, keep them finite
    if (has_lat && (rc = grow_device((void **)&d->p_lat, &d->p_lat_cap, 8 * ((size_t)n_members * lat_elems + 64), true))) return rc;
    if ((rc = grow_device((void **)&d->p_out, &d->p_out_cap, 8 * ((size_t)n_members * member_elems + 64), true))) return rc;
    // state scratch: [start-of-call state: one shared, or one per member on continued calls][member states][member q_full]
    //                [start-of-call q_full of continued UnitMuskingum pipeline calls]
    if ((rc = grow_device((void **)&d->p_q, &d->p_q_cap, 8 * (size_t)(4 * n_members) * ldp, true))) return rc;
    double *w_init = d->p_q;
    double *wf_init = d->p_q + (size_t)(3 * n_members) * ldp;
    const int64_t init_stride = (direct && !first_call) ? ldp : 0;
    const bool unit_pipe = unit && pipeline;
    const double *lat_w[RR_MAX_MEMBERS];
    double *out_w[RR_MAX_MEMBERS], *qs_w[RR_MAX_MEMBERS], *qf_w[RR_MAX_MEMBERS];
    // whole blocks of headwaters are routed by the staging kernel of the pipeline (RapidMuskingum: their lateral rows
    // pass through its registers anyway); small networks keep them in the wavefront (staging 7 forces that, 6 the former)
    int64_t hw_cut = 0;
    if (pipeline && K == 1 && mode == RR_MODE_RAPID && p->opts.staging != 7 && (p->opts.staging == 6 || n >= (1 << 18)))
        hw_cut = p->lvl0_slots;   // level 0 fills whole blocks (headwaters + padding)
    if (first_call && (rc = permute(true, q_init, n, w_init, ldp, d->inv, n, 1, stream))) return rc;
    for (int m = 0; m < n_members; ++m) {
        lat_w[m] = has_lat ? d->p_lat + (size_t)m * lat_elems : nullptr;
        out_w[m] = d->p_out + (size_t)m * member_elems;
        qs_w[m] = d->p_q + (size_t)(n_members + m) * ldp;
        qf_w[m] = d->p_q + (size_t)(2 * n_members + m) * ldp;
        if (!first_call) {
            // direct exchange reads upstream start-of-call values during the launch, so the running state (which the
            // launch overwrites in place) is first copied to the shared, read-only initial-state vector
            if ((rc = permute(true, q_state[m], n, direct ? w_init + (size_t)m * ldp : qs_w[m], ldp, d->inv, n, 1, stream))) return rc;
            if (unit && (rc = permute(true, q_full[m], n, unit_pipe ? wf_init + (size_t)m * ldp : qf_w[m], ldp, d->inv, n, 1, stream))) return rc;
        }
        if (has_lat && pipeline && K == 1) {
            rr_timer tm(1, stream);
            rc = rr_stage_in(lateral[m], lat_f32, ldl, d->p_lat + (size_t)m * lat_elems, out_w[m], d->inv, n, T, trows, p->n_blocks,
                             hw_cut, d->coef + 2 * p->n_work, d->coef + 3 * p->n_work, w_init + (size_t)m * init_stride, qs_w[m],
                             d->sm_count, stream);
            if (rc) return rc;
        } else if (has_lat && (rc = permute(true, lateral[m], ldl, d->p_lat + (size_t)m * lat_elems, ldp, d->inv, n, T, stream, trows, p->n_blocks, layout))) return rc;
    }
    rc = launch_route(p, mode, n_members, w_init, has_lat ? lat_w : nullptr, ldp, out_w, ldp, qs_w, qf_w, T, K,
                      direct ? 1 : first_call, last_call, stream, layout, out_layout, direct ? 1 : 0, pipeline ? trows : 0,
                      (unit_pipe ? p->lvl0_slots : hw_cut) / RR_BLOCK, pipeline ? 1 : 0, init_stride,
                      unit_pipe ? (first_call ? w_init : wf_init) : nullptr, unit_pipe ? p->lvl0_slots : 0);
    if (rc) return rc;
    for (int m = 0; m < n_members; ++m) {
        if (unit_pipe) {
            {
                rr_timer tm(2, stream);
                if (spec) rc = rr_stage_out_unit(out_w[m], lateral[m], ldl, spec[m].dst, spec[m].f32, spec[m].ld, d->inv, spec[m].subset,
                                                 spec[m].n_out, T, trows, p->n_blocks, p->lvl0_slots, stream);
                else rc = rr_stage_out_unit(out_w[m], lateral[m], ldl, out[m], 0, ldo, d->inv, nullptr, n, T, trows, p->n_blocks,
                                            p->lvl0_slots, stream);
            }
            if (rc) return rc;
            if ((rc = rr_unit_state_to_user(qs_w[m], qf_w[m], d->inv, n, p->lvl0_slots, last_call, lateral[m] + (size_t)(T - 1) * ldl,
                                            q_state[m], q_full[m], stream))) return rc;
            continue;
        }
        if (pipeline && K > 1) {
            rr_timer tm(2, stream);
            if (spec) rc = rr_stage_out_sub(out_w[m], spec[m].dst, spec[m].f32, spec[m].ld, d->inv, spec[m].subset, spec[m].n_out, T, trows,
                                            tpitch, p->n_blocks, (int)K, stream);
            else rc = rr_stage_out_sub(out_w[m], out[m], 0, ldo, d->inv, nullptr, n, T, trows, tpitch, p->n_blocks, (int)K, stream);
            if (rc) return rc;
        } else if (pipeline) {
            rr_timer tm(2, stream);
            if (spec) rc = rr_stage_out(out_w[m], spec[m].dst, spec[m].f32, spec[m].ld, d->inv, spec[m].subset, spec[m].n_out, T, trows, p->n_blocks, stream);
            else rc = rr_stage_out(out_w[m], out[m], 0, ldo, d->inv, nullptr, n, T, trows, p->n_blocks, stream);
            if (rc) return rc;
        } else if ((rc = permute(false, out_w[m], ldp, out[m], ldo, d->inv, n, T, stream, trows, p->n_blocks, out_layout, direct ? 1 : 0))) return rc;
        if ((rc = permute(false, qs_w[m], ldp, q_state[m], n, d->inv, n, 1, stream))) return rc;
        if (unit && !(last_call) && (rc = permute(false, qf_w[m], ldp, q_full[m], n, d->inv, n, 1, stream))) return rc;
    }
    return 0;
}

extern "C" int rr_route_dev(rr_plan *p, int mode, double *q_state, double *q_full, const double *lateral,
                            int64_t ldl, double *out, int64_t ldo, int64_t T, int64_t substeps, void *stream) {
    if (!p || !q_state || !out || (mode != RR_MODE_MUSKINGUM && !lateral)) { rr_set_error("null argument"); return 100; }
    int rc = ensure_device(p);
    if (rc) return rc;
    rr_device_state *d = p->dev;
    double *qf = nullptr;
    const int router_level = (mode != RR_MODE_UNIT) || q_full == nullptr;
    if (mode == RR_MODE_UNIT) {
        if (!q_full && !d->d_qfull) CK(cudaMalloc((void **)&d->d_qfull, sizeof(double) * (size_t)p->n));
        qf = q_full ? q_full : d->d_qfull;
    }
    const double *lat1[1] = {lateral};
    double *out1[1] = {out}, *qs1[1] = {q_state}, *qf1[1] = {qf};
    return route_any(p, mode, 1, q_state, lat1, ldl, out1, ldo, qs1, qf1, T, substeps, router_level, router_level,
                     (cudaStream_t)stream);
}

extern "C" int rr_route_ensemble_dev(rr_plan *p, int mode, const double *q_init, int32_t n_members,
                                     const double *const *lateral, int64_t ldl, double *const *out, int64_t ldo,
                                     double *const *q_final, int64_t T, int64_t substeps, void *stream) {
    if (!p || !q_init || !out || !q_final || (mode != RR_MODE_MUSKINGUM && !lateral)) { rr_set_error("null argument"); return 100; }
    if (mode == RR_MODE_UNIT) { rr_set_error("ensemble launch supports Muskingum / RapidMuskingum"); return 100; }
    return route_any(p, mode, n_members, q_init, lateral, ldl, out, ldo, q_final, nullptr, T, substeps, 1, 1,
                     (cudaStream_t)stream);
}

// ---------------------------------------------------------------------------------------------------
// Device-resident weight table (+ optional unit hydrograph) of the grid-runoff path.
// ---------------------------------------------------------------------------------------------------
struct rr_transform {
    int device = 0;
    int64_t n_rivers = 0, n_points = 0, nnz = 0;
    int32_t *indptr = nullptr, *indices = nullptr;
    double *w = nullptr, *area = nullptr;
    int64_t n_ks = 0, ld_uh = 0;
    double *uh_kernel = nullptr, *uh_state = nullptr;
};

extern "C" void rr_transform_destroy(rr_transform *t) {
    if (!t) return;
    cudaSetDevice(t->device);
    cudaDeviceSynchronize();
    void *ptrs[] = {t->indptr, t->indices, t->w, t->area, t->uh_kernel, t->uh_state};
    for (void *q : ptrs)
        if (q) cudaFree(q);
    delete t;
}

extern "C" int rr_transform_create(int64_t n_rivers, int64_t n_points, const int32_t *indptr, const int32_t *indices,
                                   const double *w, const double *area, int32_t device, rr_transform **out) {
    if (!out) { rr_set_error("null argument"); return 100; }
    *out = nullptr;
    if (n_rivers <= 0 || n_points <= 0 || !indptr || !indices || !w) { rr_set_error("bad weight table"); return 100; }
    if (indptr[0] != 0) { rr_set_error("weight table: indptr[0] must be 0"); return 100; }
    for (int64_t r = 0; r < n_rivers; ++r)
        if (indptr[r + 1] < indptr[r]) { rr_set_error("weight table: indptr must be non-decreasing"); return 100; }
    const int64_t nnz = indptr[n_rivers];
    for (int64_t j = 0; j < nnz; ++j)
        if (indices[j] < 0 || indices[j] >= n_points) {
            rr_set_error("weight table refers to grid cells outside the gathered runoff array");
            return 100;
        }
    if (!rr_cuda_available()) { rr_set_error("no CUDA device available: librr_b200 has no CPU fallback"); return 201; }
    rr_transform *t = new rr_transform();
    auto fail = [&](int rc) { rr_transform_destroy(t); return rc; };
    if (device >= 0 && cudaSetDevice(device) != cudaSuccess) { rr_set_error("cudaSetDevice failed"); return fail(200); }
    cudaGetDevice(&t->device);
    t->n_rivers = n_rivers; t->n_points = n_points; t->nnz = nnz;
    auto up = [&](void **dst, const void *src, size_t bytes) -> bool {
        if (cudaMalloc(dst, std::max<size_t>(bytes, 8)) != cudaSuccess) return false;
        return bytes == 0 || cudaMemcpy(*dst, src, bytes, cudaMemcpyHostToDevice) == cudaSuccess;
    };
    bool ok = up((void **)&t->indptr, indptr, sizeof(int32_t) * (size_t)(n_rivers + 1)) &&
              up((void **)&t->indices, indices, sizeof(int32_t) * (size_t)nnz) &&
              up((void **)&t->w, w, sizeof(double) * (size_t)nnz) &&
              (!area || up((void **)&t->area, area, sizeof(double) * (size_t)n_rivers));
    if (!ok) { rr_set_error(std::string("weight table upload: ") + cudaGetErrorString(cudaGetLastError())); return fail(200); }
    *out = t;
    return 0;
}

extern "C" int rr_transform_set_uh(rr_transform *t, int64_t n_ks, const double *kernel, int64_t ldk,
                                   const double *state, int64_t lds) {
    if (!t || !kernel || n_ks <= 0 || ldk < t->n_rivers || (state && lds < t->n_rivers)) { rr_set_error("bad unit hydrograph"); return 100; }
    CK(cudaSetDevice(t->device));
    const int64_t ld = ((t->n_rivers + 31) / 32) * 32;
    if (t->n_ks != n_ks) {
        if (t->uh_kernel) CK(cudaFree(t->uh_kernel));
        if (t->uh_state) CK(cudaFree(t->uh_state));
        t->uh_kernel = t->uh_state = nullptr;
        t->n_ks = 0;
        CK(cudaMalloc((void **)&t->uh_kernel, sizeof(double) * (size_t)n_ks * ld));
        CK(cudaMalloc((void **)&t->uh_state, sizeof(double) * (size_t)n_ks * ld));
        t->n_ks = n_ks; t->ld_uh = ld;
    }
    CK(cudaMemcpy2D(t->uh_kernel, ld * 8, kernel, ldk * 8, t->n_rivers * 8, n_ks, cudaMemcpyHostToDevice));
    if (state) CK(cudaMemcpy2D(t->uh_state, ld * 8, state, lds * 8, t->n_rivers * 8, n_ks, cudaMemcpyHostToDevice));
    else CK(cudaMemset(t->uh_state, 0, sizeof(double) * (size_t)n_ks * ld));
    return 0;
}

extern "C" int rr_transform_get_uh_state(rr_transform *t, double *state, int64_t lds) {
    if (!t || !state || !t->uh_state || lds < t->n_rivers) { rr_set_error("no unit hydrograph state"); return 100; }
    CK(cudaSetDevice(t->device));
    CK(cudaDeviceSynchronize());
    CK(cudaMemcpy2D(state, lds * 8, t->uh_state, t->ld_uh * 8, t->n_rivers * 8, t->n_ks, cudaMemcpyDeviceToHost));
    return 0;
}

// Output tail of TransformMuskingum._execute_routing on the device: mean over `k` consecutive rows
// (reshape(T/k, k, n).mean(axis=1): rows added one after the other, then divided by k; TransformMuskingum.py:128-139)
// and the cast to float32 the writer receives (:146 / Muskingum.py:259, round to nearest even like numpy's astype).
// Both kernels stride over rows by gridDim.y (at most 65535), so a chunk may hold any number of rows.
template <typename OT>
__global__ void __launch_bounds__(256) finish_output(const double *__restrict__ src, int64_t lds, OT *__restrict__ dst,
                                                     int64_t ldd, int64_t n_out, int64_t rows_out, int k,
                                                     const int32_t *__restrict__ subset) {
    const int64_t s = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= n_out) return;
    const int64_t i = subset ? (int64_t)__ldg(subset + s) : s;      // output column s shows river segment i
    for (int64_t t = blockIdx.y; t < rows_out; t += gridDim.y) {
        const double *p = src + t * k * lds + i;
        double acc = __ldg(p);
        for (int r = 1; r < k; ++r) acc += __ldg(p + (int64_t)r * lds);
        if (k > 1) acc = acc / (double)k;
        dst[t * ldd + s] = (OT)acc;
    }
}

__global__ void __launch_bounds__(256) upcast_rows(const float *__restrict__ src, int64_t lds, double *__restrict__ dst, int64_t ldd,
                                                    int64_t n, int64_t rows) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    for (int64_t t = blockIdx.y; t < rows; t += gridDim.y) dst[t * ldd + i] = (double)__ldg(src + t * lds + i);
}

static dim3 row_grid(int64_t n, int64_t rows) {
    return dim3((unsigned)((n + 255) / 256), (unsigned)std::min<int64_t>(rows, 65535));
}
// rows x n float32 -> fp64 (exact)
static int launch_upcast(const float *src, int64_t lds, double *dst, int64_t ldd, int64_t n, int64_t rows, cudaStream_t stream) {
    rr_timer tm(3, stream);
    upcast_rows<<<row_grid(n, rows), 256, 0, stream>>>(src, lds, dst, ldd, n, rows);
    CK(cudaGetLastError());
    rr_count_launch(1);
    return 0;
}
// rows_out rows of n_out columns (subset: their river segments, NULL: the first n_out), each the mean of k source rows
static int launch_finish(const double *src, int64_t lds, void *dst, int out_f32, int64_t ldd, int64_t n_out, int64_t rows_out,
                         int k, const int32_t *subset, cudaStream_t stream) {
    rr_timer tm(3, stream);
    const dim3 g = row_grid(n_out, rows_out);
    if (out_f32) finish_output<float><<<g, 256, 0, stream>>>(src, lds, (float *)dst, ldd, n_out, rows_out, k, subset);
    else finish_output<double><<<g, 256, 0, stream>>>(src, lds, (double *)dst, ldd, n_out, rows_out, k, subset);
    CK(cudaGetLastError());
    rr_count_launch(1);
    return 0;
}

int rr_weights_run(int64_t n_rivers, int64_t n_points, int64_t T, const int32_t *indptr, const int32_t *indices,
                   const double *w, const void *x, int x_is_f32, int64_t ldx, double *y, int64_t ldy, int cumulative,
                   int force_positive, const double *area, int64_t t_skip, cudaStream_t stream);

// ---- pageable callers ------------------------------------------------------------------------------
// numpy arrays are ordinary pageable memory: cudaMemcpyAsync on them is staged by the driver at a few GB/s and
// does not overlap with anything (measured: 6-10x slower end to end than pinned arrays).  The streamed path
// therefore bounces such arrays through its own pinned buffers with a few host threads doing the memcpy
// (first-touch page faults of a fresh output array included) while the GPU and the DMA engines work on the
// neighbouring chunks.  Pinned / registered arrays (rr_host_alloc, cudaHostRegister) are used in place.
enum { RR_PTR_PAGEABLE = 0, RR_PTR_PINNED = 1, RR_PTR_DEVICE = 2 };
static int host_pointer_kind(const void *p) {
    cudaPointerAttributes a;
    if (cudaPointerGetAttributes(&a, p) != cudaSuccess) { cudaGetLastError(); return RR_PTR_PAGEABLE; }
    if (a.type == cudaMemoryTypeDevice) return RR_PTR_DEVICE;
    return (a.type == cudaMemoryTypeHost || a.type == cudaMemoryTypeManaged) ? RR_PTR_PINNED : RR_PTR_PAGEABLE;
}
static int copy_threads() {
    if (const char *env = getenv("RR_COPY_THREADS")) return std::max(1, atoi(env));
    const unsigned hw = std::thread::hardware_concurrency();
    return (int)std::max(1u, std::min(8u, hw / 2));
}
// rows x row_bytes region copy, split evenly (by bytes) over the threads
static void parallel_copy_2d(char *dst, size_t dst_pitch, const char *src, size_t src_pitch, size_t row_bytes, int64_t rows) {
    const size_t total = row_bytes * (size_t)rows;
    if (total == 0) return;
    const int nt = (int)std::min<size_t>((size_t)copy_threads(), std::max<size_t>(1, total >> 20));
    auto work = [=](int i) {
        size_t a = total * (size_t)i / nt, b = total * (size_t)(i + 1) / nt;
        while (a < b) {
            const size_t r = a / row_bytes, o = a - r * row_bytes;
            const size_t len = std::min(b - a, row_bytes - o);
            std::memcpy(dst + r * dst_pitch + o, src + r * src_pitch + o, len);
            a += len;
        }
    };
    if (nt == 1) { work(0); return; }
    std::vector<std::thread> th;
    th.reserve(nt - 1);
    int started = 1;   // slice 0 runs on the calling thread; slices that could not get a thread run there too
    try {
        for (; started < nt; ++started) th.emplace_back(work, started);
    } catch (...) {
    }
    work(0);
    for (int i = started; i < nt; ++i) work(i);
    for (auto &t : th) t.join();
}

// What feeds the router, chunk by chunk: host lateral inflows (qlateral files) or gathered grid runoff that the
// weight table (and, for UnitMuskingum, the unit hydrograph) turns into lateral inflows on the device.
struct rr_stream_source {
    const void *lateral = nullptr;     // host lateral inflows, float64 or (lat_f32) float32
    int lat_f32 = 0;
    int64_t ldl = 0;
    rr_transform *tf = nullptr;
    const void *runoff = nullptr;
    int x_is_f32 = 0, cumulative = 0, force_positive = 0, as_volumes = 0;
    int64_t ldx = 0;
};

// Device copy of a host vector of the plan (output subset, thresholds), refreshed when its version changed.
template <typename T>
static int refresh(T **dev, uint64_t *dev_version, const std::vector<T> &host, uint64_t version) {
    if (*dev_version == version) return 0;
    CK(cudaDeviceSynchronize());
    if (*dev) CK(cudaFree(*dev));
    *dev = nullptr;
    if (!host.empty()) {
        CK(cudaMalloc((void **)dev, host.size() * sizeof(T)));
        CK(cudaMemcpy(*dev, host.data(), host.size() * sizeof(T), cudaMemcpyHostToDevice));
    }
    *dev_version = version;
    return 0;
}

// Chunk rows of a host call, from the caller's length model (RR_STREAM_CHUNK_ROWS overrides it; tests force many
// chunks with it): whole 16-row groups when the direct pipeline runs the call, else whole 8-row groups, then whole
// output rows, at most T.
static int64_t round_chunk(int64_t chunk, bool pipe, int64_t resample, int64_t T) {
    if (const char *env = getenv("RR_STREAM_CHUNK_ROWS")) chunk = std::max(1, atoi(env));
    if (pipe && chunk >= RR_FLAG_ROWS) chunk = chunk / RR_FLAG_ROWS * RR_FLAG_ROWS;
    else if (chunk >= 8) chunk = chunk / 8 * 8;
    chunk = std::max<int64_t>(resample, chunk / resample * resample);
    return std::min<int64_t>(chunk, T);
}

// One direction of a host call's chunk copies: n host arrays (0: nothing crosses), `width` bytes of each row, rows
// `h_pitch` bytes apart.  In a chunk buffer (device, and the pinned bounce buffer) array a starts at a * stride bytes,
// its rows d_pitch bytes apart.
struct rr_chunk_io {
    int n = 0;
    const void *const *host = nullptr;
    size_t width = 0, h_pitch = 0, d_pitch = 0, stride = 0;
    int64_t lead = 0;      // input: rows before its first row a chunk c > 0 carries too (cumulative grids: one)
    int64_t row_div = 1;   // output: chunk rows per host row (resampling)
    bool bounce = false;   // pageable host arrays: through the pinned bounce buffers, copied by host threads
    char *row(int a, int64_t r) const { return (char *)host[a] + (size_t)r * h_pitch; }
};

// Host arrays: stream the time chunks [start[c], start[c+1]) through two device buffers per direction.
//   s_in : H2D of chunk c+1        (cudaMemcpy2DAsync, pinned source gives full PCIe rate)
//   s_comp: work(c, k): the device work of chunk c, from s_inb[k] into s_outb[k]
//   s_out: D2H of chunk c-1
// finish() enqueues what follows the last chunk (the final states) before the streams are synchronised.
static int run_chunks(rr_device_state *d, const std::vector<int64_t> &start, const rr_chunk_io &in, const rr_chunk_io &out,
                      const std::function<int(int64_t, int)> &work, const std::function<int()> &finish) {
    int rc;
    for (int k = 0; k < 2; ++k) {
        if ((rc = grow_device(&d->s_inb[k], &d->s_inb_cap[k], in.n * in.stride))) return rc;
        if ((rc = grow_device(&d->s_outb[k], &d->s_outb_cap[k], out.n * out.stride))) return rc;
    }
    for (int k = 0; k < 2; ++k) {
        if (in.bounce && (rc = grow_pinned(&d->h_inb[k], &d->h_inb_cap[k], in.n * in.stride))) return rc;
        if (out.bounce && (rc = grow_pinned(&d->h_outb[k], &d->h_outb_cap[k], out.n * out.stride))) return rc;
    }
    const int64_t n_chunks = (int64_t)start.size() - 1;
    auto copy_in = [&](int64_t c) -> int {
        if (!in.n) return 0;
        const int k = (int)(c & 1);
        const int64_t r0 = start[c] - (c > 0 ? in.lead : 0), rows = start[c + 1] - r0;
        if (in.bounce) {
            if (c >= 2) CK(cudaEventSynchronize(d->ev_in[k]));           // H2D of chunk c-2 has left the bounce buffer
            for (int a = 0; a < in.n; ++a)
                parallel_copy_2d((char *)d->h_inb[k] + a * in.stride, in.d_pitch, in.row(a, r0), in.h_pitch, in.width, rows);
        }
        if (c >= 2) CK(cudaStreamWaitEvent(d->s_in, d->ev_comp[k], 0));  // buffer free once chunk c-2 was routed
        for (int a = 0; a < in.n; ++a) {
            const char *h = in.bounce ? (const char *)d->h_inb[k] + a * in.stride : in.row(a, r0);
            CK(cudaMemcpy2DAsync((char *)d->s_inb[k] + a * in.stride, in.d_pitch, h, in.bounce ? in.d_pitch : in.h_pitch,
                                 in.width, rows, cudaMemcpyHostToDevice, d->s_in));
        }
        CK(cudaEventRecord(d->ev_in[k], d->s_in));
        return 0;
    };
    // pageable output: chunk c leaves its bounce buffer once its D2H has finished
    auto drain = [&](int64_t c) -> int {
        if (!out.bounce || c < 0) return 0;
        const int k = (int)(c & 1);
        CK(cudaEventSynchronize(d->ev_out[k]));
        for (int a = 0; a < out.n; ++a)
            parallel_copy_2d(out.row(a, start[c] / out.row_div), out.h_pitch, (const char *)d->h_outb[k] + a * out.stride,
                             out.d_pitch, out.width, (start[c + 1] - start[c]) / out.row_div);
        return 0;
    };
    if ((rc = copy_in(0))) return rc;
    for (int64_t c = 0; c < n_chunks; ++c) {
        const int k = (int)(c & 1);
        if (in.n) CK(cudaStreamWaitEvent(d->s_comp, d->ev_in[k], 0));
        if (c >= 2) CK(cudaStreamWaitEvent(d->s_comp, d->ev_out[k], 0));  // out buffer drained
        if ((rc = work(c, k))) return rc;
        CK(cudaEventRecord(d->ev_comp[k], d->s_comp));
        CK(cudaStreamWaitEvent(d->s_out, d->ev_comp[k], 0));
        const int64_t rows_out = (start[c + 1] - start[c]) / out.row_div;
        for (int a = 0; a < out.n; ++a) {
            const char *b = (const char *)d->s_outb[k] + a * out.stride;
            if (out.bounce)
                CK(cudaMemcpyAsync((char *)d->h_outb[k] + a * out.stride, b, (size_t)rows_out * out.d_pitch, cudaMemcpyDeviceToHost, d->s_out));
            else
                CK(cudaMemcpy2DAsync(out.row(a, start[c] / out.row_div), out.h_pitch, b, out.d_pitch, out.width, rows_out,
                                     cudaMemcpyDeviceToHost, d->s_out));
        }
        CK(cudaEventRecord(d->ev_out[k], d->s_out));
        // host work of the neighbouring chunks while the device is busy with this one
        if (c + 1 < n_chunks && (rc = copy_in(c + 1))) return rc;
        if ((rc = drain(c - 1))) return rc;
    }
    if ((rc = drain(n_chunks - 1))) return rc;
    if ((rc = finish())) return rc;
    CK(cudaStreamSynchronize(d->s_comp));
    CK(cudaStreamSynchronize(d->s_out));
    CK(cudaStreamSynchronize(d->s_in));
    return 0;
}

// A failed host call: copies of earlier chunks may still be reading / writing the caller's arrays, so let them finish
// before the caller gets control back (and possibly frees the arrays); keep the first error message.
static int settle(rr_plan *p, int rc) {
    if (rc && p && p->dev) {
        const std::string msg = rr_last_error();
        cudaDeviceSynchronize();
        cudaGetLastError();
        rr_set_error(msg);
    }
    return rc;
}

// Single-member host calls: [weights -> unit hydrograph ->] route [-> resample / float32] per chunk, the state carried
// on the device from chunk to chunk.
static int stream_route_impl(rr_plan *p, int mode, double *q_state, double *q_full, const rr_stream_source &src, void *out,
                             int64_t ldo, int64_t T, int64_t substeps, int out_f32, int64_t resample) {
    if (!p || !q_state || !out) { rr_set_error("null argument"); return 100; }
    if (T <= 0 || substeps <= 0) { rr_set_error("T and substeps must be positive"); return 100; }
    if (resample < 1 || T % resample != 0) { rr_set_error("T must be a multiple of the output resampling factor"); return 100; }
    const bool grid = src.tf != nullptr;
    const bool has_lat = mode != RR_MODE_MUSKINGUM;
    if (has_lat && !grid && !src.lateral) { rr_set_error("null argument"); return 100; }
    if (grid) {
        if (!has_lat) { rr_set_error("Muskingum (channel only) takes no runoff"); return 100; }
        if (!src.runoff || src.ldx < src.tf->n_points) { rr_set_error("bad runoff array"); return 100; }
        if (src.tf->n_rivers != p->n) { rr_set_error("weight table rows do not match the number of river segments"); return 100; }
        if (mode == RR_MODE_UNIT && src.tf->n_ks <= 0) { rr_set_error("UnitMuskingum needs a unit hydrograph (rr_transform_set_uh)"); return 100; }
        if (src.as_volumes && !src.tf->area) { rr_set_error("as_volumes needs catchment areas in the weight table"); return 100; }
    }
    const int64_t n_out = p->out_subset.empty() ? p->n : (int64_t)p->out_subset.size();   // columns copied back
    if (ldo < n_out) { rr_set_error("output leading dimension smaller than the number of output river segments"); return 100; }
    int rc = ensure_device(p);
    if (rc) return rc;
    rr_device_state *d = p->dev;
    if (grid && src.tf->device != d->device) { rr_set_error("weight table and plan live on different devices"); return 100; }
    const int64_t n = p->n;
    const int64_t ldd = ((n + 31) / 32) * 32;  // device rows start on 256-byte boundaries
    const bool post = out_f32 || resample > 1 || !p->out_subset.empty();
    const bool uh = grid && mode == RR_MODE_UNIT;
    const bool pipe = pipeline_ok(p, mode, substeps);
    // Chunk length.  Short chunks keep the fill / drain of the three-stage pipeline small (aim: 1/16 of the call),
    // but every chunk is one wavefront launch whose dependency pipeline has to fill again (~20 us per level of the
    // block DAG): a chunk should last at least 4x that, where a row lasts as long as its slowest stage -- H2D, D2H
    // (~45 GB/s each, concurrently) or the device work (~14 ps per reach-substep).  Calls that copy little back
    // (output subsets) or little in (grids) therefore get long, device-efficient chunks; qlateral-in / all-segments-out
    // calls get short ones.  Bounded by ~1 GiB per transfer buffer and ~4 GiB of fp64 scratch rows.
    const int64_t row_bytes = ldd * 8;
    const double in_row = !has_lat ? 0.0 : (grid ? (double)src.tf->n_points * (src.x_is_f32 ? 4 : 8) : (double)n * (src.lat_f32 ? 4 : 8));
    const double out_row = (double)n_out * (out_f32 ? 4 : 8) / (double)resample;
    const double t_row = std::max({in_row / 45e9, out_row / 45e9, (double)n * (double)substeps * 14e-12});
    int64_t min_rows = (int64_t)std::ceil((double)(p->max_level + 1) * 80e-6 / t_row);
    // every chunk of a unit-hydrograph run also recomputes the n_ks - 1 rows of carry-over state
    if (uh) min_rows = std::max<int64_t>(min_rows, src.tf->n_ks);
    const int64_t xfer_cap = std::max<int64_t>(min_rows, (int64_t)((double)(1ll << 30) / std::max({in_row, out_row, 1.0})));
    const int64_t cap_rows = std::max<int64_t>(1, std::min<int64_t>(xfer_cap, (4ll << 30) / row_bytes));
    const int64_t chunk = round_chunk(std::max<int64_t>(1, std::min<int64_t>(std::max<int64_t>(T / 16, min_rows), cap_rows)), pipe,
                                      resample, T);
    // fused output tail (cast / subset written straight from the working tiles) when the direct pipeline runs the call
    const bool fused = post && resample == 1 && pipe;
    const size_t es_in = grid ? (src.x_is_f32 ? 4 : 8) : (src.lat_f32 ? 4 : 8), es_out = out_f32 ? 4 : 8;
    const int64_t ld_in = grid ? ((src.tf->n_points + 31) / 32) * 32 : ldd;
    const int64_t ldd_out = ((n_out + 31) / 32) * 32;
    if ((rc = refresh(&d->out_subset, &d->out_subset_version, p->out_subset, p->out_subset_version))) return rc;
    const void *h_src = grid ? src.runoff : (const void *)src.lateral;
    const int in_kind = has_lat ? host_pointer_kind(h_src) : RR_PTR_PINNED, out_kind = host_pointer_kind(out);
    if (in_kind == RR_PTR_DEVICE || out_kind == RR_PTR_DEVICE || host_pointer_kind(q_state) == RR_PTR_DEVICE) {
        rr_set_error("the host entry points take host pointers; use rr_route_dev for device-resident arrays");
        return 100;
    }
    rr_chunk_io in, outs;
    in.n = has_lat ? 1 : 0; in.host = &h_src; in.bounce = in_kind == RR_PTR_PAGEABLE;
    in.width = (size_t)(grid ? src.tf->n_points : n) * es_in; in.h_pitch = (size_t)(grid ? src.ldx : src.ldl) * es_in;
    in.d_pitch = (size_t)ld_in * es_in; in.stride = (size_t)(chunk + (grid ? 1 : 0)) * in.d_pitch;
    // a cumulative grid chunk starts with the last row of the previous chunk (its aggregate is the value to subtract)
    in.lead = (grid && src.cumulative) ? 1 : 0;
    const void *h_out = out;
    outs.n = 1; outs.host = &h_out; outs.bounce = out_kind == RR_PTR_PAGEABLE; outs.row_div = resample;
    outs.width = (size_t)n_out * es_out; outs.h_pitch = (size_t)ldo * es_out; outs.d_pitch = (size_t)ldd_out * es_out;
    outs.stride = (size_t)(chunk / resample) * outs.d_pitch;
    const size_t need_f64 = (size_t)chunk * ldd * 8;
    // float32 lateral inflows: the direct pipeline's staging kernel upcasts them on the fly; other paths get an exact
    // upcast into the fp64 scratch first
    const bool lat_cast = !grid && has_lat && src.lat_f32 && (!pipe || mode == RR_MODE_UNIT || substeps > 1);
    if ((grid || lat_cast) && (rc = grow_device((void **)&d->s_lat, &d->s_lat_cap, need_f64))) return rc;
    if (uh && (rc = grow_device((void **)&d->s_conv, &d->s_conv_cap, need_f64))) return rc;
    if (post && !fused && (rc = grow_device((void **)&d->s_route, &d->s_route_cap, need_f64))) return rc;
    if (!d->d_q) CK(cudaMalloc((void **)&d->d_q, sizeof(double) * (size_t)n));
    if (mode == RR_MODE_UNIT && !d->d_qfull) CK(cudaMalloc((void **)&d->d_qfull, sizeof(double) * (size_t)n));
    CK(cudaMemcpyAsync(d->d_q, q_state, sizeof(double) * (size_t)n, cudaMemcpyHostToDevice, d->s_comp));
    const int router_level = (mode != RR_MODE_UNIT) || q_full == nullptr;
    if (!router_level)
        CK(cudaMemcpyAsync(d->d_qfull, q_full, sizeof(double) * (size_t)n, cudaMemcpyHostToDevice, d->s_comp));

    // Chunk boundaries.  The pipeline cannot overlap anything with the H2D + device work of the first chunk, so the
    // first chunks are short (1/8, 1/4, 1/2 of the nominal length) when the call has enough of them.
    std::vector<int64_t> start;   // start[c] = first row of chunk c, start[n_chunks] = T
    {
        int64_t at = 0;
        const bool ramp = T >= 4 * chunk;
        for (int shift = 3; at < T; shift = std::max(0, shift - 1)) {
            int64_t len = ramp ? std::max<int64_t>(resample, ((chunk >> shift) / resample) * resample) : chunk;
            start.push_back(at);
            at += std::min<int64_t>(len, T - at);
        }
        start.push_back(T);
    }
    const int64_t n_chunks = (int64_t)start.size() - 1;
    const int32_t *sub = p->out_subset.empty() ? nullptr : d->out_subset;
    auto work = [&](int64_t c, int k) -> int {
        const int64_t rows = start[c + 1] - start[c], lead = (c > 0) ? in.lead : 0;
        const double *lat = (const double *)d->s_inb[k];
        if (lat_cast) {
            if ((rc = launch_upcast((const float *)d->s_inb[k], ld_in, d->s_lat, ldd, n, rows, d->s_comp))) return rc;
            lat = d->s_lat;
        }
        if (grid) {
            const rr_transform *t = src.tf;
            {
                rr_timer tm(3, d->s_comp);
                rc = rr_weights_run(n, t->n_points, rows + lead, t->indptr, t->indices, t->w, d->s_inb[k],
                                    src.x_is_f32, ld_in, d->s_lat, ldd, src.cumulative, src.force_positive,
                                    (src.as_volumes && !uh) ? t->area : nullptr, lead, d->s_comp);
            }
            if (rc) return rc;
            lat = d->s_lat;
            if (uh) {
                rr_timer tm(3, d->s_comp);
                rc = rr_uh_convolve_dev(n, t->n_ks, rows, d->s_lat, ldd, t->uh_kernel, t->ld_uh, t->uh_state, t->ld_uh,
                                        d->s_conv, ldd, d->s_comp);
                if (rc) return rc;
                lat = d->s_conv;
            }
        }
        double *route_out = post ? d->s_route : (double *)d->s_outb[k];
        const double *lat1[1] = {lat};
        double *out1[1] = {route_out}, *qs1[1] = {d->d_q}, *qf1[1] = {d->d_qfull};
        rr_out_spec spec;
        spec.dst = d->s_outb[k]; spec.f32 = out_f32; spec.ld = ldd_out; spec.n_out = n_out; spec.subset = sub;
        rc = route_any(p, mode, 1, d->d_q, lat1, ldd, out1, ldd, qs1, qf1, rows, substeps,
                       router_level && c == 0, router_level && c == n_chunks - 1, d->s_comp, fused ? &spec : nullptr,
                       (!grid && has_lat && src.lat_f32 && !lat_cast) ? 1 : 0);
        if (rc) return rc;
        if (post && !fused)
            return launch_finish(d->s_route, ldd, d->s_outb[k], out_f32, ldd_out, n_out, rows / resample, (int)resample, sub, d->s_comp);
        return 0;
    };
    auto finish = [&]() -> int {
        CK(cudaMemcpyAsync(q_state, d->d_q, sizeof(double) * (size_t)n, cudaMemcpyDeviceToHost, d->s_comp));
        if (!router_level)
            CK(cudaMemcpyAsync(q_full, d->d_qfull, sizeof(double) * (size_t)n, cudaMemcpyDeviceToHost, d->s_comp));
        return 0;
    };
    return run_chunks(d, start, in, outs, work, finish);
}

static int stream_route(rr_plan *p, int mode, double *q_state, double *q_full, const rr_stream_source &src, void *out,
                        int64_t ldo, int64_t T, int64_t substeps, int out_f32, int64_t resample) {
    return settle(p, stream_route_impl(p, mode, q_state, q_full, src, out, ldo, T, substeps, out_f32, resample));
}

// ---------------------------------------------------------------------------------------------------
// Ensembles from host arrays: the members of one time chunk are routed by ONE wavefront launch (tickets x members),
// every member from the same initial state (TransformMuskingum.py:121-126); chunks go through the same double-buffered
// pipeline as single-member calls (run_chunks), copied straight from and to the caller's arrays.  The member states
// stay on the device between chunks; at the end they are copied back and averaged in member order (:145-146).
// With `stats`, the members' fp64 rows stay on the device and only their statistics (rr_stats.cu) are copied back:
// out[s] / ldo / out_f32 then describe the statistic arrays, over the plan's output subset.  With `peak`, the running
// peaks of every statistic stay on the device for the whole call (-inf at the start, one D2H at the end); out may then
// be NULL, and no per-step rows are kept or copied.
// ---------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) member_mean_kernel(const double *__restrict__ states, int64_t ld, int n_members, int64_t n,
                                                           double *__restrict__ mean) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    double acc = states[i];                                  // np.array(states).mean(axis=0): rows added in member order,
    for (int m = 1; m < n_members; ++m) acc += states[(int64_t)m * ld + i];
    mean[i] = acc / (double)n_members;                       // then divided by the count
}

static int ensemble_host_impl(rr_plan *p, int mode, const double *q_init, int64_t ld_init, int M, const void *const *lateral, int lat_f32,
                              int64_t ldl, void *const *out, int64_t ldo, int out_f32, double *q_final, int64_t ldq,
                              double *q_mean, int64_t T, int64_t K, int64_t resample, const rr_stats_plan *stats = nullptr,
                              double *peak = nullptr, int32_t *peak_row = nullptr, int64_t ldk = 0) {
    if (!p || !q_init || !(out || (stats && peak)) || M < 1 || M > RR_MAX_MEMBERS) { rr_set_error("bad ensemble arguments (1..64 members)"); return 100; }
    if (mode == RR_MODE_UNIT) { rr_set_error("ensemble calls support Muskingum / RapidMuskingum"); return 100; }
    const bool has_lat = mode != RR_MODE_MUSKINGUM;
    if (has_lat && !lateral) { rr_set_error("null argument"); return 100; }
    if (T <= 0 || K <= 0 || resample < 1 || T % resample) { rr_set_error("T must be positive and a multiple of the resampling factor"); return 100; }
    if (!stats && !p->out_subset.empty()) { rr_set_error("ensemble calls copy back all river segments (clear the output subset)"); return 100; }
    if (stats && stats->n_members != M) { rr_set_error("internal: statistics prepared for another member count"); return 101; }
    int rc = ensure_device(p);
    if (rc) return rc;
    rr_device_state *d = p->dev;
    const int64_t n = p->n, ldd = ((n + 31) / 32) * 32;
    const int64_t n_out = (stats && !p->out_subset.empty()) ? (int64_t)p->out_subset.size() : n;   // columns copied back
    const int64_t ldd_out = ((n_out + 31) / 32) * 32;
    const int n_arrays = !out ? 0 : stats ? stats->n_stats : M;                                      // host arrays per row
    if ((out && ldo < n_out) || (peak && ldk < n_out) || (has_lat && ldl < n) || (q_final && ldq < n) || (ld_init != 0 && ld_init < n)) { rr_set_error("leading dimension smaller than n"); return 100; }
    const bool pipe = pipeline_ok(p, mode, K);
    const bool fused = pipe && resample == 1 && !stats;
    const bool cast_first = has_lat && lat_f32 && !(pipe && K == 1);
    const size_t es_in = lat_f32 ? 4 : 8, es_out = out_f32 ? 4 : 8;
    int64_t chunk;
    if (!stats) {
        // chunk rows: all members of a chunk are resident at once -- transfer buffers (x2), working tiles and scratch
        const double per_row = (double)M * (double)ldd * (2.0 * es_in + 2.0 * es_out + 16.0 + ((!fused) ? 8.0 : 0.0) + (cast_first ? 8.0 : 0.0));
        chunk = std::max<int64_t>(1, (int64_t)((double)(24ll << 30) / per_row));
    } else {
        // the longest chunk whose buffers fit the free device memory: what the buffers of this path hold already is
        // theirs, a larger one must fit next to everything else (one row of all members at 7M reaches is ~12 GB)
        size_t free_b = 0, total_b = 0;
        CK(cudaMemGetInfo(&free_b, &total_b));
        const double ldp = (double)(((p->n_work + 31) / 32) * 32), md = (double)M * (double)ldd;
        const double caps[] = {(double)d->s_inb_cap[0], (double)d->s_inb_cap[1], (double)d->s_outb_cap[0], (double)d->s_outb_cap[1],
                               (double)d->s_lat_cap, (double)d->s_route_cap, (double)d->p_lat_cap, (double)d->p_out_cap,
                               (double)d->p_q_cap, (double)d->ens_q_cap, (double)d->ens_peak_cap, 0.0};
        auto extra = [&](int64_t c) {
            const double tiles = (double)M * ldp * 8.0 * (double)((c + RR_FLAG_ROWS - 1) / RR_FLAG_ROWS * RR_FLAG_ROWS);
            const double outb = out ? (double)stats->n_stats * (double)(c / resample) * (double)ldd_out * (double)es_out : 0.0;
            // the last two: running peaks (12 B per statistic and column), thresholds still to upload
            const double need[] = {has_lat ? md * c * es_in : 0.0, has_lat ? md * c * es_in : 0.0, outb, outb,
                                   cast_first ? md * c * 8.0 : 0.0, md * c * 8.0, has_lat ? tiles : 0.0, tiles,
                                   4.0 * M * ldp * 8.0, (M + 2.0) * ldd * 8.0, peak ? 12.0 * stats->n_stats * ldd_out : 0.0,
                                   stats->exceed && d->thr_version != p->thr_version ? 8.0 * (double)p->n_thr * (double)n : 0.0};
            double more = 0.0;
            for (int b = 0; b < 12; ++b) more += std::max(0.0, need[b] - caps[b]);
            return more;
        };
        const double room = 0.92 * (double)free_b - (double)(256ll << 20);
        int64_t lo = 0, hi = T;   // largest chunk in [resample, T] with extra(chunk) <= room
        while (lo < hi) {
            const int64_t mid = (lo + hi + 1) / 2;
            if (extra(mid) <= room) lo = mid; else hi = mid - 1;
        }
        if (lo < resample) {
            rr_set_error("ensemble statistics: one output row of all " + std::to_string(M) + " members (" +
                         std::to_string((long long)(extra(resample) / 1e6)) + " MB of device buffers) does not fit in the " +
                         std::to_string((long long)(free_b / 1000000)) + " MB of free device memory");
            return 100;
        }
        chunk = lo;
    }
    chunk = round_chunk(chunk, pipe, resample, T);
    // one host array's rows of a chunk: a member's inflows; a member's discharge, or one statistic
    rr_chunk_io in, outs;
    in.n = has_lat ? M : 0; in.host = lateral;
    in.width = (size_t)n * es_in; in.h_pitch = (size_t)ldl * es_in; in.d_pitch = (size_t)ldd * es_in;
    in.stride = (size_t)chunk * in.d_pitch;
    outs.n = n_arrays; outs.host = out; outs.row_div = resample;
    outs.width = (size_t)n_out * es_out; outs.h_pitch = (size_t)ldo * es_out; outs.d_pitch = (size_t)ldd_out * es_out;
    outs.stride = (size_t)(chunk / resample) * outs.d_pitch;
    if (stats && (rc = refresh(&d->out_subset, &d->out_subset_version, p->out_subset, p->out_subset_version))) return rc;
    if (stats && stats->exceed && (rc = refresh(&d->thr, &d->thr_version, p->thr, p->thr_version))) return rc;
    rr_stats_ext ex;
    if (stats) {
        ex.thr = stats->exceed ? d->thr : nullptr;
        ex.ldt = n;
        if (peak) {
            if ((rc = grow_device(&d->ens_peak, &d->ens_peak_cap, (size_t)12 * stats->n_stats * ldd_out))) return rc;
            ex.peak = (double *)d->ens_peak;
            ex.peak_row = (int32_t *)(ex.peak + (size_t)stats->n_stats * ldd_out);
            ex.ldk = ldd_out;
        }
    }
    const size_t f64_member = (size_t)chunk * ldd;   // elements
    if (cast_first && (rc = grow_device((void **)&d->s_lat, &d->s_lat_cap, 8 * f64_member * M))) return rc;
    if (!fused && (rc = grow_device((void **)&d->s_route, &d->s_route_cap, 8 * f64_member * M))) return rc;
    if ((rc = grow_device((void **)&d->ens_q, &d->ens_q_cap, (size_t)(M + 2) * ldd * 8))) return rc;
    double *d_q0 = d->ens_q, *d_mean = d->ens_q + ldd, *d_qm = d->ens_q + 2 * ldd;
    // shared initial state (a reference call), or one state per member (a later time slab of the same members)
    const bool shared_init = ld_init == 0;
    if (shared_init) CK(cudaMemcpyAsync(d_q0, q_init, sizeof(double) * (size_t)n, cudaMemcpyHostToDevice, d->s_comp));
    else CK(cudaMemcpy2DAsync(d_qm, (size_t)ldd * 8, q_init, (size_t)ld_init * 8, (size_t)n * 8, M, cudaMemcpyHostToDevice, d->s_comp));
    if (ex.peak && (rc = rr_stats_peak_init(ex.peak, ex.peak_row, (int64_t)stats->n_stats * ldd_out, d->s_comp))) return rc;
    std::vector<int64_t> start;
    for (int64_t at = 0; at < T; at += chunk) start.push_back(at);
    start.push_back(T);
    const int64_t n_chunks = (int64_t)start.size() - 1;
    const int32_t *sub = p->out_subset.empty() ? nullptr : d->out_subset;
    auto work = [&](int64_t c, int k) -> int {
        const int64_t rows = start[c + 1] - start[c], rows_out = rows / resample;
        const double *lat_m[RR_MAX_MEMBERS];
        double *out_m[RR_MAX_MEMBERS], *qs_m[RR_MAX_MEMBERS];
        rr_out_spec spec[RR_MAX_MEMBERS];
        for (int m = 0; m < M; ++m) {
            const char *x = (const char *)d->s_inb[k] + in.stride * m;
            if (cast_first) {
                double *dst = d->s_lat + f64_member * m;
                if ((rc = launch_upcast((const float *)x, ldd, dst, ldd, n, rows, d->s_comp))) return rc;
                x = (const char *)dst;
            }
            lat_m[m] = (const double *)x;
            out_m[m] = fused ? nullptr : d->s_route + f64_member * m;
            qs_m[m] = d_qm + (size_t)m * ldd;
            spec[m].dst = (char *)d->s_outb[k] + outs.stride * m; spec[m].f32 = out_f32; spec[m].ld = ldd_out;
            spec[m].subset = nullptr; spec[m].n_out = n;
        }
        rc = route_any(p, mode, M, d_q0, has_lat ? lat_m : nullptr, ldd, out_m, ldd, qs_m, nullptr, rows, K, c == 0 && shared_init, c == n_chunks - 1,
                       d->s_comp, fused ? spec : nullptr, (has_lat && lat_f32 && !cast_first) ? 1 : 0);
        if (rc) return rc;
        if (stats) {
            // the members' fp64 rows in s_route -> resample -> statistics, one launch
            void *dst[RR_MAX_STATS];
            for (int s = 0; s < stats->n_stats; ++s) dst[s] = (char *)d->s_outb[k] + outs.stride * s;
            rr_timer tm(3, d->s_comp);
            ex.row0 = start[c] / resample;
            return rr_stats_launch(*stats, d->s_route, (int64_t)f64_member, ldd, (int)resample, rows_out, n_out, sub,
                                   out ? dst : nullptr, ldd_out, out_f32, ex, d->s_comp);
        }
        for (int m = 0; !fused && m < M; ++m)
            if ((rc = launch_finish(out_m[m], ldd, spec[m].dst, out_f32, ldd, n, rows_out, (int)resample, nullptr, d->s_comp))) return rc;
        return 0;
    };
    auto finish = [&]() -> int {
        if (q_mean) {
            member_mean_kernel<<<(unsigned)((n + 255) / 256), 256, 0, d->s_comp>>>(d_qm, ldd, M, n, d_mean);
            CK(cudaGetLastError());
            rr_count_launch(1);
            CK(cudaMemcpyAsync(q_mean, d_mean, sizeof(double) * (size_t)n, cudaMemcpyDeviceToHost, d->s_comp));
        }
        if (q_final) CK(cudaMemcpy2DAsync(q_final, (size_t)ldq * 8, d_qm, (size_t)ldd * 8, (size_t)n * 8, M, cudaMemcpyDeviceToHost, d->s_comp));
        if (ex.peak) {
            CK(cudaMemcpy2DAsync(peak, (size_t)ldk * 8, ex.peak, (size_t)ldd_out * 8, (size_t)n_out * 8, stats->n_stats,
                                 cudaMemcpyDeviceToHost, d->s_comp));
            CK(cudaMemcpy2DAsync(peak_row, (size_t)ldk * 4, ex.peak_row, (size_t)ldd_out * 4, (size_t)n_out * 4, stats->n_stats,
                                 cudaMemcpyDeviceToHost, d->s_comp));
        }
        return 0;
    };
    return run_chunks(d, start, in, outs, work, finish);
}

extern "C" int rr_route_ensemble_stats_host_ex(rr_plan *p, int mode, const double *q_init, int64_t ld_init, int32_t n_members,
                                               const void *const *lateral, int lateral_f32, int64_t ldl, const rr_stats_spec *stats,
                                               void *const *out, int64_t ldo, int out_f32, double *q_final, int64_t ldq,
                                               double *q_mean, int64_t T, int64_t substeps, int64_t resample, double *peak,
                                               int32_t *peak_row, int64_t ldk) {
    rr_stats_plan sp;
    int rc = rr_stats_prepare(stats, n_members, p ? p->n_thr : 0, &sp);
    if (rc) return rc;
    if (!out && !peak) { rr_set_error("no output: give per-step arrays (out), peaks (peak / peak_row) or both"); return 100; }
    if (peak && !peak_row) { rr_set_error("peak needs peak_row"); return 100; }
    for (int s = 0; out && s < sp.n_stats; ++s)
        if (!out[s]) { rr_set_error("null output array"); return 100; }
    return settle(p, ensemble_host_impl(p, mode, q_init, ld_init, n_members, lateral, lateral_f32, ldl, out, ldo, out_f32,
                                                 q_final, ldq, q_mean, T, substeps, resample, &sp, peak, peak_row, ldk));
}

extern "C" int rr_route_ensemble_stats_host(rr_plan *p, int mode, const double *q_init, int64_t ld_init, int32_t n_members,
                                            const void *const *lateral, int lateral_f32, int64_t ldl, const rr_stats_spec *stats,
                                            void *const *out, int64_t ldo, int out_f32, double *q_final, int64_t ldq,
                                            double *q_mean, int64_t T, int64_t substeps, int64_t resample) {
    if (!out) { rr_set_error("bad ensemble arguments (1..64 members)"); return 100; }
    return rr_route_ensemble_stats_host_ex(p, mode, q_init, ld_init, n_members, lateral, lateral_f32, ldl, stats, out, ldo, out_f32,
                                           q_final, ldq, q_mean, T, substeps, resample, nullptr, nullptr, 0);
}

extern "C" int rr_route_ensemble_host(rr_plan *p, int mode, const double *q_init, int64_t ld_init, int32_t n_members,
                                      const void *const *lateral, int lateral_f32, int64_t ldl, void *const *out, int64_t ldo,
                                      int out_f32, double *q_final, int64_t ldq, double *q_mean, int64_t T, int64_t substeps,
                                      int64_t resample) {
    return settle(p, ensemble_host_impl(p, mode, q_init, ld_init, n_members, lateral, lateral_f32, ldl, out, ldo, out_f32,
                                                 q_final, ldq, q_mean, T, substeps, resample));
}

extern "C" int rr_plan_set_thresholds(rr_plan *p, int32_t n_thr, const double *thr, int64_t ldt) {
    if (!p || n_thr < 0 || (n_thr > 0 && (!thr || ldt < p->n))) { rr_set_error("bad argument"); return 100; }
    p->thr.resize((size_t)n_thr * (size_t)p->n);
    for (int32_t r = 0; r < n_thr; ++r)
        std::copy(thr + (size_t)r * ldt, thr + (size_t)r * ldt + p->n, p->thr.begin() + (size_t)r * p->n);
    if (n_thr == 0) p->thr.shrink_to_fit();
    p->n_thr = n_thr;
    p->thr_version++;
    return 0;
}

extern "C" int rr_plan_set_output_subset(rr_plan *p, int64_t n_sub, const int32_t *idx) {
    if (!p || n_sub < 0 || (n_sub > 0 && !idx)) { rr_set_error("bad argument"); return 100; }
    for (int64_t s = 0; s < n_sub; ++s)
        if (idx[s] < 0 || idx[s] >= p->n) { rr_set_error("output subset refers to a river segment outside the network"); return 100; }
    p->out_subset.assign(idx, idx + n_sub);
    p->out_subset_version++;
    return 0;
}

extern "C" int rr_route_host(rr_plan *p, int mode, double *q_state, double *q_full, const double *lateral,
                             int64_t ldl, double *out, int64_t ldo, int64_t T, int64_t substeps) {
    rr_stream_source src;
    src.lateral = lateral; src.ldl = ldl;
    return stream_route(p, mode, q_state, q_full, src, out, ldo, T, substeps, 0, 1);
}

extern "C" int rr_route_host_ex(rr_plan *p, int mode, double *q_state, double *q_full, const double *lateral,
                                int64_t ldl, void *out, int64_t ldo, int64_t T, int64_t substeps, int out_f32,
                                int64_t resample) {
    rr_stream_source src;
    src.lateral = lateral; src.ldl = ldl;
    return stream_route(p, mode, q_state, q_full, src, out, ldo, T, substeps, out_f32, resample);
}

extern "C" int rr_route_host_typed(rr_plan *p, int mode, double *q_state, double *q_full, const void *lateral,
                                   int lateral_f32, int64_t ldl, void *out, int64_t ldo, int64_t T, int64_t substeps,
                                   int out_f32, int64_t resample) {
    rr_stream_source src;
    src.lateral = lateral; src.lat_f32 = lateral_f32; src.ldl = ldl;
    return stream_route(p, mode, q_state, q_full, src, out, ldo, T, substeps, out_f32, resample);
}

extern "C" int rr_runoff_route_host(rr_plan *p, rr_transform *t, int mode, double *q_state, const void *runoff,
                                    int x_is_f32, int64_t ldx, int64_t T, int cumulative, int force_positive,
                                    int as_volumes, void *out, int64_t ldo, int64_t substeps, int out_f32,
                                    int64_t resample) {
    if (!t) { rr_set_error("null argument"); return 100; }
    rr_stream_source src;
    src.tf = t; src.runoff = runoff; src.x_is_f32 = x_is_f32; src.ldx = ldx;
    src.cumulative = cumulative; src.force_positive = force_positive; src.as_volumes = as_volumes;
    return stream_route(p, mode, q_state, nullptr, src, out, ldo, T, substeps, out_f32, resample);
}

// Cycle counters of RR_PROFILE builds (zero otherwise): [0] ticket + decode, [1] constants + dependency waits,
// [2] item body, [3] release; summed over warps.  Resets after reading.
extern "C" int rr_plan_read_profile(rr_plan *p, uint64_t *out8) {
    if (!p || !p->dev || !out8) { rr_set_error("no device state"); return 100; }
    CK(cudaDeviceSynchronize());
    CK(cudaMemcpy(out8, p->dev->prof, 8 * sizeof(uint64_t), cudaMemcpyDeviceToHost));
    CK(cudaMemset(p->dev->prof, 0, 8 * sizeof(uint64_t)));
    return 0;
}

extern "C" int rr_host_alloc(void **ptr, int64_t bytes) {
    if (!ptr || bytes <= 0) { rr_set_error("bad argument"); return 100; }
    CK(cudaHostAlloc(ptr, (size_t)bytes, cudaHostAllocDefault));
    return 0;
}
extern "C" int rr_host_free(void *ptr) {
    CK(cudaFreeHost(ptr));
    return 0;
}
