// rr_direct.cu -- the routing pipeline of level-sorted plans with one routing substep per row
// (RapidMuskingum / Muskingum; river_route/routers/_numba_kernels.py rapid_route :49-84, muskingum_route :9-46):
//
//   stage_in   caller's (T, n) lateral inflows (params-file order) -> working tiles [tile][block][reach][row];
//              whole blocks of headwater reaches (level 0: no upstream, q' = c3*q + c4_dt*ql) are routed right here,
//              while their lateral rows pass through registers, and only their discharge series is written
//   wavefront  rr_direct_kernel: persistent warps, one (block of 32 same-level reaches, time tile) per ticket.  The
//              working discharge array keeps the RAW series and is the exchange buffer: a reach reads its upstream
//              reaches' series straight from their discharge tiles ("direct exchange").  done[block] counts finished
//              16-row groups (one 128-byte line per reach): blocks of narrow levels publish every group and consume
//              their upstream blocks group by group, so that deep, narrow parts of the network pipeline at a few
//              microseconds per level instead of one whole work item per level.  Networks of at most 4096 blocks hand
//              results over without flags inside a tile (narrow_item below).
//   stage_out  working discharge tiles -> caller's layout with the reference's clamp (:44-46 / :82-84), optionally cast
//              to float32 (TransformMuskingum.py:146) and restricted to an output subset.
//
// Per reach i with upstream set U(i) in ascending params-file index (the reference's summation order):
//     q'[i] = c3*q[i] + c4_dt*ql[t,i] + sum_u c2[i]*q[u] + sum_u c1[i]*q'[u]
#include <cuda_runtime.h>

#include <algorithm>
#include <string>

#include "rr_device.cuh"

using namespace rrdev;

void rr_count_launch(int64_t k);

namespace {

// RR_TRACE builds (tools/trace_chain.py; never the shipped library): lane 0 stamps {globaltimer, clock64} of six events per
// (block, 16-row group) into P.prof = [block][group][event][2]
#ifdef RR_TRACE
#define RR_NEV 6
__device__ __forceinline__ void trace_ev(const rr_route_params &P, int lane, int b, int g, int ev) {
    if (lane == 0 && P.prof) {
        unsigned long long t;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t)::"memory");
        unsigned long long *q = P.prof + (((size_t)b * ((size_t)P.n_tiles * P.gpt) + (size_t)g) * RR_NEV + ev) * 2;
        q[0] = t;
        q[1] = (unsigned long long)clock64();
    }
}
#define TR(b, g, ev) trace_ev(P, lane, b, g, ev)
#define TR_AFTER(x, b, g, ev) do { asm volatile("" ::"d"(x) : "memory"); trace_ev(P, lane, b, g, ev); } while (0)
#else
#define TR(b, g, ev) do { } while (0)
#define TR_AFTER(x, b, g, ev) do { } while (0)
#endif

// row 0 of working reach u's series in tile jj (reach-major tiles, tile_pitch doubles per reach)
__device__ __forceinline__ const double *tile_of(const double *base, const rr_route_params &P, int jj, int64_t u) {
    return base + (((size_t)jj * P.n_blocks + (size_t)(u >> 5)) * RR_BLOCK + (size_t)(u & 31)) * (size_t)P.tile_pitch;
}

__device__ __forceinline__ const double *lat_tile_of(const double *base, const rr_route_params &P, int jj, int64_t u) {
    return base + (((size_t)jj * P.n_blocks + (size_t)(u >> 5)) * RR_BLOCK + (size_t)(u & 31)) * (size_t)P.lat_pitch;
}

struct dctx {
    int m, b, j, lane, TT, deg;
    int64_t i;
    bool valid, narrow, prog;    // prog: upstream blocks were not complete at the start -> consume them group by group
    double c1, c2, c3, c4, q;
    int32_t up_u[RR_MAX_FAST_DEG];
    int32_t dep_blk;             // this lane's entry of the block's upstream-block list (-1: none)
    int32_t dep_more, dep_hi;    // further entries of this lane: dep_more, dep_more + 32, ... < dep_hi (blocks with > 32 upstream blocks)
    const int32_t *dep_idx;
    int32_t spin_ns;
    int32_t *done;               // this member's progress counters
    const double *lat0;
    double *out0;
};

// all lanes: wait until every upstream block has published `want`; sets full when they are all past `full_want`.
// Polls with acquire loads: this wait sits on the critical path of deep, narrow networks, where a separate acquire after
// a relaxed poll would add one more L2 round trip per level (the L1 invalidation an acquire costs does not matter to a
// warp that is waiting anyway).
__device__ __forceinline__ void wait_groups(const dctx &c, int32_t want, int32_t full_want, bool &full) {
    unsigned ns = (unsigned)c.spin_ns;
    for (;;) {
        int32_t p = c.dep_blk >= 0 ? ld_acquire(c.done + c.dep_blk) : 0x7fffffff;
        for (int e = c.dep_more; e < c.dep_hi; e += 32) p = min(p, ld_acquire(c.done + __ldg(c.dep_idx + e)));
        if (__all_sync(RR_FULL_MASK, p >= want)) {
            full = __all_sync(RR_FULL_MASK, p >= full_want);
            break;
        }
        if (ns) {
            __nanosleep(ns);
            if (ns < 256) ns <<= 1;
        }
    }
    __syncwarp();
}

// One work item.  Software pipeline over groups of four rows: while rows s..s+3 are computed the sectors of rows
// s+4.. and s+8.. are in flight.  Results are parked in shared memory and leave as whole 128-byte lines every 16
// rows (four back-to-back 256-bit stores per reach): a line written one sector per ~600 cycles left L2 partially
// dirty and cost DRAM read-modify-write traffic (ncu: 11.5 B written + 1.6 B read more than the 8 + 17.4 B the
// kernel asks for, per reach-timestep).
// SUB: more than one routing substep per row (dt_routing < dt_runoff).  The tiles then hold the raw SUBSTEP series
// (tile_rows x K entries per reach), the lateral value changes every K entries, and the interval mean of
// _numba_kernels.py:41-46 / :79-84 is formed by stage_out from the raw substeps (same order: sum, then x 1/K).
template <int MODE, int NS, bool SUB>
__device__ __forceinline__ void direct_item(const rr_route_params &P, const dctx &c, double *stage) {
    constexpr bool HAS_LAT = (MODE == RR_MODE_RAPID);
    constexpr int NA = NS > 0 ? NS : 1;
    const double c1 = c.c1, c2 = c.c2, c3 = c.c3, c4 = c.c4;
    const int TT = c.TT, j = c.j, lane = c.lane;
    const int32_t gbase = j * P.gpt;
    double q = c.q;
    const double *up[NA];
    bool has[NA];
    double old[NA];
    d4 nxt[NA], fut[NA];
    bool full = !c.prog;
#pragma unroll
    for (int k = 0; k < NS; ++k) {
        has[k] = k < c.deg;
        up[k] = P.out[c.m];
        old[k] = 0.0;
        nxt[k] = fut[k] = d4{0, 0, 0, 0};
        if (has[k]) {
            up[k] = tile_of(P.out[c.m], P, j, c.up_u[k]);
            // value before the tile's first row: the start-of-call state, or the last row of the previous tile
            old[k] = j == 0 ? P.q_init[(size_t)c.m * P.q_init_stride + c.up_u[k]] : tile_of(P.out[c.m], P, j - 1, c.up_u[k])[P.tile_rows * P.K - 1];
            nxt[k] = ld_sector(up[k]);                       // rows 0..7 are in group 0, which is published
            if (4 < TT) fut[k] = ld_sector(up[k] + 4);
        }
    }
    const double *lat = c.lat0;
    auto lat_group = [&](int s0) -> d4 {
        if (!(HAS_LAT && c.valid) || s0 >= TT) return d4{0, 0, 0, 0};
        if (SUB) {                                       // substeps s0..s0+3 take the lateral value of row (s0 + u) / K
            const int K = P.K, r0 = s0 / K, o0 = s0 - r0 * K;
            d4 v;
            v.a = __ldg(lat + r0);
            v.b = __ldg(lat + r0 + (o0 + 1) / K);
            v.c = __ldg(lat + r0 + (o0 + 2) / K);
            v.d = __ldg(lat + r0 + (o0 + 3) / K);   // (a row past the tile's last one is read but never used: the pitch covers it)
            return v;
        }
        return ld_sector_ro(lat + s0);
    };
    d4 lcur = lat_group(0), lnxt = lat_group(4);
    double *st = stage + lane;                     // [row & 15][lane]
    for (int s = 0; s < TT; s += 4) {
        // Upstream blocks still running (narrow levels): their series is consumed one published 16-row group at a time
        // and WITHOUT look-ahead into the next group -- waiting at row s for group (s+8)/16 made every level lag its
        // upstream by a whole extra group (measured on the 3000-reach stem of C2: ~6.5 us per level instead of ~2.5).
        if (NS > 0 && !full && (s & 15) == 0 && s > 0) {
            wait_groups(c, gbase + (s >> 4) + 1, gbase + P.gpt, full);
#pragma unroll
            for (int k = 0; k < NS; ++k)
                if (has[k]) {
                    nxt[k] = ld_sector(up[k] + s);
                    if (s + 4 < TT) fut[k] = ld_sector(up[k] + s + 4);
                }
        }
        const bool ahead = full || ((s + 8) >> 4) == (s >> 4);   // rows s+8.. lie in a published group
        d4 far[NA];
#pragma unroll
        for (int k = 0; k < NS; ++k) {
            far[k] = d4{0, 0, 0, 0};
            if (has[k] && s + 8 < TT && ahead) far[k] = ld_sector(up[k] + s + 8);
        }
        const d4 lfar = lat_group(s + 8);
        double r0, r1, r2, r3;
        {
            double r = c3 * q;                                       // _numba_kernels.py:27-28 / :68-69
            if (HAS_LAT) r = fma(c4, lcur.a, r);
#pragma unroll
            for (int k = 0; k < NS; ++k) r = fma(c2, old[k], r);     // :29-33 / :70-74, ascending upstream
#pragma unroll
            for (int k = 0; k < NS; ++k) r = fma(c1, nxt[k].a, r);   // :36-39 / :75-78 (lhs_off = -c1)
            r0 = r;
            r = c3 * r0;
            if (HAS_LAT) r = fma(c4, lcur.b, r);
#pragma unroll
            for (int k = 0; k < NS; ++k) r = fma(c2, nxt[k].a, r);
#pragma unroll
            for (int k = 0; k < NS; ++k) r = fma(c1, nxt[k].b, r);
            r1 = r;
            r = c3 * r1;
            if (HAS_LAT) r = fma(c4, lcur.c, r);
#pragma unroll
            for (int k = 0; k < NS; ++k) r = fma(c2, nxt[k].b, r);
#pragma unroll
            for (int k = 0; k < NS; ++k) r = fma(c1, nxt[k].c, r);
            r2 = r;
            r = c3 * r2;
            if (HAS_LAT) r = fma(c4, lcur.d, r);
#pragma unroll
            for (int k = 0; k < NS; ++k) r = fma(c2, nxt[k].c, r);
#pragma unroll
            for (int k = 0; k < NS; ++k) r = fma(c1, nxt[k].d, r);
            r3 = r;
        }
        const int rr = s & 15;
        st[(rr + 0) * RR_BLOCK] = r0;
        st[(rr + 1) * RR_BLOCK] = r1;
        st[(rr + 2) * RR_BLOCK] = r2;
        st[(rr + 3) * RR_BLOCK] = r3;
        q = (s + 3 < TT) ? r3 : ((s + 2 < TT) ? r2 : ((s + 1 < TT) ? r1 : r0));
        if (rr == 12 || s + 4 >= TT) {
            // one whole line (or the tail of the tile) of this reach's series; rows past TT inside the last sector are
            // never read (consumers and stage_out stop at TT)
            if (c.valid) {
                double *o = c.out0 + (s - rr);
#pragma unroll
                for (int v = 0; v < 16; v += 4)
                    if (v <= rr) st_sector(o + v, st[(v + 0) * RR_BLOCK], st[(v + 1) * RR_BLOCK], st[(v + 2) * RR_BLOCK], st[(v + 3) * RR_BLOCK]);
            }
            if (c.narrow && s + 4 < TT) {
                jitter_delay(P.jitter, c.b, j, 1 + (s >> 4));
                __syncwarp();
                if (lane == 0) st_release(c.done + c.b, gbase + (s >> 4) + 1);
            }
        }
#pragma unroll
        for (int k = 0; k < NS; ++k) { old[k] = nxt[k].d; nxt[k] = fut[k]; fut[k] = far[k]; }
        lcur = lnxt;
        lnxt = lfar;
    }
    if (c.valid) P.q_state[c.m][c.i] = q;
}


// -----------------------------------------------------------------------------------------------------------------
// Small networks (at most RR_SENTINEL_MAX_BLOCKS blocks, rr_api.cu: every level is narrow and the whole launch is bound by
// the latency of the dependency chain, not by bandwidth; kernels instantiated with SENT = true).  Larger networks keep the
// progress flags above: there the pattern costs DRAM bandwidth that the streaming part of the launch pays for
// (profiles/r02_chain_latency.md).  The results ARE the message: before the launch the discharge tiles of narrow blocks are filled with a
// signalling-NaN pattern no arithmetic result can have (fill_sentinel_kernel); a producer writes its series with
// st.relaxed.gpu, whole 128-byte lines every 16 entries, and never fences inside a tile; a consumer loads the 16 entries of
// a group with ld.relaxed.gpu (L1 bypassed) and repeats the load until none of them is the pattern (every 8-byte entry
// is written once and is single-copy atomic).  One L2 round trip per level instead of fence + flag store + flag poll +
// data load (trace of the 189-level chain of C1, tools/trace_chain.py: 4.6 us per level, of which 0.8 us fence, 1.3 us flag
// hand-over, 0.8 + 1.8 us two exposed data round trips).  done[block] is still released once per tile: own next tile,
// consumers on wide levels, and the safety net below.
// -----------------------------------------------------------------------------------------------------------------
#define RR_SENTINEL_BITS 0xFFF4A5A5DEADBEEFull   // sign 1, exponent all ones, quiet bit 0: a signalling NaN
__device__ __forceinline__ bool is_set(double v) { return (unsigned long long)__double_as_longlong(v) != RR_SENTINEL_BITS; }
__device__ __forceinline__ bool is_set(const d4 &v) { return is_set(v.a) & is_set(v.b) & is_set(v.c) & is_set(v.d); }
__device__ __forceinline__ d4 ld_sector_strong(const double *p) {
    d4 v;
    asm volatile("ld.relaxed.gpu.global.L2::128B.v4.f64 {%0, %1, %2, %3}, [%4];" : "=d"(v.a), "=d"(v.b), "=d"(v.c), "=d"(v.d) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ double ld_strong(const double *p) {
    double v;
    asm volatile("ld.relaxed.gpu.global.f64 %0, [%1];" : "=d"(v) : "l"(p) : "memory");
    return v;
}
// (two 128-bit stores: ptxas 12.9 narrowed st.relaxed.gpu.global.v4.f64 to a 64-bit STG.E.64.STRONG.GPU in the
// in-degree-4 instantiations -- cuobjdump showed one double of each sector stored)
__device__ __forceinline__ void st_sector_strong(double *p, double a, double b, double c, double d) {
    asm volatile("st.relaxed.gpu.global.v2.f64 [%0], {%1, %2};" ::"l"(p), "d"(a), "d"(b) : "memory");
    asm volatile("st.relaxed.gpu.global.v2.f64 [%0], {%1, %2};" ::"l"(p + 2), "d"(c), "d"(d) : "memory");
}

// (not inlined: its register allocation -- 64 registers of upstream entries for two upstream reaches -- stays out of the
// bandwidth path's, which keeps 0 spills)
//
// Per 16-entry group: (1) one optimistic fetch of the whole group of every upstream reach; when an entry is still the
// pattern the warp polls the group's LAST entry only (one sector per lane and upstream reach instead of four: polling
// the whole group from ~1500 waiting warps saturated L2 and slowed the producers they were waiting for), backing off,
// and then fetches what is missing; (2) the group's own lateral inflows were brought into the warp's 4 KB of shared memory
// by cp.async while the warp waited (K == 1), so the 16 dependent steps run from registers and shared memory; (3) the
// results overwrite the lateral entries in place and leave as four 256-bit strong stores per reach.
__device__ __forceinline__ void prefetch_l2(const void *p) { asm volatile("prefetch.global.L2 [%0];" ::"l"(p)); }
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
// entry e (0..15) of lane l in the warp's buffer: pairs of entries are 16-byte units, [pair][lane] (conflict-free)
__device__ __forceinline__ int buf_pair(int pair, int lane) { return (pair * RR_BLOCK + lane) * 2; }

template <int MODE, int NS, bool SUB>
__device__ __noinline__ void narrow_item(const rr_route_params &P, const dctx &c, double *stage) {
    constexpr bool HAS_LAT = (MODE == RR_MODE_RAPID);
    constexpr bool LAT_SMEM = HAS_LAT && !SUB;          // lateral group staged through shared memory by cp.async
    constexpr int NA = NS > 0 ? NS : 1;
    const double c1 = c.c1, c2 = c.c2, c3 = c.c3, c4 = c.c4;
    const int TT = c.TT, j = c.j, lane = c.lane;
    const int32_t gbase = j * P.gpt;
    (void)gbase;
    double q = c.q;
    const double *up[NA];
    bool has[NA], poll[NA];
    double old[NA];
    d4 U[NA][4];
    const double *lat = c.lat0;
    // this lane's 16-byte units of the buffer: pair p at stage + buf_pair(p, lane)
    auto stage_lateral = [&](int s0) {
        if (!LAT_SMEM) return;
        if (c.valid) {
            const uint32_t dst = smem_u32(stage + buf_pair(0, lane));
#pragma unroll
            for (int pr = 0; pr < 8; ++pr)
                asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst + (uint32_t)pr * (RR_BLOCK * 16)), "l"(lat + s0 + 2 * pr) : "memory");
        }
        asm volatile("cp.async.commit_group;" ::: "memory");
    };
    stage_lateral(0);
#pragma unroll
    for (int k = 0; k < NS; ++k) {
        has[k] = k < c.deg;
        poll[k] = false;
        up[k] = P.out[c.m];
        old[k] = 0.0;
        if (has[k]) {
            const int32_t u = c.up_u[k], ub = u >> 5;
            // upstream blocks outside the protocol (wide levels, blocks routed by the staging kernel) are complete: the
            // kernel waited for their tile flags
            poll[k] = ub >= P.poll_lo && (P.meta[ub].int_mask & RR_META_NARROW) != 0;
            up[k] = tile_of(P.out[c.m], P, j, u);
            // value before the tile's first entry: the start-of-call state, or the last entry of the previous tile
            const double *po = j == 0 ? P.q_init + ((size_t)c.m * P.q_init_stride + u) : tile_of(P.out[c.m], P, j - 1, u) + (P.tile_rows * P.K - 1);
            old[k] = (j > 0 && poll[k]) ? ld_strong(po) : *po;
        }
    }
    // Most upstream reaches of a deep block are headwaters and shallow tributaries whose entries were written hundreds of
    // microseconds ago and have left L2 (ncu on C1: 52 % L2 read hit rate, 0.7 GB of DRAM reads beyond the lateral inflows):
    // bring every line two groups ahead of its use into L2, so that the fetch on the critical path is an L2 hit (and the
    // page walk of its 2 MB page is over) whichever upstream block it comes from.  A line that is not written yet comes
    // in armed; its producer then writes into L2.
#pragma unroll
    for (int k = 0; k < NS; ++k)
        if (has[k]) {
            prefetch_l2(up[k]);
            if (16 < TT) prefetch_l2(up[k] + 16);
        }
    if (LAT_SMEM && c.valid && 16 < TT) prefetch_l2(lat + 16);
    // The series the warp watches while it waits: one reach of the DEEPEST upstream block of the whole warp (the last one
    // to deliver, as a rule).  All lanes poll that one word -- one L2 request per warp and round -- and only when it is set
    // fetch and validate their own upstream entries.  (Every lane polling its own upstream reaches cost 64 requests per
    // warp and round; with ~1500 warps waiting along the chain that was ~5 TB/s of L2 traffic and every round trip in the
    // kernel took 1-1.4 us instead of the 0.5 us a store -> load hand-over takes on an idle B200, tools/micro/pingpong.cu.)
    const double *hint = nullptr;
    if (NS > 0) {
        int best = -1;
#pragma unroll
        for (int k = 0; k < NS; ++k)
            if (poll[k]) {
                const int lv = P.meta[c.up_u[k] >> 5].level;
                if (lv > best) { best = lv; hint = up[k]; }
            }
        const int wmax = __reduce_max_sync(RR_FULL_MASK, best);
        const unsigned who = __ballot_sync(RR_FULL_MASK, best == wmax && best >= 0);
        const int src = who ? __ffs(who) - 1 : 0;
        hint = reinterpret_cast<const double *>(__shfl_sync(RR_FULL_MASK, (unsigned long long)hint, src));
        if (!who) hint = nullptr;
    }
    // (the previous tile's last entry was read by the warp that ran this block's previous tile before it released the
    // block's flag, which this warp acquired: it is set -- the loop only guards the argument)
#pragma unroll
    for (int k = 0; k < NS; ++k)
        while (j > 0 && poll[k] && !is_set(old[k])) old[k] = ld_strong(tile_of(P.out[c.m], P, j - 1, c.up_u[k]) + (P.tile_rows * P.K - 1));
    auto lat_group = [&](int s0) -> d4 {                 // SUB only: substeps s0..s0+3 take the lateral value of row (s0 + u) / K
        if (!(HAS_LAT && SUB && c.valid) || s0 >= TT) return d4{0, 0, 0, 0};
        const int K = P.K, r0 = s0 / K, o0 = s0 - r0 * K;
        d4 v;
        v.a = __ldg(lat + r0);
        v.b = __ldg(lat + r0 + (o0 + 1) / K);
        v.c = __ldg(lat + r0 + (o0 + 2) / K);
        v.d = __ldg(lat + r0 + (o0 + 3) / K);
        return v;
    };
    d4 lcur = lat_group(0), lnxt = lat_group(4);
    const int32_t full_want = (j + 1) * P.gpt;
    for (int s0 = 0; s0 < TT; s0 += 16) {
        const int nv = min(4, (TT - s0 + 3) >> 2);       // 32-byte sectors of this group that hold entries of the tile
        TR(c.b, gbase + (s0 >> 4), 5);
        if (s0 + 32 < TT) {
#pragma unroll
            for (int k = 0; k < NS; ++k)
                if (has[k]) prefetch_l2(up[k] + s0 + 32);
            if (LAT_SMEM && c.valid) prefetch_l2(lat + s0 + 32);
        } else if (j + 1 < P.n_tiles) {
            // the first lines of the block's next tile (another work item, possibly another warp)
            const int g2 = (s0 + 32 - TT) >> 4;          // 0 or 1
#pragma unroll
            for (int k = 0; k < NS; ++k)
                if (has[k]) prefetch_l2(tile_of(P.out[c.m], P, j + 1, c.up_u[k]) + 16 * g2);
            if (LAT_SMEM && c.valid) prefetch_l2(lat_tile_of(P.lateral[c.m], P, j + 1, c.i) + 16 * g2);
        }
        if (NS > 0) {
            bool ok = true;
#pragma unroll
            for (int k = 0; k < NS; ++k)
#pragma unroll
                for (int v = 0; v < 4; ++v) {
                    U[k][v] = d4{0, 0, 0, 0};
                    if (has[k] && v < nv) {
                        U[k][v] = poll[k] ? ld_sector_strong(up[k] + s0 + 4 * v) : ld_sector(up[k] + s0 + 4 * v);
                    }
                }
            // the watched word travels with the optimistic fetch: when the group is not complete yet the warp already knows
            // whether the deepest upstream block has delivered, one round trip earlier
            const int last = min(s0 + 15, TT - 1);
            double hv = hint ? ld_strong(hint + last) : 0.0;
#pragma unroll
            for (int k = 0; k < NS; ++k)
#pragma unroll
                for (int v = 0; v < 4; ++v)
                    if (poll[k] && v < nv) ok &= is_set(U[k][v]);
            if (!__all_sync(RR_FULL_MASK, ok)) {
                // a warp at the head of a tile may be far ahead of the wave: it backs off further than one inside a tile
                const unsigned cap = s0 == 0 ? 1024u : 128u;
                unsigned ns = (unsigned)P.spin_ns, spins = 0;
                bool accept = false;
                for (;;) {
                    // phase 1: the watched word (uniform address: one request per warp)
                    if (hint) {
                        for (; !is_set(hv); hv = ld_strong(hint + last)) {
                            if ((++spins & 255u) == 0) {
                                // safety net: an upstream block that has released this tile has written every entry of
                                // it -- whatever the entries look like
                                bool fin = true;
#pragma unroll
                                for (int k = 0; k < NS; ++k)
                                    if (poll[k]) fin &= ld_acquire(c.done + (c.up_u[k] >> 5)) >= full_want;
                                if (__all_sync(RR_FULL_MASK, fin)) { accept = true; break; }
                            }
                            if (ns) {            // (spin_ns == 0: poll without sleeping)
                                __nanosleep(ns);
                                if (ns < cap) ns *= 2u;
                            }
                        }
                    }
                    // phase 2: this lane's own upstream entries (normally all there: one more round trip)
                    ok = true;
#pragma unroll
                    for (int k = 0; k < NS; ++k)
#pragma unroll
                        for (int v = 0; v < 4; ++v)
                            if (poll[k] && v < nv && (accept || !is_set(U[k][v]))) {
                                U[k][v] = ld_sector_strong(up[k] + s0 + 4 * v);
                                ok &= accept || is_set(U[k][v]);
                            }
                    if (__all_sync(RR_FULL_MASK, ok)) break;
                    // another upstream block is later than the watched one: keep going, gently
                    if ((++spins & 255u) == 0) {
                        bool fin = true;
#pragma unroll
                        for (int k = 0; k < NS; ++k)
                            if (poll[k]) fin &= ld_acquire(c.done + (c.up_u[k] >> 5)) >= full_want;
                        if (__all_sync(RR_FULL_MASK, fin)) accept = true;
                    }
                    if (P.spin_ns) __nanosleep(64);
                }
#ifdef RR_TRACE
                if (lane == 0 && P.prof) P.prof[(((size_t)c.b * ((size_t)P.n_tiles * P.gpt) + (size_t)(gbase + (s0 >> 4))) * RR_NEV + 0) * 2 + 1] = spins;
#endif
            }
        }
        TR(c.b, gbase + (s0 >> 4), 1);
        if (LAT_SMEM) asm volatile("cp.async.wait_group 0;" ::: "memory");
#pragma unroll
        for (int v = 0; v < 4; ++v) {
            const int s = s0 + 4 * v;
            if (v < nv) {
                double2 *bp0 = reinterpret_cast<double2 *>(stage + buf_pair(2 * v, lane));
                double2 *bp1 = reinterpret_cast<double2 *>(stage + buf_pair(2 * v + 1, lane));
                d4 lfar = d4{0, 0, 0, 0};
                if (LAT_SMEM) {
                    const double2 x = *bp0, y = *bp1;
                    lcur = d4{x.x, x.y, y.x, y.y};
                    if (!c.valid) lcur = d4{0, 0, 0, 0};
                } else {
                    lfar = lat_group(s + 8);
                }
                double r = c3 * q;                                       // _numba_kernels.py:27-28 / :68-69
                if (HAS_LAT) r = fma(c4, lcur.a, r);
#pragma unroll
                for (int k = 0; k < NS; ++k) r = fma(c2, old[k], r);     // :29-33 / :70-74, ascending upstream
#pragma unroll
                for (int k = 0; k < NS; ++k) r = fma(c1, U[k][v].a, r);  // :36-39 / :75-78 (lhs_off = -c1)
                const double r0 = r;
                if (v == 0) TR_AFTER(r0, c.b, gbase + (s0 >> 4), 2);
                r = c3 * r0;
                if (HAS_LAT) r = fma(c4, lcur.b, r);
#pragma unroll
                for (int k = 0; k < NS; ++k) r = fma(c2, U[k][v].a, r);
#pragma unroll
                for (int k = 0; k < NS; ++k) r = fma(c1, U[k][v].b, r);
                const double r1 = r;
                r = c3 * r1;
                if (HAS_LAT) r = fma(c4, lcur.c, r);
#pragma unroll
                for (int k = 0; k < NS; ++k) r = fma(c2, U[k][v].b, r);
#pragma unroll
                for (int k = 0; k < NS; ++k) r = fma(c1, U[k][v].c, r);
                const double r2 = r;
                r = c3 * r2;
                if (HAS_LAT) r = fma(c4, lcur.d, r);
#pragma unroll
                for (int k = 0; k < NS; ++k) r = fma(c2, U[k][v].c, r);
#pragma unroll
                for (int k = 0; k < NS; ++k) r = fma(c1, U[k][v].d, r);
                const double r3 = r;
                *bp0 = make_double2(r0, r1);                             // in place of the lateral entries just used
                *bp1 = make_double2(r2, r3);
                q = (s + 3 < TT) ? r3 : ((s + 2 < TT) ? r2 : ((s + 1 < TT) ? r1 : r0));
#pragma unroll
                for (int k = 0; k < NS; ++k) old[k] = U[k][v].d;
                if (!LAT_SMEM) { lcur = lnxt; lnxt = lfar; }
            }
        }
        jitter_delay(P.jitter, c.b, j, 1 + (s0 >> 4));
        TR_AFTER(q, c.b, gbase + (s0 >> 4), 3);
        if (c.valid) {
            // one whole line (or the tail of the tile) of this reach's series; entries past TT inside the last sector are
            // never used (consumers and stage_out stop at TT)
            double *o = c.out0 + s0;
#pragma unroll
            for (int v = 0; v < 4; ++v)
                if (v < nv) {
                    const double2 x = *reinterpret_cast<const double2 *>(stage + buf_pair(2 * v, lane));
                    const double2 y = *reinterpret_cast<const double2 *>(stage + buf_pair(2 * v + 1, lane));
                    st_sector_strong(o + 4 * v, x.x, x.y, y.x, y.y);
                }
        }
        if (s0 + 16 < TT) stage_lateral(s0 + 16);      // lands while the warp waits for the next group's upstream entries
        TR(c.b, gbase + (s0 >> 4), 4);
    }
    if (c.valid) P.q_state[c.m][c.i] = q;
}


// -----------------------------------------------------------------------------------------------------------------
// UnitMuskingum (unit_route, _numba_kernels.py:88-171) in the same pipeline.  Headwater reaches (level 0) pass their
// convolved lateral inflow through (:122-123) and never enter the wavefront: their blocks are left out of the schedule
// and stage_out writes their rows.  An inner reach reads, per upstream reach, its lateral series (lateral tiles) and --
// for inner upstreams -- its q_ch series (discharge tiles, raw); q_full of an upstream before a step is its q_ch plus its
// lateral of the previous step (:165).  The discharge tiles hold q_ch; stage_out forms max(q_ch + lateral, 0) (:165-171).
// -----------------------------------------------------------------------------------------------------------------
template <int NS>
__device__ __forceinline__ void unit_item(const rr_route_params &P, const dctx &c, double qf, double *stage) {
    constexpr int NA = NS > 0 ? NS : 1;
    const double c1 = c.c1, c2 = c.c2, c3 = c.c3;
    const int TT = c.TT, j = c.j, lane = c.lane;
    const int32_t gbase = j * P.gpt;
    const bool inner = c.deg > 0;
    double q = c.q;
    const double *ex[NA], *lu[NA];
    bool has[NA], hw[NA];
    double qfo[NA];                 // upstream q_full before the next step
    d4 exn[NA], exf[NA], lun[NA];   // upstream q_ch: rows s.., s+4.. (s+8.. in flight); upstream lateral: rows s.. (s+4.. in flight)
    bool full = !c.prog;
#pragma unroll
    for (int k = 0; k < NS; ++k) {
        has[k] = k < c.deg;
        hw[k] = false;
        ex[k] = P.out[c.m];
        lu[k] = P.lateral[c.m];
        qfo[k] = 0.0;
        exn[k] = exf[k] = lun[k] = d4{0, 0, 0, 0};
        if (has[k]) {
            const int64_t u = c.up_u[k];
            hw[k] = u < P.hw_slots;
            lu[k] = tile_of(P.lateral[c.m], P, j, u);
            lun[k] = ld_sector_ro(lu[k]);
            if (!hw[k]) {
                ex[k] = tile_of(P.out[c.m], P, j, u);
                qfo[k] = j == 0 ? P.qf_init[(size_t)c.m * P.q_init_stride + u]
                                : tile_of(P.out[c.m], P, j - 1, u)[P.tile_rows - 1] + tile_of(P.lateral[c.m], P, j - 1, u)[P.tile_rows - 1];
                exn[k] = ld_sector(ex[k]);
                if (4 < TT) exf[k] = ld_sector(ex[k] + 4);
            }
        }
    }
    const double *lat = c.lat0;
    auto own = [&](int s0) -> d4 { return (c.valid && s0 < TT) ? ld_sector_ro(lat + s0) : d4{0, 0, 0, 0}; };
    d4 lcur = own(0), lnxt = own(4);
    double *st = stage + lane;
    for (int s = 0; s < TT; s += 4) {
        if (NS > 0 && !full && (s & 15) == 0 && s > 0) {
            wait_groups(c, gbase + (s >> 4) + 1, gbase + P.gpt, full);
#pragma unroll
            for (int k = 0; k < NS; ++k)
                if (has[k] && !hw[k]) {
                    exn[k] = ld_sector(ex[k] + s);
                    if (s + 4 < TT) exf[k] = ld_sector(ex[k] + s + 4);
                }
        }
        const bool ahead = full || ((s + 8) >> 4) == (s >> 4);
        d4 exr[NA], lur[NA];
#pragma unroll
        for (int k = 0; k < NS; ++k) {
            exr[k] = lur[k] = d4{0, 0, 0, 0};
            if (has[k] && s + 4 < TT) lur[k] = ld_sector_ro(lu[k] + s + 4);
            if (has[k] && !hw[k] && ahead && s + 8 < TT) exr[k] = ld_sector(ex[k] + s + 8);
        }
        const d4 lfar = own(s + 8);
        const double lv[4] = {lcur.a, lcur.b, lcur.c, lcur.d};
        double r4[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            double a_in = 0.0, a_hw = 0.0;                               // :126-139, ascending upstream per class
#pragma unroll
            for (int k = 0; k < NS; ++k) {
                const double l = u == 0 ? lun[k].a : (u == 1 ? lun[k].b : (u == 2 ? lun[k].c : lun[k].d));
                if (has[k]) { if (hw[k]) a_hw += l; else a_in += l; }
            }
            double r = c1 * (a_in + a_hw) + c2 * a_hw;                   // :142-143, :151
            r = r + c3 * q;
#pragma unroll
            for (int k = 0; k < NS; ++k)
                if (has[k] && !hw[k]) r = fma(c2, qfo[k], r);            // :152-156  c2 * q_full_old[upstream]
#pragma unroll
            for (int k = 0; k < NS; ++k) {
                const double qn = u == 0 ? exn[k].a : (u == 1 ? exn[k].b : (u == 2 ? exn[k].c : exn[k].d));
                if (has[k] && !hw[k]) r = fma(c1, qn, r);                // :159-162  lhs_off = -c1
            }
#pragma unroll
            for (int k = 0; k < NS; ++k) {
                const double qn = u == 0 ? exn[k].a : (u == 1 ? exn[k].b : (u == 2 ? exn[k].c : exn[k].d));
                const double l = u == 0 ? lun[k].a : (u == 1 ? lun[k].b : (u == 2 ? lun[k].c : lun[k].d));
                qfo[k] = qn + l;                                         // the upstream's q_full after this step (:165-166)
            }
            r4[u] = r;
            if (s + u < TT && inner) { q = r; qf = r + lv[u]; }
        }
        const int rr = s & 15;
        st[(rr + 0) * RR_BLOCK] = r4[0];
        st[(rr + 1) * RR_BLOCK] = r4[1];
        st[(rr + 2) * RR_BLOCK] = r4[2];
        st[(rr + 3) * RR_BLOCK] = r4[3];
        if (rr == 12 || s + 4 >= TT) {
            if (c.valid) {
                double *o = c.out0 + (s - rr);
#pragma unroll
                for (int v = 0; v < 16; v += 4)
                    if (v <= rr) st_sector(o + v, st[(v + 0) * RR_BLOCK], st[(v + 1) * RR_BLOCK], st[(v + 2) * RR_BLOCK], st[(v + 3) * RR_BLOCK]);
            }
            if (c.narrow && s + 4 < TT) {
                jitter_delay(P.jitter, c.b, j, 1 + (s >> 4));
                __syncwarp();
                if (lane == 0) st_release(c.done + c.b, gbase + (s >> 4) + 1);
            }
        }
#pragma unroll
        for (int k = 0; k < NS; ++k) { exn[k] = exf[k]; exf[k] = exr[k]; lun[k] = lur[k]; }
        lcur = lnxt;
        lnxt = lfar;
    }
    if (c.valid && inner) { P.q_state[c.m][c.i] = q; P.q_full[c.m][c.i] = qf; }
}

}  // namespace

template <int MAXNS>
__global__ void __launch_bounds__(256, 2) rr_direct_unit_kernel(const __grid_constant__ rr_route_params P) {
    __shared__ double stage_all[8][16 * RR_BLOCK];
    const int lane = threadIdx.x & 31;
    double *stage = stage_all[threadIdx.x >> 5];
    int m, b, j, dep_lo, dep_hi;
    while (next_ticket(P, lane, m, b, j, dep_lo, dep_hi)) {
        dctx c;
        const int64_t i = (int64_t)b * RR_BLOCK + lane;
        const bool valid = i < P.n;
        const int64_t ic = valid ? i : P.n - 1;
        c.m = m; c.b = b; c.j = j; c.lane = lane; c.i = i; c.valid = valid;
        c.c1 = __ldg(P.c1 + ic); c.c2 = __ldg(P.c2 + ic); c.c3 = __ldg(P.c3 + ic); c.c4 = 0.0;
        const int e0 = __ldg(P.up_ptr + ic);
        c.deg = valid ? __ldg(P.up_ptr + ic + 1) - e0 : 0;
        const rr_blk_meta M = P.meta[b];
        c.narrow = (M.int_mask & RR_META_NARROW) != 0;
        c.TT = min(P.tile_rows, P.T - j * P.tile_rows);
        c.dep_blk = dep_lo + lane < dep_hi ? __ldg(P.dep_idx + dep_lo + lane) : -1;
        c.dep_more = dep_lo + 32 + lane; c.dep_hi = dep_hi; c.dep_idx = P.dep_idx; c.spin_ns = P.spin_ns;
#pragma unroll
        for (int k = 0; k < MAXNS; ++k) c.up_u[k] = k < c.deg ? __ldg(P.up_idx + e0 + k) : 0;
        c.done = P.done + (size_t)m * P.n_blocks;
        c.lat0 = tile_of(P.lateral[m], P, j, i);
        c.out0 = const_cast<double *>(tile_of(P.out[m], P, j, i));
        const int32_t full_want = (j + 1) * P.gpt;
        jitter_delay(P.jitter, b, j, 100);
        if (lane == 0 && j > 0) wait_ge(c.done + b, j * P.gpt);
        c.prog = false;
        if (c.narrow && dep_hi > dep_lo) {
            bool full = false;
            wait_groups(c, j * P.gpt + 1, full_want, full);
            c.prog = !full;
        } else {
            if (c.dep_blk >= 0) wait_ge(c.done + c.dep_blk, full_want);
            for (int e = dep_lo + 32 + lane; e < dep_hi; e += 32) wait_ge(c.done + __ldg(P.dep_idx + e), full_want);
        }
        __syncwarp();
        c.q = 0.0;
        double qf = 0.0;
        if (valid) {
            c.q = (j == 0) ? P.q_init[(size_t)m * P.q_init_stride + i] : P.q_state[m][i];
            qf = (j == 0) ? P.qf_init[(size_t)m * P.q_init_stride + i] : P.q_full[m][i];
        }
        if (MAXNS <= 2) {
            switch (M.max_deg) {
                case 0: unit_item<0>(P, c, qf, stage); break;
                case 1: unit_item<1>(P, c, qf, stage); break;
                default: unit_item<2>(P, c, qf, stage); break;
            }
        } else {
            switch (M.max_deg) {
                case 0: unit_item<0>(P, c, qf, stage); break;
                case 1: unit_item<1>(P, c, qf, stage); break;
                case 2: unit_item<2>(P, c, qf, stage); break;
                case 3: unit_item<3>(P, c, qf, stage); break;
                default: unit_item<RR_MAX_FAST_DEG>(P, c, qf, stage); break;
            }
        }
        jitter_delay(P.jitter, b, j, 200);
        __syncwarp();
        if (lane == 0) st_release(c.done + b, full_want);
        __syncwarp();
    }
}

namespace {
}  // namespace

// MAXNS: largest in-degree of the network, 2 or RR_MAX_FAST_DEG.  Networks with confluences of three or four rivers get
// a kernel of their own so that the register-hungry instantiations do not set the register allocation -- and the
// spills -- of the common case (at most two upstream reaches).
template <int MODE, int MAXNS, bool SUB, bool SENT>
__global__ void __launch_bounds__(256, 2) rr_direct_kernel(const __grid_constant__ rr_route_params P) {
    __shared__ double stage_all[8][16 * RR_BLOCK];
    constexpr bool HAS_LAT = (MODE == RR_MODE_RAPID);
    const int lane = threadIdx.x & 31;
    double *stage = stage_all[threadIdx.x >> 5];
    int m, b, j, dep_lo, dep_hi;
    while (next_ticket(P, lane, m, b, j, dep_lo, dep_hi)) {
        dctx c;
        const int64_t i = (int64_t)b * RR_BLOCK + lane;
        const bool valid = i < P.n;
        const int64_t ic = valid ? i : P.n - 1;
        c.m = m; c.b = b; c.j = j; c.lane = lane; c.i = i; c.valid = valid;
        c.c1 = __ldg(P.c1 + ic); c.c2 = __ldg(P.c2 + ic); c.c3 = __ldg(P.c3 + ic);
        c.c4 = HAS_LAT ? __ldg(P.c4 + ic) : 0.0;
        const int e0 = __ldg(P.up_ptr + ic);
        c.deg = valid ? __ldg(P.up_ptr + ic + 1) - e0 : 0;
        const rr_blk_meta M = P.meta[b];
        c.narrow = (M.int_mask & RR_META_NARROW) != 0;
        const int t0 = j * P.tile_rows;
        c.TT = min(P.tile_rows, P.T - t0) * (SUB ? P.K : 1);   // routing substeps in this tile
        c.dep_blk = dep_lo + lane < dep_hi ? __ldg(P.dep_idx + dep_lo + lane) : -1;
        c.dep_more = dep_lo + 32 + lane; c.dep_hi = dep_hi; c.dep_idx = P.dep_idx; c.spin_ns = P.spin_ns;
#pragma unroll
        for (int k = 0; k < MAXNS; ++k) c.up_u[k] = k < c.deg ? __ldg(P.up_idx + e0 + k) : 0;
        c.done = P.done + (size_t)m * P.n_blocks;
        c.lat0 = HAS_LAT ? lat_tile_of(P.lateral[m], P, j, i) : nullptr;
        c.out0 = const_cast<double *>(tile_of(P.out[m], P, j, i));
        // ---- dependencies: own previous tile complete; upstream blocks complete, or (narrow levels with at most 32
        //      upstream blocks) their first group published ----
        const int32_t full_want = (j + 1) * P.gpt;
        jitter_delay(P.jitter, b, j, 100);
        if (lane == 0 && j > 0) wait_ge(c.done + b, j * P.gpt);
        c.prog = false;
        if (SENT) {
            // small networks (every level narrow): upstream blocks hand their series over entry by entry (narrow_item); only
            // upstream blocks outside that protocol (routed by the staging kernel) must have finished the tile
            for (int e = dep_lo + lane; e < dep_hi; e += 32) {
                const int32_t db = __ldg(P.dep_idx + e);
                if (!(db >= P.poll_lo && (P.meta[db].int_mask & RR_META_NARROW) != 0)) wait_ge(c.done + db, full_want);
            }
            __syncwarp();
            c.q = 0.0;
            if (valid) c.q = (j == 0) ? P.q_init[(size_t)m * P.q_init_stride + i] : P.q_state[m][i];
            if (MAXNS <= 2) {
                switch (M.max_deg) {
                    case 0: narrow_item<MODE, 0, SUB>(P, c, stage); break;
                    case 1: narrow_item<MODE, 1, SUB>(P, c, stage); break;
                    default: narrow_item<MODE, 2, SUB>(P, c, stage); break;
                }
            } else {
                switch (M.max_deg) {
                    case 0: narrow_item<MODE, 0, SUB>(P, c, stage); break;
                    case 1: narrow_item<MODE, 1, SUB>(P, c, stage); break;
                    case 2: narrow_item<MODE, 2, SUB>(P, c, stage); break;
                    case 3: narrow_item<MODE, 3, SUB>(P, c, stage); break;
                    default: narrow_item<MODE, RR_MAX_FAST_DEG, SUB>(P, c, stage); break;
                }
            }
        } else {
        if (c.narrow && dep_hi > dep_lo) {
            bool full = false;
            wait_groups(c, j * P.gpt + 1, full_want, full);
            c.prog = !full;
        } else {
            if (c.dep_blk >= 0) wait_ge(c.done + c.dep_blk, full_want);
            for (int e = dep_lo + 32 + lane; e < dep_hi; e += 32) wait_ge(c.done + __ldg(P.dep_idx + e), full_want);
        }
        __syncwarp();
        c.q = 0.0;
        if (valid) c.q = (j == 0) ? P.q_init[(size_t)m * P.q_init_stride + i] : P.q_state[m][i];
        if (MAXNS <= 2) {
            switch (M.max_deg) {
                case 0: direct_item<MODE, 0, SUB>(P, c, stage); break;
                case 1: direct_item<MODE, 1, SUB>(P, c, stage); break;
                default: direct_item<MODE, 2, SUB>(P, c, stage); break;
            }
        } else {
            switch (M.max_deg) {
                case 0: direct_item<MODE, 0, SUB>(P, c, stage); break;
                case 1: direct_item<MODE, 1, SUB>(P, c, stage); break;
                case 2: direct_item<MODE, 2, SUB>(P, c, stage); break;
                case 3: direct_item<MODE, 3, SUB>(P, c, stage); break;
                default: direct_item<MODE, RR_MAX_FAST_DEG, SUB>(P, c, stage); break;
            }
        }
        }
        jitter_delay(P.jitter, b, j, 200);
        __syncwarp();
        if (lane == 0) st_release(c.done + b, full_want);
        __syncwarp();
    }
}

// sentinel != 0: the hand-over of small networks (narrow_item); the kernels without it are the round's bandwidth kernels
// unchanged, instruction for instruction
cudaError_t rr_launch_direct(int mode, int max_deg, const rr_route_params &P, int grid, cudaStream_t stream, int sentinel) {
    const bool wide = max_deg > 2, sub = P.K > 1;
#define RR_LAUNCH2(M, S) do {                                                                               \
        if (wide) { if (sub) rr_direct_kernel<M, RR_MAX_FAST_DEG, true, S><<<grid, 256, 0, stream>>>(P);  \
                    else rr_direct_kernel<M, RR_MAX_FAST_DEG, false, S><<<grid, 256, 0, stream>>>(P); }   \
        else { if (sub) rr_direct_kernel<M, 2, true, S><<<grid, 256, 0, stream>>>(P);                     \
               else rr_direct_kernel<M, 2, false, S><<<grid, 256, 0, stream>>>(P); }                      \
    } while (0)
#define RR_LAUNCH(M) do { if (sentinel) RR_LAUNCH2(M, true); else RR_LAUNCH2(M, false); } while (0)
    if (mode == RR_MODE_UNIT) {
        if (sub) return cudaErrorInvalidValue;
        if (wide) rr_direct_unit_kernel<RR_MAX_FAST_DEG><<<grid, 256, 0, stream>>>(P);
        else rr_direct_unit_kernel<2><<<grid, 256, 0, stream>>>(P);
    } else if (mode == RR_MODE_MUSKINGUM) RR_LAUNCH(RR_MODE_MUSKINGUM);
    else if (mode == RR_MODE_RAPID) RR_LAUNCH(RR_MODE_RAPID);
    else return cudaErrorInvalidValue;
#undef RR_LAUNCH
#undef RR_LAUNCH2
    return cudaGetLastError();
}

int rr_direct_occupancy(int mode, int max_deg) {
    int nb = 0;
    const bool wide = max_deg > 2;
    cudaError_t e;
    if (mode == RR_MODE_UNIT)
        e = wide ? cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, rr_direct_unit_kernel<RR_MAX_FAST_DEG>, 256, 0)
                 : cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, rr_direct_unit_kernel<2>, 256, 0);
    else if (mode == RR_MODE_MUSKINGUM)   // (the substep instantiations have the same launch bounds; 2 CTAs per SM either way)
        e = wide ? cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, rr_direct_kernel<RR_MODE_MUSKINGUM, RR_MAX_FAST_DEG, true, true>, 256, 0)
                 : cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, rr_direct_kernel<RR_MODE_MUSKINGUM, 2, true, true>, 256, 0);
    else
        e = wide ? cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, rr_direct_kernel<RR_MODE_RAPID, RR_MAX_FAST_DEG, true, true>, 256, 0)
                 : cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, rr_direct_kernel<RR_MODE_RAPID, 2, true, true>, 256, 0);
    return e == cudaSuccess ? nb : -1;
}

// -----------------------------------------------------------------------------------------------------------------
// stage_in / stage_out
// -----------------------------------------------------------------------------------------------------------------
namespace {

__device__ __forceinline__ int64_t tile_index(int64_t t, int64_t k, int64_t tile_rows, int64_t pitch, int64_t n_blocks) {
    const int64_t j = t / tile_rows, r = t - j * tile_rows;
    return ((j * n_blocks + (k >> 5)) * RR_BLOCK + (k & 31)) * pitch + r;
}

// One thread per river segment of the caller's array (coalesced reads of the caller's rows), 16 rows per iteration:
// every store is one whole 128-byte line of the segment's series.  Segments whose working index is below hw_cut are
// headwaters in whole-headwater blocks: their recursion q' = c3*q + c4_dt*ql (_numba_kernels.py:68-69 with no
// upstream terms) runs here and their RAW discharge series goes to the discharge tiles instead.
// ST = float: lateral inflows stored as float32 (qlateral files may be; the reference upcasts them with
// astype(float64), TransformMuskingum.py:36 -- the conversion is exact, so doing it here changes no bit).
template <bool ROUTE_HW, typename ST>
__global__ void __launch_bounds__(256) stage_in_kernel(const ST *__restrict__ src, int64_t lds, double *__restrict__ lat_w,
                                                       double *__restrict__ out_w, const int32_t *__restrict__ inv, int64_t n,
                                                       int64_t T, int64_t tile_rows, int64_t pitch, int64_t n_blocks,
                                                       int64_t hw_cut, const double *__restrict__ c3, const double *__restrict__ c4,
                                                       const double *__restrict__ q_init, double *__restrict__ q_final,
                                                       int64_t rows_per_slice) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const int64_t k = __ldg(inv + i);
    const bool hw = ROUTE_HW && k < hw_cut;
    // plain copies split time over grid.y; with headwater routing every thread walks the whole call (a headwater's rows
    // are a recursion, and letting its neighbours take other slices would read each sector of the caller's rows twice)
    const int64_t ta = (int64_t)blockIdx.y * rows_per_slice, tb = min(T, ta + rows_per_slice);
    double q = 0.0, a3 = 0.0, a4 = 0.0;
    if (hw) { q = q_init[k]; a3 = __ldg(c3 + k); a4 = __ldg(c4 + k); }
    double *dst = hw ? out_w : lat_w;
    for (int64_t t0 = ta; t0 < tb; t0 += 16) {
        double v[16];
#pragma unroll
        for (int r = 0; r < 16; ++r) v[r] = (t0 + r < T) ? (double)__ldg(src + (t0 + r) * lds + i) : 0.0;
        if (hw) {
#pragma unroll
            for (int r = 0; r < 16; ++r)
                if (t0 + r < T) { q = fma(a4, v[r], a3 * q); v[r] = q; }
        }
        double *p = dst + tile_index(t0, k, tile_rows, pitch, n_blocks);
#pragma unroll
        for (int r = 0; r < 16; r += 4) st_sector(p + r, v[r], v[r + 1], v[r + 2], v[r + 3]);
    }
    if (hw) q_final[k] = q;
}

// The stage_out kernels take one row group (or time tile) per grid row.  grid.y is capped at 65535; a call with more
// groups launches the STRIDE instantiation, whose CTAs stride over them by gridDim.y.  Without STRIDE the loop body runs
// once and compiles to the one-group-per-CTA code, with its registers and occupancy.

// working discharge tiles -> caller's rows: column s of the output shows segment subset[s] (or s); clamp as the
// reference does on the interval mean (K == 1: the value itself); OT = float rounds like numpy's astype(float32)
template <typename OT, bool STRIDE>
__global__ void __launch_bounds__(256) stage_out_kernel(const double *__restrict__ out_w, OT *__restrict__ dst, int64_t ldd,
                                                        const int32_t *__restrict__ inv, const int32_t *__restrict__ subset,
                                                        int64_t n_out, int64_t T, int64_t tile_rows, int64_t pitch,
                                                        int64_t n_blocks) {
    const int64_t s = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= n_out) return;
    const int64_t i = subset ? (int64_t)__ldg(subset + s) : s;
    const int64_t k = __ldg(inv + i);
    int64_t t0 = (int64_t)blockIdx.y * 16;
    do {
        const double *p = out_w + tile_index(t0, k, tile_rows, pitch, n_blocks);
        double v[16];
#pragma unroll
        for (int r = 0; r < 16; r += 4) {
            const d4 x = ld_sector_ro(p + r);
            v[r] = x.a; v[r + 1] = x.b; v[r + 2] = x.c; v[r + 3] = x.d;
        }
#pragma unroll
        for (int r = 0; r < 16; ++r)
            if (t0 + r < T) {
                const double val = v[r] > 0.0 ? v[r] : 0.0;              // _numba_kernels.py:44-46 / :82-84
                dst[(t0 + r) * ldd + s] = (OT)val;
            }
    } while (STRIDE && (t0 += (int64_t)gridDim.y * 16) < T);
}

// More than one routing substep per row: the tiles hold the raw substep series; an output row is the clamped mean of its K
// substeps, accumulated in substep order and multiplied by 1/K exactly as _numba_kernels.py:19, :41-46 / :60, :79-84 do.
template <typename OT, bool STRIDE>
__global__ void __launch_bounds__(256) stage_out_sub_kernel(const double *__restrict__ out_w, OT *__restrict__ dst, int64_t ldd,
                                                            const int32_t *__restrict__ inv, const int32_t *__restrict__ subset,
                                                            int64_t n_out, int64_t T, int64_t tile_rows, int64_t pitch,
                                                            int64_t n_blocks, int K) {
    const int64_t s = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= n_out) return;
    const int64_t i = subset ? (int64_t)__ldg(subset + s) : s;
    const int64_t k = __ldg(inv + i);
    const double inv_k = 1.0 / (double)K;
    const int64_t n_tiles = (T + tile_rows - 1) / tile_rows;
    int64_t j = blockIdx.y;
    do {   // one time tile per grid row
        const double *p = out_w + ((j * n_blocks + (k >> 5)) * RR_BLOCK + (k & 31)) * pitch;
        const int64_t t0 = j * tile_rows, rows = min(tile_rows, T - t0);
        for (int64_t r = 0; r < rows; ++r) {
            double acc = 0.0;
            for (int q = 0; q < K; ++q) acc += p[r * K + q];
            const double val = acc * inv_k;
            dst[(t0 + r) * ldd + s] = (OT)(val > 0.0 ? val : 0.0);
        }
    } while (STRIDE && (j += gridDim.y) < n_tiles);
}

// UnitMuskingum: the discharge tiles hold q_ch of the inner reaches.  Output = the convolved lateral inflow itself for
// headwaters (unclamped, _numba_kernels.py:122-123), max(q_ch + lateral, 0) for inner reaches (:165-171, one substep
// per row); the lateral rows are read from the caller's array (coalesced, column i = segment i).
template <typename OT, bool STRIDE>
__global__ void __launch_bounds__(256) stage_out_unit_kernel(const double *__restrict__ out_w, const double *__restrict__ lat,
                                                             int64_t ldl, OT *__restrict__ dst, int64_t ldd,
                                                             const int32_t *__restrict__ inv, const int32_t *__restrict__ subset,
                                                             int64_t n_out, int64_t T, int64_t tile_rows, int64_t pitch,
                                                             int64_t n_blocks, int64_t hw_slots) {
    const int64_t s = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= n_out) return;
    const int64_t i = subset ? (int64_t)__ldg(subset + s) : s;
    const int64_t k = __ldg(inv + i);
    const bool hw = k < hw_slots;
    int64_t t0 = (int64_t)blockIdx.y * 16;
    do {
        double v[16];
#pragma unroll
        for (int r = 0; r < 16; ++r) v[r] = 0.0;
        if (!hw) {
            const double *p = out_w + tile_index(t0, k, tile_rows, pitch, n_blocks);
#pragma unroll
            for (int r = 0; r < 16; r += 4) {
                const d4 x = ld_sector_ro(p + r);
                v[r] = x.a; v[r + 1] = x.b; v[r + 2] = x.c; v[r + 3] = x.d;
            }
        }
#pragma unroll
        for (int r = 0; r < 16; ++r)
            if (t0 + r < T) {
                const double l = __ldg(lat + (t0 + r) * ldl + i);
                double val = l;
                if (!hw) { val = v[r] + l; val = val > 0.0 ? val : 0.0; }
                dst[(t0 + r) * ldd + s] = (OT)val;
            }
    } while (STRIDE && (t0 += (int64_t)gridDim.y * 16) < T);
}

// UnitMuskingum state hand-back in the caller's order.  last != 0: the recombined vector of UnitMuskingum.py:94-98
// (headwaters: lateral inflow of the last row, inner: q_full).  Otherwise the kernel-level pair: q_ch and q_full of the
// inner reaches; headwater entries are left untouched.
__global__ void __launch_bounds__(256) unit_state_kernel(const double *__restrict__ qs_w, const double *__restrict__ qf_w,
                                                         const int32_t *__restrict__ inv, int64_t n, int64_t hw_slots, int last,
                                                         const double *__restrict__ lat_last, double *__restrict__ q_state,
                                                         double *__restrict__ q_full) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const int64_t k = __ldg(inv + i);
    if (k < hw_slots) {
        if (last) q_state[i] = __ldg(lat_last + i);
        return;
    }
    if (last) q_state[i] = qf_w[k];
    else { q_state[i] = qs_w[k]; q_full[i] = qf_w[k]; }
}

}  // namespace

#define CKD(call)                                                                                  \
    do {                                                                                           \
        cudaError_t e_ = (call);                                                                   \
        if (e_ != cudaSuccess) {                                                                   \
            rr_set_error(std::string(#call) + ": " + cudaGetErrorString(e_));                      \
            return 200;                                                                            \
        }                                                                                          \
    } while (0)

// Discharge tiles of the narrow blocks of one member <- the "not written yet" pattern (narrow_item).  One CTA per
// (narrow block, tile): the block's tile is 32 x pitch contiguous doubles.  grid.y is capped at 65535: with more tiles
// a CTA strides over them (STRIDE).
template <bool STRIDE>
__global__ void __launch_bounds__(256) fill_sentinel_kernel(double *__restrict__ out_w, const int32_t *__restrict__ narrow_blocks,
                                                            int32_t first_block, int64_t n_blocks, int64_t n_tiles, int64_t pitch) {
    const int32_t b = __ldg(narrow_blocks + blockIdx.x);
    if (b < first_block) return;
    const double sv = __longlong_as_double((long long)RR_SENTINEL_BITS);
    int64_t j = blockIdx.y;
    do {
        double *p = out_w + (((size_t)j * n_blocks + (size_t)b) * RR_BLOCK) * (size_t)pitch;
        for (int64_t e = (int64_t)threadIdx.x * 4; e < RR_BLOCK * pitch; e += 256 * 4) st_sector(p + e, sv, sv, sv, sv);
    } while (STRIDE && (j += gridDim.y) < n_tiles);
}

int rr_fill_sentinel(double *out_w, const int32_t *narrow_blocks, int64_t n_narrow, int64_t first_block, int64_t n_blocks,
                     int64_t n_tiles, int64_t pitch, cudaStream_t stream) {
    if (n_narrow <= 0) return 0;
    dim3 grid((unsigned)n_narrow, (unsigned)std::min<int64_t>(n_tiles, 65535));
    if (n_tiles > 65535) fill_sentinel_kernel<true><<<grid, 256, 0, stream>>>(out_w, narrow_blocks, (int32_t)first_block, n_blocks, n_tiles, pitch);
    else fill_sentinel_kernel<false><<<grid, 256, 0, stream>>>(out_w, narrow_blocks, (int32_t)first_block, n_blocks, n_tiles, pitch);
    CKD(cudaGetLastError());
    rr_count_launch(1);
    return 0;
}

// tile_rows must be a multiple of 16 (the caller checks).  hw_cut = 0 copies every segment's lateral inflows.
int rr_stage_in(const void *src, int src_f32, int64_t lds, double *lat_w, double *out_w, const int32_t *inv, int64_t n, int64_t T,
                int64_t tile_rows, int64_t n_blocks, int64_t hw_cut, const double *c3, const double *c4,
                const double *q_init, double *q_final, int sm_count, cudaStream_t stream) {
    const int64_t pitch = (tile_rows + 3) & ~(int64_t)3;
    const unsigned gx = (unsigned)((n + 255) / 256);
    // enough slices to fill the machine a few times over, each a whole number of 16-row groups
    int64_t slices = std::max<int64_t>(1, std::min<int64_t>((T + 15) / 16, ((int64_t)sm_count * 8 * 4 + gx - 1) / gx));
    if (hw_cut > 0) slices = 1;
    int64_t rows_per_slice = (((T + slices - 1) / slices + 15) / 16) * 16;
    slices = (T + rows_per_slice - 1) / rows_per_slice;
    dim3 grid(gx, (unsigned)slices);
#define STAGE_IN(HW, ST) stage_in_kernel<HW, ST><<<grid, 256, 0, stream>>>((const ST *)src, lds, lat_w, out_w, inv, n, T, tile_rows, \
                                                                          pitch, n_blocks, hw_cut, c3, c4, q_init, q_final, rows_per_slice)
    if (hw_cut > 0) { if (src_f32) STAGE_IN(true, float); else STAGE_IN(true, double); }
    else { if (src_f32) STAGE_IN(false, float); else STAGE_IN(false, double); }
#undef STAGE_IN
    CKD(cudaGetLastError());
    rr_count_launch(1);
    return 0;
}

int rr_stage_out(const double *out_w, void *dst, int dst_f32, int64_t ldd, const int32_t *inv, const int32_t *subset,
                 int64_t n_out, int64_t T, int64_t tile_rows, int64_t n_blocks, cudaStream_t stream) {
    const int64_t pitch = (tile_rows + 3) & ~(int64_t)3;
    dim3 grid((unsigned)((n_out + 255) / 256), (unsigned)std::min<int64_t>((T + 15) / 16, 65535));
#define STAGE_OUT(OT, S) stage_out_kernel<OT, S><<<grid, 256, 0, stream>>>(out_w, (OT *)dst, ldd, inv, subset, n_out, T, tile_rows, pitch, n_blocks)
    if ((T + 15) / 16 > 65535) { if (dst_f32) STAGE_OUT(float, true); else STAGE_OUT(double, true); }
    else { if (dst_f32) STAGE_OUT(float, false); else STAGE_OUT(double, false); }
#undef STAGE_OUT
    CKD(cudaGetLastError());
    rr_count_launch(1);
    return 0;
}

int rr_stage_out_unit(const double *out_w, const double *lat, int64_t ldl, void *dst, int dst_f32, int64_t ldd, const int32_t *inv,
                      const int32_t *subset, int64_t n_out, int64_t T, int64_t tile_rows, int64_t n_blocks, int64_t hw_slots,
                      cudaStream_t stream) {
    const int64_t pitch = (tile_rows + 3) & ~(int64_t)3;
    dim3 grid((unsigned)((n_out + 255) / 256), (unsigned)std::min<int64_t>((T + 15) / 16, 65535));
#define STAGE_OUT(OT, S) stage_out_unit_kernel<OT, S><<<grid, 256, 0, stream>>>(out_w, lat, ldl, (OT *)dst, ldd, inv, subset, n_out, T, \
                                                                             tile_rows, pitch, n_blocks, hw_slots)
    if ((T + 15) / 16 > 65535) { if (dst_f32) STAGE_OUT(float, true); else STAGE_OUT(double, true); }
    else { if (dst_f32) STAGE_OUT(float, false); else STAGE_OUT(double, false); }
#undef STAGE_OUT
    CKD(cudaGetLastError());
    rr_count_launch(1);
    return 0;
}

int rr_unit_state_to_user(const double *qs_w, const double *qf_w, const int32_t *inv, int64_t n, int64_t hw_slots, int last,
                          const double *lat_last, double *q_state, double *q_full, cudaStream_t stream) {
    unit_state_kernel<<<(unsigned)((n + 255) / 256), 256, 0, stream>>>(qs_w, qf_w, inv, n, hw_slots, last, lat_last, q_state, q_full);
    CKD(cudaGetLastError());
    rr_count_launch(1);
    return 0;
}

int rr_stage_out_sub(const double *out_w, void *dst, int dst_f32, int64_t ldd, const int32_t *inv, const int32_t *subset,
                     int64_t n_out, int64_t T, int64_t tile_rows, int64_t pitch, int64_t n_blocks, int K, cudaStream_t stream) {
    dim3 grid((unsigned)((n_out + 255) / 256), (unsigned)std::min<int64_t>((T + tile_rows - 1) / tile_rows, 65535));
#define STAGE_OUT(OT, S) stage_out_sub_kernel<OT, S><<<grid, 256, 0, stream>>>(out_w, (OT *)dst, ldd, inv, subset, n_out, T, tile_rows, pitch, n_blocks, K)
    if ((T + tile_rows - 1) / tile_rows > 65535) { if (dst_f32) STAGE_OUT(float, true); else STAGE_OUT(double, true); }
    else { if (dst_f32) STAGE_OUT(float, false); else STAGE_OUT(double, false); }
#undef STAGE_OUT
    CKD(cudaGetLastError());
    rr_count_launch(1);
    return 0;
}
