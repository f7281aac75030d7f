// Internal declarations shared by the host plan builder and the CUDA translation units.
#pragma once
#include <cstdint>
#include <string>
#include <vector>

#include "rr_b200.h"

#define RR_BLOCK 32          // reaches per block == lanes per warp
#define RR_MAX_FAST_DEG 4    // upstream slots held in registers by the kernel
#define RR_SLOT_HW_BIT 0x40000000  // external slot: upstream reach is a headwater (in-degree 0)
#define RR_META_FAST 0x40    // rr_blk_meta::int_mask: no in-block edges, in-degree <= RR_MAX_FAST_DEG
#define RR_META_NARROW 0x20  // rr_blk_meta::int_mask: fewer than RR_NARROW_BLOCKS blocks in the block's level -- launches are
                             // dependency-latency bound there: such blocks publish and consume progress per 16-row group
#define RR_NARROW_BLOCKS 4096
#define RR_SENTINEL_MAX_BLOCKS 4096   // networks of at most this many blocks use the sentinel hand-over (rr_direct.cu, narrow_item)
#define RR_FLAG_ROWS 16      // direct kernel: rows per progress unit of done[] (one 128-byte line of a reach's series)

void rr_set_error(const std::string &msg);

// Per-block metadata packed for one 8-byte load by the kernel.
struct rr_blk_meta {
    uint16_t max_deg;     // largest in-degree of a lane
    uint8_t max_skew;     // largest systolic delay in the block
    uint8_t int_mask;     // bit k (k < RR_MAX_FAST_DEG): some lane's k-th upstream is in-block;
                          // bit 7: some lane has an in-block upstream at slot >= RR_MAX_FAST_DEG;
                          // bit 6 (0x40): fast-path eligible; bit 5 (0x20): the block's level is narrow
    int32_t level;        // level in the block dependency DAG
};

struct rr_device_state;  // defined in rr_api.cu

struct rr_plan {
    int64_t n = 0, n_edges = 0, n_blocks = 0, n_export = 0, n_internal = 0, n_outlets = 0;
    int64_t n_work = 0;              // working slots: n, or more when a renumbered plan pads every level to whole blocks
    int64_t lvl0_slots = 0;          // renumbered plans: slots of level 0 (whole blocks of headwaters and padding); else 0
    int64_t n_hw = 0;                // reaches without upstream (level 0)
    bool all_fast = false;           // every block is fast-path eligible (RR_META_FAST)
    rr_plan_opts opts{};
    std::vector<int32_t> down;       // [n_work] downstream slot in the WORKING order (user order unless renumbered)
    std::vector<int32_t> perm, inv;  // renumbered plans: perm[working slot] = user index (-1: padding), inv[user] = slot
    int32_t reach_depth = 0;         // longest upstream-to-outlet path, in reaches
    bool auto_tile = true;           // choose the tile length per call (opts.time_tile is then the largest one)
    std::vector<int32_t> up_ptr;     // [n+1]
    std::vector<int32_t> up_idx;     // [edges] ascending upstream index per row
    std::vector<int32_t> slot_src;   // [edges] encoded source (see rr_b200.h)
    std::vector<uint8_t> skew;       // [n]
    std::vector<uint8_t> is_hw;      // [n] in-degree == 0
    std::vector<int32_t> export_id;  // [n]
    std::vector<rr_blk_meta> meta;   // [n_blocks]
    std::vector<int32_t> blk_level;  // [n_blocks]
    std::vector<int32_t> dep_ptr, dep_idx;  // distinct external upstream blocks
    std::vector<int32_t> exp_span;   // [n_export] level(consumer block) - level(producer block) >= 1
    std::vector<int32_t> lvl_ptr;    // [max_level+2] blocks bucketed by level
    std::vector<int32_t> lvl_blk;    // [n_blocks] block ids sorted by (level, id)
    int32_t max_level = 0, max_skew = 0, max_deg = 0;
    // coefficients (host copies; uploaded lazily)
    std::vector<double> c1, c2, c3, c4;
    bool have_c4 = false;
    uint64_t coeff_version = 0;
    std::vector<int32_t> out_subset;   // river segments (user indices) the host streaming calls copy back; empty = all
    uint64_t out_subset_version = 0;
    std::vector<double> thr;           // [n_thr][n] per-river thresholds (user order) of RR_STAT_EXCEED; uploaded lazily
    int64_t n_thr = 0;
    uint64_t thr_version = 0;
    rr_device_state *dev = nullptr;
};

// Ticket schedule for one launch: items ordered by key = level(block) + tile * delta, plus the
// exchange-ring geometry that this delta makes safe (ring depth = span / delta + 1 per exported reach).
struct rr_schedule {
    int64_t n_items = 0;
    int32_t delta = 1;
    int64_t n_keys = 0;
    std::vector<int64_t> key_start;  // [n_keys+1] prefix sum of items per key
    std::vector<int32_t> exp_ro;     // [n_export][2] {first row, ring depth} of each exported series
    std::vector<int32_t> edge_ro;    // [edges][2] the same pair for the upstream of each upstream-CSR entry
    int64_t raw_rows = 0;            // total rows (per ensemble member)
};
// delta = ticket-key distance between consecutive tiles of one block (0: smallest power of two whose
// rings fit `budget_rows` rows).
void rr_build_schedule(const rr_plan &p, int64_t n_tiles, int32_t delta, int64_t budget_rows, rr_schedule &s);
void rr_build_rings(const rr_plan &p, int32_t delta, int64_t budget_rows, rr_schedule &s);
// first_block > 0 leaves blocks [0, first_block) out of the schedule (whole-headwater blocks of a level-sorted plan that
// the staging kernel routes; they are level-0 blocks)
void rr_build_keys(const rr_plan &p, int64_t n_tiles, rr_schedule &s, int64_t first_block = 0);
void rr_build_items(const rr_plan &p, int64_t n_tiles, const rr_schedule &s, std::vector<int32_t> &items,
                    int64_t first_block = 0);  // [n_items][4] block, tile, dep range
// Host mirror of the kernel's ticket decode.
void rr_decode_ticket(const rr_plan &p, const rr_schedule &s, int64_t n_tiles, int64_t ticket,
                      int32_t *block, int32_t *tile);

void rr_device_release(rr_plan *p);  // frees p->dev (rr_api.cu)

// rr_stats.cu: a validated rr_stats_spec with the percentile positions resolved for M members
struct rr_stats_plan {
    int32_t n_stats = 0, n_members = 0, sort = 0, exceed = 0;
    int32_t kind[RR_MAX_STATS] = {}, lo[RR_MAX_STATS] = {}, hi[RR_MAX_STATS] = {};   // exceed: lo = threshold row
    double g[RR_MAX_STATS] = {};
};
// n_thr: threshold rows the exceed entries may index (0: none)
int rr_stats_prepare(const rr_stats_spec *spec, int32_t n_members, int64_t n_thr, rr_stats_plan *out);
// thresholds and running peaks of one launch (rr_ensemble_stats_dev_ex); all NULL: per-step rows only
struct rr_stats_ext {
    const double *thr = nullptr;       // [n_thr][ldt] by reach
    int64_t ldt = 0;
    double *peak = nullptr;            // [n_stats][ldk], read and updated
    int32_t *peak_row = nullptr;
    int64_t ldk = 0, row0 = 0;         // row0: global row of the launch's first output row
};
// out[s] + t * ldo + c = statistic s of row t: the members' rows t*k .. t*k+k-1 averaged first (k = resample); out NULL
// (or out[s] NULL): no per-step rows
int rr_stats_launch(const rr_stats_plan &sp, const double *x, int64_t member_stride, int64_t ld, int k, int64_t rows_out,
                    int64_t n_out, const int32_t *subset, void *const *out, int64_t ldo, int out_f32, const rr_stats_ext &ex,
                    void *stream);
// peak[0 .. count) = -inf, peak_row[0 .. count) = 0
int rr_stats_peak_init(double *peak, int32_t *peak_row, int64_t count, void *stream);
