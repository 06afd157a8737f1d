// Which forward kernel one mlb_forward call runs, and the launch geometry that the launch and the fused all-gather depend
// on.  Pure host code (C++17 and the public header only) so that the selection can be checked without a GPU
// (tests/test_forward_plan_cpu.py).
#pragma once
#include "../../include/monoloco_b200.h"

namespace mlb {

enum { FWD_FORCE_MASK = MLB_FWD_FORCE_TILE | MLB_FWD_FORCE_CLUSTER | MLB_FWD_FORCE_WIDE | MLB_FWD_FORCE_TC | MLB_FWD_FORCE_WIDE2 };

// What the choice depends on.  Everything but `disabled` is fixed when the handle is created.
struct FwdPlanInputs {
    unsigned have;      // bit MLB_KERNEL_k: this handle has kernel family k
    unsigned disabled;  // bit MLB_KERNEL_k: a cooperative launch of k was refused, so only a forced request still gets it
    double t_cluster_wave, t_tile_a, t_tile_b, t_tc_wave;  // per-wave times (ms, calibrate()); a row-tile wave is a + b * TM
    int n_sms;
    int small_conc;     // co-resident 8-CTA clusters of the cluster kernel
    int tc_clusters;    // co-resident clusters of the tensor-core kernel (its persistent grid)
    int tile_ctas[2];   // resident CTAs of the row-tile kernel with the residual in [0] Tensor Memory, [1] the scratch
};

struct FwdPlan {
    int kernel;         // MLB_KERNEL_*, or -1 and `error` says why
    const char* error;
    int tm, grid;       // tile: rows per group, CTAs
    int clusters;       // cluster, tc: clusters launched
    int launches;       // wide: one launch per 32 rows
    int arrivals;       // arrivals on the fused all-gather's done counter: CTAs (tile), cluster leaders, or 1
};

// minimise waves(tm) * tm (time ~ rows per CTA per wave), prefer the larger tile on ties
inline int pick_rows_per_group(int n_rows, int n_ctas) {
    int best = 16;
    long best_cost = -1;
    for (int tm = 16; tm >= 8; tm -= 2) {
        const long tiles = (n_rows + 2 * tm - 1) / (2 * tm);
        const long waves = (tiles + n_ctas - 1) / n_ctas;
        const long cost = waves * tm;
        if (best_cost < 0 || cost < best_cost) best_cost = cost, best = tm;
    }
    return best;
}

// At most one MLB_FWD_FORCE_* flag, and it must name a kernel this handle has for this many rows.  A forced kernel ignores
// rows_per_group; without one, rows_per_group != 0 means row tiles.  Otherwise, in order: the tensor cores when the width
// has no FFMA kernel or when their waves are cheaper than the better FFMA kernel (measured wave times); the
// second-generation latency kernel up to 16 rows; the whole-grid kernel up to 64 rows; FFMA clusters when cheaper than
// row tiles; row tiles.
inline FwdPlan plan_forward(const FwdPlanInputs& in, int n_rows, int flags, int rows_per_group) {
    FwdPlan pl = {};
    pl.kernel = -1;
    auto has = [&](int k) { return ((in.have >> k) & 1u) != 0; };
    auto usable = [&](int k) { return has(k) && ((in.disabled >> k) & 1u) == 0; };
    auto fail = [&](const char* msg) {
        pl.error = msg;
        return pl;
    };
    auto pick = [&](int k, int arrivals) {
        pl.kernel = k, pl.arrivals = arrivals;
        return pl;
    };
    const int forced = flags & FWD_FORCE_MASK;
    if (forced & (forced - 1)) return fail("mlb_forward: at most one MLB_FWD_FORCE_* flag may be set");
    const bool tc_only = !has(MLB_KERNEL_TILE);  // the width has no FFMA kernel (linear_size > 1024)
    if ((forced == MLB_FWD_FORCE_TC || tc_only) && !has(MLB_KERNEL_TC))
        return fail("mlb_forward: the tensor-core kernel is not available for this model (linear_size % 256 != 0)");
    if (forced == MLB_FWD_FORCE_WIDE2 && (!has(MLB_KERNEL_WIDE2) || n_rows > 16))
        return fail("mlb_forward: the second-generation latency kernel needs <= 16 rows and a supported model / device");
    if (tc_only && ((forced & (MLB_FWD_FORCE_TILE | MLB_FWD_FORCE_CLUSTER | MLB_FWD_FORCE_WIDE)) || rows_per_group != 0))
        return fail("mlb_forward: this model width runs on the tensor-core kernel only");
    if (forced == MLB_FWD_FORCE_WIDE && !has(MLB_KERNEL_WIDE))
        return fail("mlb_forward: the whole-grid kernel is not available for this model / device");
    if (forced == MLB_FWD_FORCE_CLUSTER && !has(MLB_KERNEL_CLUSTER))
        return fail("mlb_forward: the cluster kernel needs linear_size == 1024");
    const bool automatic = forced == 0 && rows_per_group == 0;

    // FFMA cost: waves of `small_conc` 8-CTA clusters (16 rows each) against waves of row tiles at the best rows per group
    const int n_clusters = (n_rows + 15) / 16;
    const double t_cluster = has(MLB_KERNEL_CLUSTER)
                                 ? in.t_cluster_wave * (double)((n_clusters + in.small_conc - 1) / in.small_conc)
                                 : 1e30;
    const int tm_c = pick_rows_per_group(n_rows, in.n_sms);
    const long tiles_c = (n_rows + 2 * tm_c - 1) / (2 * tm_c);
    const double t_tile = (in.t_tile_a + in.t_tile_b * tm_c) * (double)((tiles_c + in.n_sms - 1) / in.n_sms);

    // tensor cores: persistent clusters over 128-row tiles
    const int tc_tiles = (n_rows + 127) / 128;
    bool tc_cheaper = false;
    if (automatic && has(MLB_KERNEL_TC) && n_rows > 64) {
        const double t_tc = in.t_tc_wave * (double)((tc_tiles + in.tc_clusters - 1) / in.tc_clusters);
        tc_cheaper = t_tc < (t_tile < t_cluster ? t_tile : t_cluster);
    }
    if (forced == MLB_FWD_FORCE_TC || tc_only || tc_cheaper) {
        pl.clusters = tc_tiles < in.tc_clusters ? tc_tiles : in.tc_clusters;
        return pick(MLB_KERNEL_TC, pl.clusters);
    }
    if (forced == MLB_FWD_FORCE_WIDE2 || (automatic && usable(MLB_KERNEL_WIDE2) && n_rows <= 16)) return pick(MLB_KERNEL_WIDE2, 1);
    if (forced == MLB_FWD_FORCE_WIDE || (automatic && usable(MLB_KERNEL_WIDE) && n_rows <= 64)) {
        pl.launches = (n_rows + 31) / 32;
        return pick(MLB_KERNEL_WIDE, 1);
    }
    if (forced == MLB_FWD_FORCE_CLUSTER || (automatic && t_cluster < t_tile)) {
        pl.clusters = n_clusters < in.small_conc ? n_clusters : in.small_conc;
        return pick(MLB_KERNEL_CLUSTER, pl.clusters);
    }
    const int max_ctas = in.tile_ctas[(flags & MLB_FWD_RES_SCRATCH) ? 1 : 0];
    pl.tm = rows_per_group != 0 ? rows_per_group : pick_rows_per_group(n_rows, max_ctas);
    if (pl.tm < 8 || pl.tm > 16 || (pl.tm & 1)) return fail("mlb_forward: rows_per_group must be 0 or one of 8,10,12,14,16");
    const int tiles = (n_rows + 2 * pl.tm - 1) / (2 * pl.tm);
    pl.grid = tiles < max_ctas ? tiles : max_ctas;
    return pick(MLB_KERNEL_TILE, pl.grid);  // every CTA owns >= 1 tile and arrives once
}

}  // namespace mlb
