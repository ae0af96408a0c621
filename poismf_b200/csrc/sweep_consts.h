// poismf_b200 — sizes shared by the half-sweep kernels and the row planner (row_plan.h).
// Host-only constants: the planner's shared-memory and register arithmetic must see the values the kernels
// are compiled with.
#pragma once
#include <stddef.h>

// minimum resident CTAs the (sub-)warp kernels are compiled for: caps registers at 80/thread
// so that three 256-thread CTAs fit an SM when their shared-memory slices allow it
#ifndef PMF_WARP_KERNEL_MIN_CTAS
#define PMF_WARP_KERNEL_MIN_CTAS 3
#endif

namespace pmf {

constexpr size_t SMEM_PER_SM = 233472;      // 228 KB
constexpr size_t SMEM_CTA_MAX = 232448;     // 227 KB opt-in maximum per CTA
constexpr size_t SMEM_CTA_RESERVED = 1024;  // per-CTA system reservation

// registers per thread the (sub-)warp kernels are compiled for (__launch_bounds__ of rows_warp_kernel)
constexpr int WARP_KERNEL_REGS = (65536 / (256 * PMF_WARP_KERNEL_MIN_CTAS)) / 8 * 8;

constexpr int GANG_XSLOTS = 272;                 // reals per cluster exchange buffer (>= kp of any supported k, >= 16)
constexpr int GANG_XBYTES = 2 * GANG_XSLOTS * 8; // a cluster CTA's two exchange buffers, in its shared slice
constexpr int TN_NUM_VECS = 24;                  // k-vectors of the tncg solver

constexpr int DN_TILE_ROWS = 256;   // lock-step path: rows of the fixed matrix per tile
constexpr int DN_GROUPS = 1024 / 16;  // lock-step gaxpy pass: groups of 16 lanes of its 1024-thread CTA
constexpr int DN_LS_CHUNK = 2048;   // lock-step line search: non-zeros per CTA
constexpr int DN_TRIALS = 20;       // lock-step line search: trials evaluated per pass, ALL of them (max_ls of nonnegcg.c)
constexpr int DN_TILE_COUNTERS = 64;  // lock-step dots passes: ring of tile counters, one per pass of a half-sweep

}  // namespace pmf
