// variants.h -- which compiled kernel serves a render or trace call.  Plain C++ (a host compiler can test it):
// kernels.cu instantiates exactly the kernels this table lists, and launches the one select_variant picks.
#pragma once
#include <vector_types.h>

#include "layout.h"

namespace bt {

// kernel families (kernels.cu): render_kernel, render_kernel_stats (work counters), render_pool_kernel,
// render_pool_kernel_pstats (scheduling counters), render_pool_bvh_kernel, trace_kernel
enum { V_LANE = 1, V_LANE_STATS = 2, V_POOL = 4, V_POOL_STATS = 8, V_POOL_BVH = 16, V_TRACE = 32 };

// One compiled shape <LENS, EXACT, NL, BVH, C> and the families instantiated with it.  NL = 1: the stepper
// specialised for one mass; 0: any number.  C: the CT_* content the kernel carries code for (trace_kernel has no C).
struct Variant { bool lens, exact; int nl; bool bvh; int c, families; };

// A family's kernel for a call is its first row that serves the call (select_variant), so the
// content-specialised rows come first, then the generic ones without and with the LIGHT Cuboid code.
constexpr int CT_NO_CUBOID_LIGHT = CT_ALL & ~CT_CUBOID_LIGHT;
constexpr Variant kVariants[] = {
    {false, false, 0, false, CT_RECTS, V_LANE | V_POOL | V_POOL_STATS},                          // cornell (C1)
    {false, false, 0, false, CT_RECTS | CT_METAL, V_LANE | V_POOL | V_POOL_STATS},               // cornell2 (C2)
    {false, false, 0, false, CT_SPHERES | CT_VOLUMES, V_LANE | V_POOL | V_POOL_STATS},           // cloud, volume
    {false, false, 0, false, CT_SPHERES | CT_METAL | CT_GLASS, V_LANE | V_POOL | V_POOL_STATS},  // scene
    {true, false, 1, false, CT_SPHERES | CT_METAL | CT_GLASS, V_LANE | V_POOL | V_POOL_STATS},   // scene + one mass (C3, C5)
    {true, false, 1, false, CT_SPHERES | CT_VOLUMES, V_LANE | V_POOL | V_POOL_STATS},            // cloud / volume + one mass
    {true, true, 1, false, CT_SPHERES | CT_VOLUMES, V_POOL | V_POOL_STATS},                      // ... exact stepper (C4-cloud-lens)
    {false, false, 0, false, CT_NO_CUBOID_LIGHT, V_LANE | V_POOL},
    {false, false, 0, true, CT_NO_CUBOID_LIGHT, V_LANE | V_POOL_BVH},
    {true, true, 0, true, CT_NO_CUBOID_LIGHT, V_LANE},
    {true, false, 0, true, CT_NO_CUBOID_LIGHT, V_LANE},
    {true, false, 1, false, CT_NO_CUBOID_LIGHT, V_LANE | V_POOL},
    {true, false, 0, false, CT_NO_CUBOID_LIGHT, V_LANE | V_POOL},
    {true, true, 0, false, CT_NO_CUBOID_LIGHT, V_LANE | V_POOL},
    {false, false, 0, false, CT_ALL, V_LANE | V_LANE_STATS | V_POOL | V_TRACE},
    {false, false, 0, true, CT_ALL, V_LANE | V_LANE_STATS | V_POOL_BVH | V_TRACE},
    {true, true, 0, true, CT_ALL, V_LANE | V_LANE_STATS | V_TRACE},
    {true, false, 0, true, CT_ALL, V_LANE | V_LANE_STATS | V_TRACE},
    {true, false, 1, false, CT_ALL, V_LANE | V_LANE_STATS | V_POOL | V_TRACE},
    {true, false, 0, false, CT_ALL, V_LANE | V_LANE_STATS | V_POOL | V_TRACE},
    {true, true, 0, false, CT_ALL, V_LANE | V_LANE_STATS | V_POOL | V_TRACE},
};
constexpr int kNumVariants = sizeof kVariants / sizeof kVariants[0];

// The families row `v` is compiled for in a flavour.  The exact flavour renders every lensed scene with the
// exact stepper (engine.cu: build_params sets lens_exact), so it compiles no fast-stepper lensed kernel.
constexpr int variant_families(const Variant& v, bool exact_flavour) {
    return exact_flavour && v.lens && !v.exact ? 0 : v.families;
}

// The pooled kernel packs a path's counters into 8 bits each and its volume object into 7 (render_pool.cuh:
// pack_misc): it serves max_bounces, max_volume_bounces <= POOL_MAX_BOUNCES and scan scenes of up to
// POOL_MAX_OBJECTS primitives; BVH scenes hold no volumetric spheres, so nothing limits them.
enum { POOL_MAX_BOUNCES = 254, POOL_MAX_OBJECTS = 126 };

// The family of a render call (trace calls are V_TRACE); 0: none (pool counters outside the pooled kernel's reach).
inline int render_family(const RenderParams& p) {
    const bool bvh_pool = p.scene.n_bvh != 0 && p.scene.n_lens == 0;  // (lensed BVH scenes run the lane kernel)
    const bool pool_ok = p.pool_w != 0 && (p.scene.n_bvh == 0 || bvh_pool) && p.max_bounces <= POOL_MAX_BOUNCES &&
                         p.max_volume_bounces <= POOL_MAX_BOUNCES && (p.scene.n_prims <= POOL_MAX_OBJECTS || bvh_pool);
    if (p.pool_stats) return pool_ok ? V_POOL_STATS : 0;
    if (p.stats) return V_LANE_STATS;
    if (pool_ok) return bvh_pool ? V_POOL_BVH : V_POOL;
    return V_LANE;
}

// Index of the first row of `family` that serves the call, -1 when none does.  A row serves it when LENS and BVH
// are the scene's, EXACT is the scene's lens_exact (lensed rows), NL is 0 or the number of masses, and C holds
// the scene's content (plus CT_AOV for an Albedo / Normal / Depth output).
inline int select_variant(const RenderParams& p, int family, bool exact_flavour) {
    const uint32_t ct = p.scene.content | (p.output != 0 ? (uint32_t)CT_AOV : 0u);
    const bool lens = p.scene.n_lens != 0, bvh = p.scene.n_bvh != 0, exact = p.scene.lens_exact != 0;
    for (int i = 0; i < kNumVariants; ++i) {
        const Variant& v = kVariants[i];
        if ((variant_families(v, exact_flavour) & family) && v.lens == lens && v.bvh == bvh && (!lens || v.exact == exact) &&
            (v.nl == 0 || (uint32_t)v.nl == p.scene.n_lens) && (ct & ~(uint32_t)v.c) == 0)
            return i;
    }
    return -1;
}

}  // namespace bt
