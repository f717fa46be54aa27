// A C ABI over the kernel-variant table and its selection (bendy_tracer_b200/csrc/variants.h) for
// test_variant_table.py: host code only, built with the host compiler.
#include <vector_types.h>

#include "variants.h"

extern "C" {

int vt_count() { return bt::kNumVariants; }

// out = {LENS, EXACT, NL, BVH, C, families compiled in this flavour}
void vt_row(int i, int exact_flavour, int* out) {
    const bt::Variant& v = bt::kVariants[i];
    const int row[6] = {v.lens, v.exact, v.nl, v.bvh, v.c, bt::variant_families(v, exact_flavour != 0)};
    for (int k = 0; k < 6; ++k) out[k] = row[k];
}

// mode: 0 render, 1 work counters (bt_render_stats), 2 pool counters (bt_render_pool_stats), 3 trace.
// Returns the row the call launches (-1: none), its family in *family.
int vt_select(uint32_t content, int32_t output, uint32_t n_lens, uint32_t lens_exact, uint32_t n_bvh, uint32_t pool_w,
              uint32_t max_bounces, uint32_t n_prims, int mode, int exact_flavour, int* family) {
    static unsigned long long counters[17];
    bt::RenderParams p = {};
    p.scene.content = content;
    p.scene.n_lens = n_lens;
    p.scene.lens_exact = lens_exact;
    p.scene.n_bvh = n_bvh;
    p.scene.n_prims = n_prims;
    p.output = output;
    p.pool_w = pool_w;
    p.max_bounces = p.max_volume_bounces = max_bounces;
    p.stats = mode == 1 || mode == 2 ? counters : nullptr;
    p.pool_stats = mode == 2;
    *family = mode == 3 ? bt::V_TRACE : bt::render_family(p);
    return bt::select_variant(p, *family, exact_flavour != 0);
}
}
