// layout.h -- the flattened, vectorised SoA scene layout shared by the host flattener (scene.cpp)
// and the device kernels (device.cuh).  Everything is float4 records in ONE contiguous blob that
// each CTA stages into shared memory once (shipped scenes: <= 2.5 KB), so the per-segment linear
// scan of reference ChunkState::try_hit (src/tracer/mod.rs:389-402) reads broadcast LDS.128.
#pragma once
#include <stdint.h>

namespace bt {

// ---- primitive record: PRIM_STRIDE float4 -------------------------------------------------
//   q4 = (type, material index, volume index | rect area, object index)   [int bits except area]
// SPHERE (reference src/scene/object/sphere.rs:11-16; translation only, :121-148)
//   q0 = (cx, cy, cz, r)   q1 = (r*r, PI*r*r, 2e-5/r [free-distance margin], -)
// RECT / CUBOID_FACE (reference rect.rs:110-155 with everything ray-independent hoisted:
//   n = M*z, the full affine inverse and the local axes folded into two plane equations)
//   q0 = (n.xyz, hw^2/|x|^2)  q1 = (T.xyz, hh^2/|y|^2)
//   q2 = (ax.xyz, cx)  q3 = (ay.xyz, cy)   with local.x = dot(pos, ax) + cx
// RECT_AA: a Rect whose world normal and both plane-equation axes are exact +-unit coordinate axes
//   (every wall of the Cornell box).  Same record, with the in-plane axes ordered so that q2 lies on
//   axis (k+1)%3 and q3 on (k+2)%3, k = the normal's axis; the scan then runs rect_test_aa<k>, which
//   picks components instead of forming dot products and rounds exactly like the general test.
enum { PRIM_SPHERE = 0, PRIM_RECT = 1, PRIM_CUBOID_FACE = 2, PRIM_RECT_AA = 3 };
enum { PRIM_STRIDE = 5 };
// q4.x = type | (k << 2) | (canonical primitive index << PRIM_CANON_SHIFT): under a BVH the records are
// stored in tree order and the canonical index decides exact-distance ties the way the reference's
// scan order does.
enum { PRIM_CANON_SHIFT = 4 };

// ---- BVH node: BVH_STRIDE float4 = one 128-byte line (extension: built when a scene exceeds the linear-scan budget)
//   a 4-wide inner node holds the boxes of its (up to) four children, one float4 per bound and axis, so a child is
//   only visited when its box is hit and one fetch decides four subtrees:
//   n0 = min.x[0..3]  n1 = max.x[0..3]  n2 = min.y  n3 = max.y  n4 = min.z  n5 = max.z  n6 = child references  n7 = -
//   child reference: inner node index, BVH_LEAF | kind << 29 | count << 24 | first record (count <= BVH_LEAF_MAX;
//   kind: BVH_KIND_SPHERES / BVH_KIND_RECTS when every record of the leaf is a sphere / none is, else 0), or BVH_EMPTY
//   Traversal stack: BVH_STACK_SMEM entries per lane in shared memory, the (rarely reached) rest up to BVH_STACK in
//   local memory; the builder keeps the tree shallow enough that 3 pushes per level never exceed BVH_STACK.
enum { BVH_STRIDE = 8, BVH_WIDTH = 4, BVH_LEAF = 0x80000000u, BVH_EMPTY = 0xfffffffeu, BVH_STACK_SMEM = 16, BVH_STACK = 40, BVH_MAX_DEPTH2 = 24,
       BVH_LEAF_MAX = 31, BVH_KIND_SPHERES = 1, BVH_KIND_RECTS = 2 };

// ---- material record: MAT_STRIDE float4 (reference src/scene/data/material.rs:22-44) -------
//   m0 = (albedo.rgb, kind)   m1 = (roughness, ior, intensity, -)
enum { MAT_FLAT = 0, MAT_DIFFUSE = 1, MAT_METALLIC = 2, MAT_GLASS = 3, MAT_EMISSIVE = 4 };
enum { MAT_STRIDE = 2 };

// ---- light record: LIGHT_STRIDE float4 (objects with ObjectFlags::LIGHT, object/mod.rs:23-28)
//   l0 = (type, first primitive, primitive count, object index)
//   SPHERE: l1 = (c.xyz, r)
//   RECT:   l1 = (x.xyz, -hw) l2 = (y.xyz, -hh) l3 = (Mx.xyz, scale_x) l4 = (My.xyz, scale_y)
//           l5 = (Mz.xyz, -) l6 = (T.xyz, -)       (rect.rs:82-86: Uniform::new_inclusive(-h, h))
//   POINT:  l1 = (T.xyz, -)                        (object/mod.rs:150)
//   CUBOID: l1 = (cum0..cum3) l2 = (cum4, Uniform::new(0, total).scale, first face sub-record, -)
//           WeightedIndex over the face areas (cuboid.rs:48-54).  The six faces follow the n_lights
//           object records as LIGHT_RECT sub-records (never picked by the light index) with the
//           face transform and l5.w = Rect::area; Cuboid::pdf (cuboid.rs:56-81) walks them.
enum { LIGHT_SPHERE = 0, LIGHT_RECT = 1, LIGHT_POINT = 2, LIGHT_CUBOID = 3 };
enum { LIGHT_STRIDE = 7 };

// ---- volume record: VOL_STRIDE float4 (reference src/scene/data/volume.rs:75-82) -----------
//   v0 = (width, height, depth, grid offset in floats) [ints]   v1 = (size.xyz, -)
enum { VOL_STRIDE = 2 };

// ---- lens record: LENS_STRIDE float4 (extension) -------------------------------------------
//   e0 = (c.xyz, -1.5 r_s)   e1 = (r_s, r_far * r_s, -, -)   (stage evaluations read e0 only)
enum { LENS_STRIDE = 2 };

// ---- box record: BOX_STRIDE float4 (a Cuboid whose faces form one rectangular box) ------------
//   b0 = (C.xyz, h0)  b1 = (a0.xyz, h1)  b2 = (a1.xyz, h2)  b3 = (a2.xyz, bits)
//   centre, unit axes, half extents; faces 2k / 2k+1 sit at -h_k / +h_k along a_k; bit i: the
//   stored normal of face i points along -a_k.  The FIRST face record of such a cuboid carries
//   1 + box index in q4.z (0: test the six rects).
enum { BOX_STRIDE = 4 };

// ---- primitive bound record: BOUND_STRIDE float4 (extension; free-distance query of the stepper)
//   b0 = (lo.xyz, -)   b1 = (hi.xyz, -)   world AABB of a rect; unused for spheres (exact formula)
enum { BOUND_STRIDE = 2 };

// ---- content bits: SceneHeader::content, and the template mask C of the kernel variants (variants.h)
// CT_AOV: the call renders Output::Albedo / Normal / Depth (the first-hit latches of mod.rs:306-315).
// CT_CUBOID_LIGHT: a Cuboid carries ObjectFlags::LIGHT (WeightedIndex face pick, cuboid.rs:48-81; generic kernels only).
enum { CT_SPHERES = 1, CT_RECTS = 2, CT_VOLUMES = 4, CT_METAL = 8, CT_GLASS = 16, CT_AOV = 32, CT_CUBOID_LIGHT = 64, CT_ALL = 127 };

struct SceneHeader {
    uint32_t n_prims, prim_off;      // offsets in float4 units into the blob
    uint32_t n_mats, mat_off;
    uint32_t n_lights, light_off;
    uint32_t n_vols, vol_off;
    uint32_t n_lens, lens_off;
    uint32_t n_boxes, box_off;       // BOX records (linear-scan scenes)
    uint32_t bound_off;              // per-primitive world AABBs, BOUND_STRIDE float4 each (lensed linear-scan scenes)
    uint32_t blob_f4;                // total float4 count
    uint32_t n_bvh, bvh_off;         // BVH nodes (0: linear scan over shared memory)
    uint32_t stage_off, stage_f4;    // the part of the blob every CTA stages into shared memory
    uint32_t has_volume_prims;       // any sphere with volume != None
    uint32_t content;                // CT_* bits of the scene (CT_AOV comes from the call): picks a kernel without the unused code
    // root material folded to what sample_root returns (src/tracer/mod.rs:429-452)
    float root_color[3], root_albedo[3];
    uint32_t root_keeps_normal;      // 1: normal = -dir, depth = clip_max; 0: normal = 0, depth = inf
    // lens stepping
    float kappa, h_min, h_max;
    uint32_t max_steps;
    uint32_t lens_exact;             // BT_LENS_EXACT_RSQRT
    uint32_t lens_skip;              // 0: every chord is intersected (BT_LENS_NO_SKIP); 1: chords shorter than the free distance are
                                     // not, the distance tracked per flight (nearest sphere exactly, the rest decaying);
                                     // 3: the same, the distance read from the grid below
    // ---- free-distance grid (extension; lensed linear-scan scenes): dist[(z * ny + y) * nx + x] * dist_q is a lower bound on the
    // distance from ANY point of the cell to the surface of ANY primitive, already reduced by the rounding margins of the hit
    // tests.  The box spans every primitive but the `n_far` scene-spanning spheres listed in far_prim, with dist_pad to spare:
    // outside it the bound is min(distance to the box + dist_pad, exact distance to those spheres).
    float dist_lo[3], dist_hi[3];
    float dist_cell, dist_inv_cell, dist_q, dist_pad;
    uint32_t dist_nx, dist_ny, dist_nz;
    uint32_t n_far;
    int32_t far_prim[2];
};

struct CameraBlock {                 // reference src/tracer/mod.rs:244-267 hoisted per render call
    float m[9];                      // transform_world matrix3 columns
    float t[3];
    float yfov, xfov, pixel_width, pixel_height;
    float su_low, su_scale, sv_low, sv_scale;   // Uniform::from(min..max) for the jitter
    float sub_width;                 // 1/n, 0 for Subsample::None
    uint32_t sub_n;                  // n (1 for None)
    uint32_t has_focus;
    float focus, aperture;
    float disk_x[3], disk_y[3];      // UnitDisk::new(NEG_Z) basis
};

struct RenderParams {
    SceneHeader scene;
    CameraBlock cam;
    const float4* blob;
    const float* grids;
    const uint8_t* dist;             // the free-distance grid (SceneHeader::dist_*), device memory
    const float4* env;               // environment map (bt_scene_set_environment): env_w x env_h texels, .w unused, device memory
    uint32_t env_w, env_h;           // env_w == 0: no map
    float4* fb;
    uint32_t width, height;
    uint32_t paths_per_pixel;        // samples * subpixel_count of this call
    uint32_t sub_count;
    uint64_t seed, path_base;        // path index of the first path of this call
    uint64_t light_zone;             // UniformInt<usize>::new(0, n_lights): the acceptance zone (rand 0.8.5), hoisted per call
    uint32_t row0, row_end;          // this launch renders pixel rows [row0, row_end) (bt_render pipelines a host frame in bands)
    int32_t output;
    uint32_t max_bounces, max_volume_bounces;
    float clip_min, clip_max, volume_step;
    float tau_scale, one_scale;      // Uniform::new_inclusive(0, TAU).scale, (0, 1).scale
    uint32_t compact_lanes, compact_patience;  // per-warp step compaction thresholds (LENS kernels)
    uint32_t regen_lanes, regen_patience;      // idle lanes a warp collects before it runs the ray-generation phase
    uint32_t scan_lanes, scan_patience;
    uint32_t steps_per_turn;                   // RK4 steps a flying lane takes between two rounds of ballots        // pending chords a warp collects before it runs the intersection phase
    // the pooled kernel (render_pool.cuh): 0 = render_body (one path per lane), W > 0 = 32 W path slots per warp
    uint32_t pool_w;
    uint32_t pool_refill;            // STEP: lanes that wait for a flight before the warp pays for a refill round
    uint32_t pool_step_min;          // STEP: with the stack empty, keep stepping while at least this many lanes fly
    uint32_t pool_threads;           // CTA size of the pooled kernel
    uint32_t bvh_stack_k;            // BVH traversal: stack levels kept in shared memory (clamped to what the kernel allocates)
    unsigned long long* pool_counter;  // ... and its tile counter (zeroed before every launch)
    char* pool_q;                    // the pooled kernel's path-state arena: pool_q_bytes per warp of its grid (device memory)
    uint64_t pool_q_cap;             // bytes available at pool_q (bounds the grid)
    uint32_t pool_stats;             // launch the pooled kernel's counter variant (bt_render_pool_stats): stats[0..11]
    unsigned long long* stats;       // render_kernel_stats only: {paths, scan calls, RK4 steps, events}
};

}  // namespace bt
