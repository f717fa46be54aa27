// kernels.cu -- the CUDA kernels of the per-sample render loop (sm_100a).
//
// render_kernel: one lane = one pixel; the lane walks its pixel's paths in the reference's order
// (pass-major, sub-pixel minor: src/tracer/mod.rs:277-278) and regenerates a new path the moment
// the previous one terminates, so path-length divergence never idles a lane ("persistent lane
// with in-register path regeneration").  Path state lives in registers, the scene blob in shared
// memory; HBM traffic is one float4 read-modify-write per pixel per call (buffer.rs:159-178).
// Pixel sums are formed in the reference's order, so the result is deterministic.
#include "device.cuh"
#include "kernels.h"
#include "variants.h"

#include <algorithm>
#include <cstdlib>
#include <utility>

#ifdef BT_EXACT_SCAN
#define BT_SFX(name) name##_exact
constexpr bool kExactFlavour = true;
#else
#define BT_SFX(name) name##_fast
constexpr bool kExactFlavour = false;
#endif

namespace bt {

namespace {

struct SceneView {
    const float4* nodes;   // BVH nodes in global memory (BVH kernels only)
    uint32_t* stack;       // BVH traversal stack in shared memory
    const float4* prims;
    const float4* mats;
    const float4* lights;
    const float4* vols;
    const float4* lens;
    const float4* bounds;  // per-primitive AABBs (lensed scan scenes)
    const float4* boxes;   // BOX records of box-shaped cuboids (scan scenes)
    const float* grids;
};

template <bool BVH>
BT_DEV SceneView stage_scene(const RenderParams& p, float4* smem) {
    const uint32_t base = p.scene.stage_off;
    for (uint32_t i = threadIdx.x; i < p.scene.stage_f4; i += blockDim.x) smem[i] = p.blob[base + i];
    __syncthreads();
    SceneView s;
    s.prims = BVH ? p.blob + p.scene.prim_off : smem + (p.scene.prim_off - base);
    s.nodes = p.blob + p.scene.bvh_off;
    s.stack = reinterpret_cast<uint32_t*>(smem + p.scene.stage_f4);
    s.mats = smem + (p.scene.mat_off - base);
    s.lights = smem + (p.scene.light_off - base);
    s.vols = smem + (p.scene.vol_off - base);
    s.lens = smem + (p.scene.lens_off - base);
    s.bounds = smem + (p.scene.bound_off - base);
    s.boxes = smem + (p.scene.box_off - base);
    s.grids = p.grids;
    return s;
}

struct Traced {
    Hit h;            // h.prim < 0: miss (or capture)
    V3 o, d;          // the straight piece the hit lies on (chord under lensing) / escape direction
    float t_total;    // accumulated length up to the hit
    uint32_t steps;
    uint32_t scans;   // scan_prims calls (= chords intersected)
    bool captured;
};

// try_hit / try_hit_volume of the reference: one straight segment.
template <bool BVH, int C = CT_ALL>
BT_DEV Traced trace_straight(const RenderParams& p, const SceneView& sc, V3 o, V3 d, float tmin, float tmax, int vol_obj) {
    Traced r;
    if (BVH)
        r.h = bvh_closest(sc.prims, sc.nodes, sc.stack, o, d, tmin, tmax);
    else
        r.h = scan_prims<C>(sc.prims, sc.boxes, (int)p.scene.n_prims, o, d, tmin, tmax, vol_obj);
    r.steps = 0;
    r.scans = 1;
    r.captured = false;
    r.o = o;
    r.d = d;
    r.t_total = r.h.t;
    return r;
}

// A geodesic in flight: the state a lane carries between steps (x, v live in the caller's registers; they and xp are
// held in the stepper's paired layout, P3).
// Nothing else is written inside the flight loop: the event a resolved flight hands to shading is
// rebuilt from this state afterwards (flight_result), which keeps the loop free of merge copies.
struct Flight {
    float travelled;
    uint32_t steps, scans;
    float free;  // no primitive surface lies within this distance of x (<= 0: unknown)
    float rest;  // the same for every primitive but `near`, whose distance is re-evaluated at each step
    int near;    // the sphere that bounded `free` at the last intersection pass (-1: none / not a sphere)
    P3 xp;       // start of the last chord xp -> x that needed / needs an intersection test
    Hit h;       // FL_HIT / FL_HIT_FAR: the hit on that chord (t relative to its start)
};
// Lane states.  In flight: FL_FLY ready for the next RK4 step; FL_PEND the step is taken (x, v
// advanced) but its chord awaits the intersection phase; FL_PEND_FAR beyond r_far of every mass and
// receding -- the rest of the ray is one straight segment.  Resolved (bit 2): FL_HIT on the chord,
// FL_HIT_FAR on the final straight segment, FL_ESCAPED, FL_CAPTURED.  Not a flight (bit 3): FL_IDLE
// (no path), FL_STRAIGHT (a straight segment traced by try_hit / try_hit_volume, event ready).
enum { FL_FLY = 0, FL_PEND = 1, FL_PEND_FAR = 2, FL_HIT = 4, FL_HIT_FAR = 5, FL_ESCAPED = 6, FL_CAPTURED = 7, FL_IDLE = 8,
       FL_STRAIGHT = 12 };

BT_DEV void flight_reset(Flight& f) {
    f.travelled = 0.0f;
    f.steps = f.scans = 0;
    f.free = f.rest = 0.0f;
    f.near = -1;
    f.xp = p3(make_float2(0.0f, 0.0f), 0.0f);
    f.h.t = 0.0f;
    f.h.prim = -1;
    f.h.face = 0;
}
// Lower bound on the distance from x to the nearest primitive surface, from the scene's free-distance grid
// (SceneHeader::dist_*, built by scene.cpp: build_dist_grid) and the exact distance of its scene-spanning spheres.
// One byte load.  It is split in two so that the load is ISSUED before the RK4 arithmetic of the step that needs it
// and its value first TOUCHED after (grid_bound_finish): L2 latency then hides under ~150 instructions.
// One straight sequence for every refreshing lane: the byte load is predicated on "inside the box", the outside bound is
// computed by all and selected away inside -- a warp whose refreshing lanes sit on both sides of the box faces runs the
// block once, not an in-box and an out-of-box path one after the other.  The outside part is skipped, warp-uniformly, when
// no lane running the block is outside.  The far spheres come from the call's constants (SceneHeader::far_c / far_k),
// unrolled on the uniform n_far.
struct GridFetch {
    uint32_t raw;   // the cell's byte (inside the box)
    float other;    // min(outside-the-box bound or +inf, the scene-spanning spheres' exact bounds)
    bool inside;
};
BT_DEV float far_sphere_bound(const SceneHeader& s, int i, V3 x) {
    const float4 q0 = make_float4(s.far_c[i][0], s.far_c[i][1], s.far_c[i][2], s.far_c[i][3]);
    const float4 q1 = make_float4(0.0f, 0.0f, s.far_k[i], 0.0f);
    const V3 oc = x - v3(q0);
    return sphere_free_bound(q0, q1, fmaf(oc.z, oc.z, fmaf(oc.y, oc.y, oc.x * oc.x)));
}
BT_DEV GridFetch grid_bound_fetch(const RenderParams& p, P3 px) {
    const SceneHeader& s = p.scene;
    // cell index: a negative coordinate converts to a negative int, i.e. a huge unsigned one
    const float2 cxy = __ffma2_rn(px.xy, f2(s.dist_inv_cell), make_float2(s.dist_off[0], s.dist_off[1]));
    const uint32_t ix = (uint32_t)__float2int_rd(cxy.x), iy = (uint32_t)__float2int_rd(cxy.y),
                   iz = (uint32_t)__float2int_rd(__fmaf_rn(px.z, s.dist_inv_cell, s.dist_off[2]));
    const bool inside = ix < s.dist_nx && iy < s.dist_ny && iz < s.dist_nz;
    GridFetch g;
    g.inside = inside;
    g.raw = 0xffffu;  // (x q: beyond every stored value -- the box does not bound this point, `other` does)
    if (inside) g.raw = __ldg(p.dist + ((iz * s.dist_ny + iy) * s.dist_nx + ix));
    g.other = __int_as_float(0x7f800000);
    // (every lane that runs this block takes part in the vote, so an outside lane always sees it true)
    if (__any_sync(__activemask(), !inside)) {
        // outside the box: every gridded primitive lies dist_pad inside its faces; the scene-spanning spheres exactly
        const V3 x = v3(px);
        const float dx = fmaxf(fmaxf(s.dist_lo[0] - x.x, x.x - s.dist_hi[0]), 0.0f);
        const float dy = fmaxf(fmaxf(s.dist_lo[1] - x.y, x.y - s.dist_hi[1]), 0.0f);
        const float dz = fmaxf(fmaxf(s.dist_lo[2] - x.z, x.z - s.dist_hi[2]), 0.0f);
        float other = (sqrt_approx(fmaf(dz, dz, fmaf(dy, dy, dx * dx))) + s.dist_pad) * 0.999f - 1e-3f;
        if (s.n_far > 0) other = fminf(other, far_sphere_bound(s, 0, x));
        if (s.n_far > 1) other = fminf(other, far_sphere_bound(s, 1, x));
        if (!inside) g.other = other;
    }
    return g;
}
// `late`: any value computed at the end of the step.  The byte is converted only after it (late != late is false for every
// finite value; the compiler cannot know), which keeps ptxas from scheduling the first use of the load right behind it.
BT_DEV float grid_bound_finish(const RenderParams& p, const GridFetch& g, float late) {
    return fminf((float)(g.raw + (late != late ? 1u : 0u)) * p.scene.dist_q, g.other);
}
// STEP phase: one RK4 step of a bent ray.  A chord shorter than the free distance cannot touch
// anything and is committed at once; otherwise it is left pending for the intersection phase.
// The free distance decays with the distance flown, except for the sphere that bounded it at the
// last intersection pass: its distance is evaluated afresh at the chord's start, so a ray that flies
// along a large surface (the r = 100 ground sphere, a unit or three below most of every path) keeps its
// free distance instead of spending it after a few steps (C3: 23.7 -> 12.8 intersection passes per path, cloud + lens 28.6 -> 18.8).
// `refreshed` (the pooled kernel's counters only): 0 no grid refresh in this step, 1 from a cell of the grid, 2 outside its box.
template <bool EXACT, int C, class L>
BT_DEV int geodesic_step(const RenderParams& p, const L& lens, const float4* prims, P3& x, P3& v, Flight& f, float tmax,
                         int* refreshed = nullptr) {
    if (refreshed) *refreshed = 0;
    float rmin;
    bool captured, far;
    D0Cache<L> cache;
    const P3 k1 = lens_accel<2, EXACT, 0>(lens, cache, x, 0.0f, v, v, rmin, captured, far);
    if (captured) return FL_CAPTURED;
    if (far) return FL_PEND_FAR;
    // the chord's start is kept where a pending chord needs it (f.xp): the step writes the new position into x and nothing
    // is copied afterwards, whatever the chord turns out to be
    f.xp = x;
    float free = f.free;
    GridFetch gf;
    gf.raw = 0;
    gf.other = 0.0f;
    gf.inside = false;
    // Grid mode: the bound decays with the distance flown (f.free) and is re-read from the grid only when the coming chord
    // (about as long as the last one, f.rest) could outrun it -- a byte gather by all 32 lanes at every step is 32 L1
    // wavefronts per warp instruction and made the step L1-bound (C3: -6 %); a quarter of the lanes is not.
    const bool grid = p.scene.lens_skip == 3, refresh = grid && free <= 1.4f * f.rest;
    if (grid) {
        if (refresh) gf = grid_bound_fetch(p, f.xp);
        if (refreshed && refresh) *refreshed = gf.inside ? 1 : 2;
    } else if ((C & CT_SPHERES) && f.near >= 0) {
        const float4* q = prims + f.near * PRIM_STRIDE;
        const float4 q0 = q[0], q1 = q[1];
        const V3 oc = v3(f.xp) - v3(q0);
        free = fminf(sphere_free_bound(q0, q1, fmaf(oc.z, oc.z, fmaf(oc.y, oc.y, oc.x * oc.x))), f.rest);
    }
    rk4_from_k1<EXACT>(lens, cache, x, v, k1, step_size(p.scene.kappa, p.scene.h_min, p.scene.h_max, rmin));
    float len;
    (void)normalize_fma<EXACT>(x - f.xp, &len);
    if (refresh) free = fmaxf(free, grid_bound_finish(p, gf, len));
    if (len * 1.02f < free) {  // nothing within reach: the chord needs no intersection test
        f.free = free - len;
        f.rest = grid ? len : f.rest - len;
        f.travelled += len;
        f.steps++;
        return (f.travelled >= tmax || f.steps >= p.scene.max_steps) ? FL_ESCAPED : FL_FLY;
    }
    return FL_PEND;
}
// INTERSECTION phase: the pending chord (or the final straight segment) against the scene; the
// same pass refreshes the free distance.  Returns a resolved state or FL_FLY.
template <bool EXACT, bool BVH, int C = CT_ALL>
BT_DEV int geodesic_scan(const RenderParams& p, const SceneView& sc, P3 x, P3 v, Flight& f, int state, float tmin, float tmax) {
    const bool far = state == FL_PEND_FAR;
    const float remaining = tmax - f.travelled;
    const float cmin = fmaxf(tmin - f.travelled, 0.0f);
    const V3 o = v3(far ? x : f.xp);
    float len;
    const V3 dir = normalize_fma<EXACT>(far ? v : x - f.xp, &len);
    const float cmax = far ? remaining : fminf(len, remaining);
    FreeInfo bound;
    bound.nearest = bound.rest = 0.0f;
    bound.sphere = -1;
    if (BVH)
        f.h = bvh_closest<!EXACT>(sc.prims, sc.nodes, sc.stack, o, dir, cmin, cmax);
    else if (p.scene.lens_skip != 0 && p.scene.lens_skip != 3)
        f.h = scan_prims_t<true, C, !EXACT>(sc.prims, sc.bounds, sc.boxes, (int)p.scene.n_prims, o, dir, cmin, cmax, -1, &bound);
    else
        f.h = scan_prims_t<false, C, !EXACT>(sc.prims, nullptr, sc.boxes, (int)p.scene.n_prims, o, dir, cmin, cmax, -1, nullptr);
    f.scans++;
    if (f.h.prim >= 0) return far ? FL_HIT_FAR : FL_HIT;
    if (far) return FL_ESCAPED;
    f.travelled += len;
    f.steps++;
    f.free = bound.nearest - len;  // the bounds were taken at the chord's start (grid mode: unknown, 0 -- the next step reads the grid)
    f.rest = p.scene.lens_skip == 3 ? len : bound.rest - len;
    f.near = bound.sphere;
    return (f.travelled >= tmax || f.steps >= p.scene.max_steps) ? FL_ESCAPED : FL_FLY;
}
// the event of a resolved flight
template <bool EXACT>
BT_DEV Traced flight_result(int state, P3 x, P3 v, const Flight& f) {
    Traced r;
    const bool chord = state == FL_HIT;
    r.o = v3(chord ? f.xp : x);
    r.d = normalize_fma<EXACT>(chord ? x - f.xp : v, 0);
    r.h = f.h;
    if (state >= FL_ESCAPED) r.h.prim = -1;
    r.captured = state == FL_CAPTURED;
    r.t_total = f.travelled + f.h.t;
    r.steps = f.steps;
    r.scans = f.scans;
    return r;
}

// One "ray" of the render loop, start to end (the probe kernel; the render kernel interleaves the
// phases of its 32 lanes instead, see render_body).
template <bool LENS, bool EXACT, bool BVH, class L>
BT_DEV Traced trace_ray(const RenderParams& p, const SceneView& sc, const L& lens, V3 o, V3 d, float tmin, float tmax, int vol_obj) {
    if (!LENS || vol_obj >= 0) return trace_straight<BVH>(p, sc, o, d, tmin, tmax, vol_obj);
    Flight f;
    flight_reset(f);
    P3 x = p3(o), v = p3(d);
    int st = FL_FLY;
#pragma unroll 1
    while (st < FL_HIT) {
        st = geodesic_step<EXACT, CT_ALL>(p, lens, sc.prims, x, v, f, tmax);
        if (st == FL_PEND || st == FL_PEND_FAR) st = geodesic_scan<EXACT, BVH>(p, sc, x, v, f, st, tmin, tmax);
    }
    return flight_result<EXACT>(st, x, v, f);
}

// NL: 0 = lens table walked in shared memory, N > 0 = exactly N masses held in registers
template <int NL>
struct LensSel {
    typedef LensRegs<NL> type;
    static BT_DEV type make(const float4* p, int) { return type(p); }
};
template <>
struct LensSel<0> {
    typedef LensShared type;
    static BT_DEV type make(const float4* p, int n) {
        LensShared l;
        l.p = p;
        l.count = n;
        return l;
    }
};

// what an event does next
enum { EV_TERMINAL = 0, EV_DIFFUSE = 1, EV_SPECULAR = 2 /* metallic, glass */, EV_VOLUME = 3 };
// how its new direction is sampled: every variant consumes the same two u32 draws (r1, r2)
enum { SK_NONE = 0, SK_COSINE = 1, SK_HEMI = 2, SK_SPHERE = 3, SK_RECT = 4 };

// The state a path carries from event to event (the recursion of ChunkState::sample, mod.rs:322-342, unrolled):
// its RNG stream, the throughput T, the bounce / volume-bounce counters, the volume being marched and the
// first-hit AOV latches (mod.rs:306-315).
struct PathQ {
    Rng rng;
    V3 T;
    uint32_t bounce, vb;
    int vol_obj;
    bool latched;
    V3 aov_albedo, aov_normal;
    float aov_depth;
};
BT_DEV void path_reset(PathQ& q) {
    q.T = v3(1.0f, 1.0f, 1.0f);
    q.bounce = 0;
    q.vb = 0;
    q.vol_obj = -1;
    q.latched = false;
    q.aov_albedo = v3(0.0f, 0.0f, 0.0f);
    q.aov_normal = v3(0.0f, 0.0f, 0.0f);
    q.aov_depth = __int_as_float(0x7f800000);
}

// One event of a path: classify the traced segment (sample_root / sample_surface / sample_volume), draw the
// new direction with the shared sampler and update the path state.  Returns true when the path ends --
// `contrib` is then what Chunk::write_* adds to the pixel for this path (buffer.rs:222-260); otherwise
// (o, d) is the scattered ray.  Called by every lane that holds an event; the three stages below are
// laid out so that the lanes of a warp meet again at the sampler and at the scattered-ray code.
template <int C>
BT_DEV bool shade_event(const RenderParams& p, const SceneView& sc, const Consts& k, const Traced& tr, PathQ& q, V3& o, V3& d,
                        V3& contrib) {
    const float inf = __int_as_float(0x7f800000);
    Rng& rng = q.rng;
    int ev = EV_TERMINAL, sk = SK_NONE;
    bool finish = false;
    V3 fin_color = v3(0.0f, 0.0f, 0.0f), fin_albedo = v3(0.0f, 0.0f, 0.0f), fin_normal = v3(0.0f, 0.0f, 0.0f);
    float fin_depth = inf;
    V3 pos = tr.o, nrm = tr.d, A = q.T, dir0 = tr.d;  // event geometry (defaults are placeholders)
    const V3 din = tr.d;
    float rough = 0.0f;
    const float hit_t = tr.t_total;
    int face = 0, hit_obj = -1;
    const float4* light = sc.lights;   // the light object picked by a Diffuse event (its pdf)
    const float4* lsamp = sc.lights;   // the record its point is sampled from (a cuboid's face)
    bool vol_scatter = false;
    const bool in_volume = (C & CT_VOLUMES) && q.vol_obj >= 0;

    // ---- 1. classify the event ----------------------------------------------------------------
    if (tr.h.prim < 0) {
        finish = true;
        if (!tr.captured) {  // sample_root, mod.rs:429-452 (times the environment map in the escape direction)
            fin_color = v3(p.scene.root_color[0], p.scene.root_color[1], p.scene.root_color[2]);
            if (p.env_w != 0) fin_color = fin_color * env_lookup(p.env, p.env_w, p.env_h, tr.d);
            fin_albedo = v3(p.scene.root_albedo[0], p.scene.root_albedo[1], p.scene.root_albedo[2]);
            if (p.scene.root_keeps_normal) {
                fin_normal = -tr.d;
                fin_depth = p.clip_max;
            }
        }
    } else {
        const Surface s = resolve_hit<C>(sc.prims, tr.h, tr.o, tr.d);
        pos = s.position;
        nrm = s.normal;
        face = s.face;
        hit_obj = s.obj;
        if (!(C & CT_VOLUMES) || s.face <= 1) {
            // ---- sample_surface, mod.rs:454-486 + Material::shade, material.rs:81-199 ----
            const float4 m0 = sc.mats[s.mat * MAT_STRIDE], m1 = sc.mats[s.mat * MAT_STRIDE + 1];
            const int mk = __float_as_int(m0.w);
            A = v3(m0);
            if (mk == MAT_FLAT) {
                finish = true;  // ColorData::from_emitted(albedo)
                fin_color = A;
                fin_albedo = A;
            } else if (mk == MAT_EMISSIVE) {
                finish = true;
                fin_color = A * m1.z;
                fin_albedo = fin_color;
            } else if (mk == MAT_DIFFUSE) {
                ev = EV_DIFFUSE;
                light = sc.lights + uniform_index(rng, p.scene.n_lights, p.light_zone) * LIGHT_STRIDE;
                lsamp = light;
                if (gen_bool(rng, 0.5f)) {  // Pdf::Mix: true selects the light (material.rs:269-275)
                    if ((C & CT_CUBOID_LIGHT) && (C & CT_RECTS) && __float_as_int(light[0].x) == LIGHT_CUBOID) {
                        // Cuboid::random_point, cuboid.rs:48-54: WeightedIndex (one Uniform::new(0, total)
                        // draw, partition_point(w <= chosen)), then that face's Rect::random_point
                        const float4 c1 = light[1], c2 = light[2];
                        const float chosen = uniform_f32(rng, 0.0f, c2.y);
                        const int idx = (c1.x <= chosen) + (c1.y <= chosen) + (c1.z <= chosen) + (c1.w <= chosen) + (c2.x <= chosen);
                        lsamp = sc.lights + (__float_as_int(c2.z) + idx) * LIGHT_STRIDE;
                    }
                    const int lt = __float_as_int(lsamp[0].x);
                    sk = ((C & CT_SPHERES) && lt == LIGHT_SPHERE) ? SK_SPHERE : (((C & CT_RECTS) && lt == LIGHT_RECT) ? SK_RECT : SK_NONE);
                } else {
                    sk = SK_COSINE;
                }
            } else if (C & (CT_METAL | CT_GLASS)) {
                ev = EV_SPECULAR;
                sk = SK_HEMI;
                rough = m1.x;
                if (!(C & CT_GLASS) || ((C & CT_METAL) && mk == MAT_METALLIC)) {
                    dir0 = reflect(din, nrm);
                } else {  // MAT_GLASS, material.rs:231-261
                    float ior = m1.y;
                    if (s.face == 0) ior = m_rcp(ior);
                    const float cos_theta = fminf(dot(-din, nrm), 1.0f);
                    const float sin_theta = m_sqrt(1.0f - cos_theta * cos_theta);
                    const float fr = fresnel(din, nrm, ior);
                    if (ior * sin_theta > 1.0f || gen_bool(rng, fr))
                        dir0 = reflect(din, nrm);
                    else
                        dir0 = refract(din, nrm, ior);
                }
            }
        } else {
            // ---- sample_volume, mod.rs:488-523 + Volume::shade, volume.rs:26-60 ----
            ev = EV_VOLUME;
            if (!in_volume) q.vb = 0;  // entered from sample(): volume_bounce = 0
            const V3 bmin = v3(s.center.x - s.radius, s.center.y - s.radius, s.center.z - s.radius);
            const V3 bmax = v3(s.center.x + s.radius, s.center.y + s.radius, s.center.z + s.radius);
            const V3 coord = m_div(s.position - bmin, bmax - bmin);
            const float density = p.volume_step * density_trilinear(sc.vols + s.vol * VOL_STRIDE, sc.grids, coord);
            if (density >= 1.0f || gen_bool(rng, density)) {
                vol_scatter = true;
                sk = SK_SPHERE;
                if (s.face == 2) pos = pos - din * p.volume_step * standard_f32(rng);
            }
        }
    }

    // ---- 2. the shared direction sampler: two u32 draws, one sincos, one basis --------------
    // UnitSphere / UnitHemisphere / Cosine (math/distr.rs:7-103) and Rect::random_point
    // (rect.rs:82-86) all draw (r1, r2) in this order; only the combination differs.
    V3 vec = v3(0.0f, 0.0f, 0.0f);
    if (sk != SK_NONE) {
        const float4 l1 = lsamp[1], l2 = lsamp[2];
        const bool rect = (C & CT_RECTS) && sk == SK_RECT;
        const float r1 = uniform_f32(rng, rect ? l1.w : 0.0f, rect ? lsamp[3].w : k.tau_scale);
        const float r2 = uniform_f32(rng, rect ? l2.w : 0.0f, rect ? lsamp[4].w : k.one_scale);
        float cx = r1, sy = r2, z = 0.0f;
        V3 X = v3(l1), Y = v3(l2), Z = v3(0.0f, 0.0f, 0.0f);
        if (!rect) {
            float sn, cs;
            bt_sincos(r1, &sn, &cs);
            const float w = m_sqrt(sk == SK_COSINE ? r2 : r2 * (1.0f - r2));
            const float two = sk == SK_COSINE ? 1.0f : 2.0f;
            cx = cs * two * w;
            sy = sn * two * w;
            z = sk == SK_COSINE ? m_sqrt(1.0f - r2) : (((C & (CT_METAL | CT_GLASS)) && sk == SK_HEMI) ? 1.0f - r2 : 1.0f - 2.0f * r2);
            X = v3(1.0f, 0.0f, 0.0f);
            Y = v3(0.0f, 1.0f, 0.0f);
            Z = v3(0.0f, 0.0f, 1.0f);
            if (sk != SK_SPHERE) {
                Z = normalize_s(nrm);
                any_orthonormal_pair(Z, X, Y);
            }
        }
        vec = (X * cx + Y * sy) + Z * z;
    }

    // ---- 3. the scattered ray ------------------------------------------------------------
    if (ev != EV_TERMINAL) {
        V3 dirvec = vec;  // Cosine, volume scatter
        if (ev == EV_DIFFUSE && sk != SK_COSINE) {  // Pdf::Light: random_point(light) - origin
            V3 point = v3(lsamp[1]);                                        // POINT: the translation
            if (sk == SK_SPHERE) point = v3(lsamp[1]) + vec * lsamp[1].w;   // sphere.rs:40-42
            if (sk == SK_RECT) point = mat_vec(v3(lsamp[3]), v3(lsamp[4]), v3(lsamp[5]), vec) + v3(lsamp[6]);
            dirvec = point - pos;
        }
        if ((C & (CT_METAL | CT_GLASS)) && ev == EV_SPECULAR) dirvec = dir0 + vec * rough;
        if (ev == EV_VOLUME && !vol_scatter) dirvec = din;
        const V3 nd = normalize_a(dirvec);  // Ray::new

        if ((C & CT_VOLUMES) && ev == EV_VOLUME) {
            o = pos;
            d = nd;
            if (vol_scatter) {
                if ((C & CT_AOV) && !q.latched) {
                    q.latched = true;
                    q.aov_albedo = v3(0.8f, 0.8f, 0.8f);
                    q.aov_normal = nrm;
                    q.aov_depth = hit_t;
                }
                q.T = q.T * 0.8f;
            }
            if (face == 4) {  // VolumeBack: leave the medium through sample(ray, bounce + 1)
                q.vol_obj = -1;
                ++q.bounce;
                if (q.bounce > p.max_bounces) finish = true;
            } else {          // keep marching: sample_volumetric(.., volume_bounce + 1)
                q.vol_obj = hit_obj;
                ++q.vb;
                if (q.vb > p.max_volume_bounces) finish = true;
            }
        } else {
            float pdf = 1.0f, mpdf = 1.0f;
            if (ev == EV_DIFFUSE) {
                mpdf = dot(nrm, nd) * 0.318309886183790671538f;
                const float pb = light_pdf<C>(sc.prims, sc.lights, light, pos, nd, p.clip_min, p.clip_max);
                pdf = lerpf(mpdf, pb, 0.5f);
            }
            if (fabsf(pdf) <= 1e-5f) {
                finish = true;  // no scatter: from_emitted(BLACK)
            } else {
                if ((C & CT_AOV) && !q.latched) {
                    q.latched = true;
                    q.aov_albedo = A;
                    q.aov_normal = nrm;
                    q.aov_depth = hit_t;
                }
                q.T = q.T * ((A * mpdf) * m_rcp(pdf));
                o = pos;
                d = nd;
                q.vol_obj = -1;
                ++q.bounce;
                if (q.bounce > p.max_bounces) finish = true;  // sample(): black, AOVs already latched
            }
        }
    }

    if (finish) {
        if ((C & CT_AOV) && !q.latched) {
            q.aov_albedo = fin_albedo;
            q.aov_normal = fin_normal;
            q.aov_depth = fin_depth;
        }
        switch ((C & CT_AOV) ? p.output : 0) {  // mod.rs:306-315
            case 0:  // (rounded separately from the pixel sum in every flavour: the product may travel through shared memory)
                contrib = v3(__fmul_rn(q.T.x, fin_color.x), __fmul_rn(q.T.y, fin_color.y), __fmul_rn(q.T.z, fin_color.z));
                break;
            case 1: contrib = q.aov_albedo; break;
            case 2: contrib = q.aov_normal; break;
            default: {
                float dn = (q.aov_depth - p.clip_min) * m_rcp(p.clip_max - p.clip_min);
                dn = fminf(fmaxf(dn, 0.0f), 1.0f);
                contrib = v3(dn, dn, dn);
            }
        }
    }
    return finish;
}

template <bool STATS, bool LENS, bool EXACT, int NL, bool BVH, int C>
BT_DEV void render_body(const RenderParams& p) {
    extern __shared__ float4 smem[];
    const SceneView sc = stage_scene<BVH>(p, smem);
    const typename LensSel<NL>::type lens = LensSel<NL>::make(sc.lens, (int)p.scene.n_lens);
    Consts k;
    k.tau_scale = p.tau_scale;
    k.one_scale = p.one_scale;

    // block = 16x16 pixels, warp = 8x4 pixel tile (coherent first hits, 128 B framebuffer rows)
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t px = blockIdx.x * 16 + (warp & 1) * 8 + (lane & 7);
    const uint32_t py = p.row0 + blockIdx.y * (blockDim.x >> 4) + (warp >> 1) * 4 + (lane >> 3);  // 256 threads: 16 rows, 128: 8
    const bool valid = px < p.width && py < p.row_end;
    const uint64_t pixel = (uint64_t)py * p.width + px;
    const float inf = __int_as_float(0x7f800000);
    // path_seed(seed, pixel, index) with its pixel-dependent prefix hoisted out of the path loop
    const uint64_t pixel_key = splitmix_mix(splitmix_mix(p.seed + 0x9e3779b97f4a7c15ULL) + 0x9e3779b97f4a7c15ULL * (pixel + 1));

    V3 acc = v3(0.0f, 0.0f, 0.0f);
    uint32_t path = 0;
    uint32_t sub_i = 0, sub_j = 0;  // sub-pixel of the next path: path_base is a multiple of sub_count, so a call starts at (0, 0)
    bool alive = false, done = !valid;
    uint32_t st_scans = 0, st_steps = 0, st_events = 0;  // STATS only

    // per-path state
    PathQ q;
    path_reset(q);
    V3 o, d;
    Flight fl;  // LENS: the geodesic this lane is flying (x, v alias o, d)
    flight_reset(fl);
    int fstate = FL_FLY;
    BvhTrav btrav;  // BVH && !LENS: the traversal this lane is in
    BvhSpill bspill;
    const BvhStack bstack = bvh_lane_stack(sc.stack, bspill, p.bvh_stack_k);
    bvh_begin(btrav, 0.0f);
    int bstate = 0;  // 0 none, 1 traversing, 2 done

    uint32_t regen_waited = 0;
#pragma unroll 1
    for (;;) {
        // Regeneration phase (ray generation is ~400 instructions): run it for all idle lanes at once,
        // and only when enough of them are idle -- in a warp that marches through a volume or flies
        // long geodesics a lane ends a path every few iterations, and regenerating one lane at a time
        // would execute this block nearly every iteration with 1/32 of the warp.
        const unsigned m_idle = __ballot_sync(0xffffffffu, !alive && !done);
        const bool regen = m_idle != 0 && ((uint32_t)__popc(m_idle) >= p.regen_lanes || ++regen_waited >= p.regen_patience ||
                                           !__any_sync(0xffffffffu, alive));
        if (regen) regen_waited = 0;
        if (regen && !alive && !done) {
            if (path < p.paths_per_pixel) {
                q.rng.seed_from_u64(splitmix_mix(pixel_key + 0xd1342543de82ef95ULL * (p.path_base + path + 1)));
                camera_ray(p.cam, k, q.rng, px, py, sub_i, sub_j, o, d);
                if (++sub_i == p.cam.sub_n) {  // the next path's sub-pixel, counted instead of divided out
                    sub_i = 0;
                    if (++sub_j == p.cam.sub_n) sub_j = 0;
                }
                path_reset(q);
                flight_reset(fl);
                fstate = FL_FLY;
                alive = true;
                ++path;
            } else {
                done = true;
            }
        }
        if (__all_sync(0xffffffffu, done)) break;

        // ---- 1. trace one segment ---------------------------------------------------------------
        const bool in_volume = (C & CT_VOLUMES) && q.vol_obj >= 0;

        // Per-warp phase compaction: a bent ray is NOT traced to its end here.  Lanes in flight are
        // in one of two phases -- STEP (an RK4 step; chords shorter than the free distance commit at
        // once) or INTERSECT (a pending chord against the scene).  Every turn of the loop below runs
        // the STEP phase for the lanes that can step, and the INTERSECT phase only once enough lanes
        // have a chord pending (ballot / popc), so the expensive scan runs with a well-filled warp.
        // The warp leaves the loop to shade / regenerate as soon as enough lanes hold a resolved
        // segment; lanes still in flight keep their phase and resume next time.
        Traced tr;
        bool has_event = false;
        if (BVH && !LENS) {
            // BVH phase compaction: a traversal alternates between inner-node visits and leaf tests, and the
            // lanes of a warp want different ones at any moment.  Every turn runs ONE kind of unit -- the
            // kind more lanes are waiting for -- so neither runs with a handful of lanes while the rest
            // idle (one unit = descend-to-leaf + leaf ran the descent at 6.8 lanes: profiles/r2_ncu_bvh.md).
            // The warp leaves to shade once enough lanes are done, the others resume.
            // (Scenes with volumetric spheres never use the BVH, so every segment here is a full ray.)
            if (alive && bstate == 0) {
                bvh_begin(btrav, p.clip_max);
                bstate = 1;
            }
            const V3 inv = v3(m_rcp(d.x), m_rcp(d.y), m_rcp(d.z));
            const uint32_t sgn = bvh_signs(inv);
            uint32_t waited = 0;
#pragma unroll 1
            for (;;) {
                const bool at_leaf = (btrav.cur & BVH_LEAF) != 0;
                const unsigned m_node = __ballot_sync(0xffffffffu, bstate == 1 && !at_leaf);
                const unsigned m_leaf = __ballot_sync(0xffffffffu, bstate == 1 && at_leaf);
                if ((m_node | m_leaf) == 0) break;
                if (__popc(m_node) >= __popc(m_leaf)) {
                    if (bstate == 1 && !at_leaf) bvh_node(btrav, sc.nodes, bstack, o, inv, sgn, p.clip_min);
                } else {
                    if (bstate == 1 && at_leaf) bvh_leaf(btrav, sc.prims, bstack, o, d, p.clip_min);
                }
                if (bstate == 1 && btrav.cur == BVH_DONE) bstate = 2;
                const unsigned m_done = __ballot_sync(0xffffffffu, bstate == 2);
                if (m_done != 0 && ((uint32_t)__popc(m_done) >= p.compact_lanes || ++waited >= p.compact_patience)) break;
            }
            if (bstate == 2) {
                tr.h = btrav.h;
                tr.o = o;
                tr.d = d;
                tr.t_total = btrav.h.t;
                tr.steps = 0;
                tr.scans = 1;
                tr.captured = false;
                has_event = true;
                bstate = 0;
            }
        } else if (alive && (!LENS || in_volume)) {
            tr = trace_straight<BVH, C>(p, sc, o, d, in_volume ? 0.0f : p.clip_min, in_volume ? p.volume_step : p.clip_max, q.vol_obj);
            has_event = true;
        }
        if (LENS) {
            int ls = !alive ? FL_IDLE : (in_volume ? FL_STRAIGHT : fstate);
            const uint32_t patience = __any_sync(0xffffffffu, ls == FL_STRAIGHT) ? 4u : p.compact_patience;  // straight (volume-march) lanes wait less
            uint32_t waited = 0, scan_waited = 0;
            P3 x = p3(o), v = p3(d);
#pragma unroll 1
            for (;;) {
#pragma unroll 1
                for (uint32_t r = 0; r < p.steps_per_turn; ++r)  // several steps per turn amortise the ballots below
                    if (ls == FL_FLY) ls = geodesic_step<EXACT, C>(p, lens, sc.prims, x, v, fl, p.clip_max);
                const bool pend = ls == FL_PEND || ls == FL_PEND_FAR;
                unsigned m_pend = __ballot_sync(0xffffffffu, pend);
                unsigned m_fly = __ballot_sync(0xffffffffu, ls == FL_FLY);
                if (m_pend != 0 && (m_fly == 0 || (uint32_t)__popc(m_pend) >= p.scan_lanes || ++scan_waited >= p.scan_patience)) {
                    scan_waited = 0;
                    if (pend) ls = geodesic_scan<EXACT, BVH, C>(p, sc, x, v, fl, ls, p.clip_min, p.clip_max);
                    m_pend = 0;
                    m_fly = __ballot_sync(0xffffffffu, ls == FL_FLY);
                }
                if ((m_fly | m_pend) == 0) break;
                const unsigned waiting = __ballot_sync(0xffffffffu, (ls & 4) != 0);
                if (waiting != 0 && ((uint32_t)__popc(waiting) >= p.compact_lanes || ++waited >= patience)) break;
            }
            o = v3(x);
            d = v3(v);
            if (ls < FL_IDLE) {
                fstate = ls;
                if (ls >= FL_HIT) {
                    tr = flight_result<EXACT>(ls, x, v, fl);
                    has_event = true;
                }
            }
        }
        // ---- 2. classify + shade the event, sample the scattered ray (shade_event) ----------------
        if (alive && has_event) {
            if (STATS) {
                st_scans += tr.scans;
                st_steps += tr.steps;
                st_events++;
            }
            V3 contrib;
            if (shade_event<C>(p, sc, k, tr, q, o, d, contrib)) {
                acc = v3(__fadd_rn(acc.x, contrib.x), __fadd_rn(acc.y, contrib.y), __fadd_rn(acc.z, contrib.z));
                alive = false;
            } else {
                flight_reset(fl);  // the scattered ray starts a new flight
                fstate = FL_FLY;
            }
        }
    }

    if (valid) {  // Buffer::write_color: rgb += value, alpha untouched (buffer.rs:159-178)
        float4 v = p.fb[pixel];
        v.x += acc.x;
        v.y += acc.y;
        v.z += acc.z;
        p.fb[pixel] = v;
    }
    if (STATS) {
        const uint32_t a = __reduce_add_sync(0xffffffffu, valid ? path : 0u), b = __reduce_add_sync(0xffffffffu, st_scans);
        const uint32_t c = __reduce_add_sync(0xffffffffu, st_steps), e = __reduce_add_sync(0xffffffffu, st_events);
        if (lane == 0) {
            atomicAdd(p.stats + 0, (unsigned long long)a);
            atomicAdd(p.stats + 1, (unsigned long long)b);
            atomicAdd(p.stats + 2, (unsigned long long)c);
            atomicAdd(p.stats + 3, (unsigned long long)e);
        }
    }
}

// Lensed variants carry the flight state on top of the path state: 128-thread CTAs at 5 per SM give
// them 96 registers (20 warps / SM) instead of 80 with spills (24 warps / SM).  The flat variants keep
// the 85-register cap of (256, 3) and are launched with 128 threads as well (launch_lane).
#ifndef BT_BVH_CTAS
#define BT_BVH_CTAS 7  // (measured 4 .. 7: the traversal is latency-bound, every CTA more is +6 .. +15 %)
#endif
template <bool LENS, bool EXACT, int NL, bool BVH, int C = CT_ALL>
__global__ void __launch_bounds__(128, LENS ? 5 : (BVH ? BT_BVH_CTAS : 7)) render_kernel(const __grid_constant__ RenderParams p) {
    render_body<false, LENS, EXACT, NL, BVH, C>(p);
}
// the same kernel + work counters for bench.py's roofline accounting (never timed)
template <bool LENS, bool EXACT, int NL, bool BVH, int C = CT_ALL>
__global__ void __launch_bounds__(256, 2) render_kernel_stats(const __grid_constant__ RenderParams p) {
    render_body<true, LENS, EXACT, NL, BVH, C>(p);
}

#include "render_pool.cuh"
// 128-thread CTAs: five of a lensed variant per SM (20 warps at <= 96 registers; 32 W slots x 64 B of shared memory
// per warp), six of a flat one.
#define BT_POOL_BOUNDS(LENS) __launch_bounds__(128, (LENS) ? 5 : 6)
template <bool LENS, bool EXACT, int NL, int C = CT_ALL>
__global__ void BT_POOL_BOUNDS(LENS) render_pool_kernel(const __grid_constant__ RenderParams p) {
    render_pool_body<LENS, EXACT, NL, C>(p);
}
// BVH scenes under a flat field: the scan is a pooled traversal (NODE / LEAF phases)
#ifndef BT_BVH_POOL_CTAS
#define BT_BVH_POOL_CTAS 5  // (96 registers, no spills; W = 3: 238 Msamples/s on the 32 k-primitive scene against 223 .. 232 at 6 CTAs x 80 registers, W = 2)
#endif
template <int C>
__global__ void __launch_bounds__(128, BT_BVH_POOL_CTAS) render_pool_bvh_kernel(const __grid_constant__ RenderParams p) {
    render_pool_body<false, false, 0, C, false, true>(p);
}
// the same kernel + scheduling counters (bt_render_pool_stats; the content-specialised variants only; never timed)
template <bool LENS, bool EXACT, int NL, int C>
__global__ void BT_POOL_BOUNDS(LENS) render_pool_kernel_pstats(const __grid_constant__ RenderParams p) {
    render_pool_body<LENS, EXACT, NL, C, true>(p);
}

template <bool LENS, bool EXACT, int NL, bool BVH>
__global__ void __launch_bounds__(256) trace_kernel(const __grid_constant__ RenderParams p, uint32_t n, const float* __restrict__ origins,
                                                    const float* __restrict__ dirs, DeviceSegment* __restrict__ out) {
    extern __shared__ float4 smem[];
    const SceneView sc = stage_scene<BVH>(p, smem);
    const typename LensSel<NL>::type lens = LensSel<NL>::make(sc.lens, (int)p.scene.n_lens);
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;  // (after the staging barrier)
    V3 o = v3(origins[3 * i], origins[3 * i + 1], origins[3 * i + 2]);
    V3 d = v3(dirs[3 * i], dirs[3 * i + 1], dirs[3 * i + 2]);
    Traced tr = trace_ray<LENS, EXACT, BVH>(p, sc, lens, o, d, p.clip_min, p.clip_max, -1);
    DeviceSegment seg;
    seg.steps = tr.steps;
    seg.obj = -1;
    seg.t = 0.0f;
    for (int c = 0; c < 3; ++c) seg.position[c] = seg.normal[c] = seg.direction[c] = 0.0f;
    if (tr.h.prim >= 0) {
        Surface s = resolve_hit(sc.prims, tr.h, tr.o, tr.d);
        seg.face = s.face;
        seg.obj = s.obj;
        seg.t = tr.t_total;
        seg.position[0] = s.position.x; seg.position[1] = s.position.y; seg.position[2] = s.position.z;
        seg.normal[0] = s.normal.x; seg.normal[1] = s.normal.y; seg.normal[2] = s.normal.z;
        seg.direction[0] = tr.d.x; seg.direction[1] = tr.d.y; seg.direction[2] = tr.d.z;
    } else if (tr.captured) {
        seg.face = -2;
    } else {
        seg.face = -1;
        seg.position[0] = tr.o.x; seg.position[1] = tr.o.y; seg.position[2] = tr.o.z;
        seg.direction[0] = tr.d.x; seg.direction[1] = tr.d.y; seg.direction[2] = tr.d.z;
    }
    out[i] = seg;
}

__global__ void camera_rays_kernel(const __grid_constant__ RenderParams p, uint32_t n, const uint32_t* __restrict__ xs,
                                   const uint32_t* __restrict__ ys, const uint64_t* __restrict__ path_index, float* __restrict__ out) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    Consts k;
    k.tau_scale = p.tau_scale;
    k.one_scale = p.one_scale;
    Rng rng;
    const uint64_t pixel = (uint64_t)ys[i] * p.width + xs[i];
    rng.seed_from_u64(path_seed(p.seed, pixel, p.path_base + path_index[i]));
    V3 o, d;
    const uint32_t sub = (uint32_t)(path_index[i] % p.sub_count);
    camera_ray(p.cam, k, rng, xs[i], ys[i], sub % p.cam.sub_n, sub / p.cam.sub_n, o, d);
    out[6 * i] = o.x; out[6 * i + 1] = o.y; out[6 * i + 2] = o.z;
    out[6 * i + 3] = d.x; out[6 * i + 4] = d.y; out[6 * i + 5] = d.z;
}

// The geodesic stepper in isolation: n_steps RK4 steps per ray, state in registers, the lens
// table in shared memory.  No memory traffic in the loop: this is the FP32-roofline kernel.
template <bool EXACT, int NL>
__global__ void __launch_bounds__(256) integrate_kernel(const __grid_constant__ IntegrateParams p) {
    extern __shared__ float4 slens[];
    for (uint32_t i = threadIdx.x; i < p.n_lens * LENS_STRIDE; i += blockDim.x)
        slens[i] = p.n_lens <= INTEGRATE_INLINE_LENSES ? p.inline_lens[i] : p.lens[i];
    __syncthreads();
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= p.n) return;
    float* s = p.xv + 6 * (size_t)i;
    P3 x = p3(make_float2(s[0], s[1]), s[2]), v = p3(make_float2(s[3], s[4]), s[5]);
    const typename LensSel<NL>::type lens = LensSel<NL>::make(slens, (int)p.n_lens);
#pragma unroll 1
    for (uint32_t it = 0; it < p.n_steps; ++it) {
        float rmin;
        bool captured, far;
        D0Cache<typename LensSel<NL>::type> cache;
        P3 k1 = lens_accel<1, EXACT, 0>(lens, cache, x, 0.0f, v, v, rmin, captured, far);
        rk4_from_k1<EXACT>(lens, cache, x, v, k1, step_size(p.kappa, p.h_min, p.h_max, rmin));
    }
    s[0] = x.xy.x; s[1] = x.xy.y; s[2] = x.z; s[3] = v.xy.x; s[4] = v.xy.y; s[5] = v.z;
}

// Buffer::preview, buffer.rs:117-138
BT_DEV float linear_to_srgb(float x) {  // color.rs:14-20
    if (x <= 0.0031308f) return 12.92f * x;
    return 1.055f * powf(x, 1.0f / 2.4f) - 0.055f;
}
BT_DEV unsigned char f32_to_u8(float x) {  // color.rs:22-24, Rust saturating cast (NaN -> 0)
    float v = x * 255.0f;
    if (!(v > 0.0f)) return 0;
    if (v >= 255.0f) return 255;
    return (unsigned char)v;
}
__global__ void resolve_kernel(const float4* __restrict__ fb, uint32_t n, float samples_recip, int color_space, uchar4* __restrict__ out) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const float4 px = fb[i];
    V3 c = v3(px.x, px.y, px.z) * samples_recip;
    if (color_space == 1) {
        c = (normalize_s(c) + v3(1.0f, 1.0f, 1.0f)) * 0.5f;
    } else if (color_space == 3) {
        c = v3(linear_to_srgb(c.x), linear_to_srgb(c.y), linear_to_srgb(c.z));
    }
    uchar4 o;
    o.x = f32_to_u8(c.x);
    o.y = f32_to_u8(c.y);
    o.z = f32_to_u8(c.z);
    o.w = f32_to_u8(px.w);
    out[i] = o;
}

// The framebuffer reduce of a multi-device render: dst.rgb += sum of the peers' slices (Buffer::write_color over
// the slices rendered on the other GPUs; alpha untouched).  The peers' frames are read IN PLACE through peer
// mappings (NVLink / NVSwitch loads, coalesced float4): the transfer and the sum are one kernel on the device that
// owns the caller's frame, and no staging copy of W x H x 16 B per peer exists.
__global__ void __launch_bounds__(256) accumulate_frames_kernel(float4* __restrict__ dst, const PeerFrames pf, uint32_t n_pixels) {
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n_pixels; i += gridDim.x * blockDim.x) {
        float4 v = dst[i];
#pragma unroll 1
        for (int g = 0; g < pf.n; ++g) {
            const float4 s = pf.src[g][i];
            v.x += s.x;
            v.y += s.y;
            v.z += s.z;
        }
        dst[i] = v;
    }
}

// FP32 peak probe: FP32_PEAK_CHAINS independent FMA chains per thread.
__global__ void __launch_bounds__(FP32_PEAK_THREADS) fp32_peak_kernel(float* out, uint32_t iters) {
    float a[FP32_PEAK_CHAINS];
    const float m = 1.0f + 1e-7f * (float)threadIdx.x, c = 1e-9f * (float)blockIdx.x;
#pragma unroll
    for (int j = 0; j < FP32_PEAK_CHAINS; ++j) a[j] = (float)j;
#pragma unroll 1
    for (uint32_t it = 0; it < iters; ++it) {
#pragma unroll
        for (int u = 0; u < FP32_PEAK_UNROLL; ++u)
#pragma unroll
            for (int j = 0; j < FP32_PEAK_CHAINS; ++j) a[j] = fmaf(a[j], m, c);
    }
    float s = 0.0f;
#pragma unroll
    for (int j = 0; j < FP32_PEAK_CHAINS; ++j) s += a[j];
    out[blockIdx.x * blockDim.x + threadIdx.x] = s;
}

template <class K>
cudaError_t ensure_smem(K kernel, size_t bytes) {
    if (bytes > 48 * 1024) return cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
    return cudaSuccess;
}

}  // namespace

#ifndef BT_EXACT_SCAN
size_t render_pool_arena_bytes(uint32_t pool_w, int sm_count, bool bvh) {
    return 256 /* the tile counter */ + (size_t)sm_count * 8 /* CTAs per SM at most */ * (bvh ? 4 : 6) /* warps per CTA at most */ * pool_q_bytes(pool_w, bvh);
}
size_t render_smem_bytes(const RenderParams& p, unsigned threads) {
    return (size_t)p.scene.stage_f4 * sizeof(float4) + (p.scene.n_bvh ? (size_t)BVH_STACK_SMEM * threads * 2 * sizeof(uint32_t) : 0);
}

#endif

namespace {
// persistent grid of the pooled kernel: as many CTAs as fit the GPU at once, or fewer when the frame has fewer
// 8 x 4 tiles than that (the warps draw their tiles from one counter: render_pool.cuh)
template <class K>
cudaError_t launch_pool(K kernel, const RenderParams& p, bool lens, cudaStream_t stream) {
    const unsigned cap = 128;  // BT_POOL_BOUNDS
    const unsigned threads = p.pool_threads ? std::min(p.pool_threads, cap) : cap, warps = threads / 32;
    const bool bvh = p.scene.n_bvh != 0;
    const size_t smem = (size_t)p.scene.stage_f4 * sizeof(float4) + warps * pool_warp_bytes(p.pool_w, lens, bvh);
    cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    int per_sm = 0, dev = 0, sms = 0;
    if ((e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, (int)threads, smem)) != cudaSuccess) return e;
    if ((e = cudaGetDevice(&dev)) != cudaSuccess) return e;
    if ((e = cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev)) != cudaSuccess) return e;
    if (per_sm < 1) return cudaErrorInvalidConfiguration;
    const uint64_t tiles = (uint64_t)((p.width + 7) / 8) * ((p.row_end - p.row0 + 3) / 4);
    const uint64_t need = (tiles + warps - 1) / warps, fit = (uint64_t)per_sm * sms;
    const uint64_t room = p.pool_q_cap / (pool_q_bytes(p.pool_w, bvh) * warps);  // CTAs the path-state arena has room for
    if (room < 1 || !p.pool_q || !p.pool_counter) return cudaErrorMemoryAllocation;
    if ((e = cudaMemsetAsync(p.pool_counter, 0, sizeof(unsigned long long), stream)) != cudaSuccess) return e;
    kernel<<<(unsigned)std::max<uint64_t>(1, std::min(std::min(need, fit), room)), threads, smem, stream>>>(p);
    return cudaGetLastError();
}

// the lane kernels: a CTA renders 16 x (threads / 16) pixels.  128-thread CTAs (16 x 8 pixels): at <= 72 registers seven
// of them fit an SM (28 warps) where three 256-thread CTAs gave 24 -- cornell2 +3.7 % (the work-counter variant keeps 256)
template <class K>
cudaError_t launch_lane(K kernel, const RenderParams& p, unsigned threads, cudaStream_t stream) {
    const uint32_t rows = p.row_end - p.row0, h = threads / 16;
    const size_t smem = render_smem_bytes(p, threads);
    cudaError_t e = ensure_smem(kernel, smem);
    if (e != cudaSuccess) return e;
    kernel<<<dim3((p.width + 15) / 16, (rows + h - 1) / h), threads, smem, stream>>>(p);
    return cudaGetLastError();
}

struct TraceArgs { uint32_t n; const float *origins, *dirs; DeviceSegment* out; };

// row I of the variant table (variants.h): the kernels of the families it lists, and nothing else, are instantiated
template <size_t I>
cudaError_t launch_variant(int family, const RenderParams& p, const TraceArgs& t, cudaStream_t stream) {
    constexpr Variant v = kVariants[I];
    constexpr int F = variant_families(v, kExactFlavour);
    if constexpr ((F & V_LANE) != 0) if (family == V_LANE) return launch_lane(render_kernel<v.lens, v.exact, v.nl, v.bvh, v.c>, p, 128, stream);
    if constexpr ((F & V_LANE_STATS) != 0) if (family == V_LANE_STATS) return launch_lane(render_kernel_stats<v.lens, v.exact, v.nl, v.bvh, v.c>, p, 256, stream);
    if constexpr ((F & V_POOL) != 0) if (family == V_POOL) return launch_pool(render_pool_kernel<v.lens, v.exact, v.nl, v.c>, p, v.lens, stream);
    if constexpr ((F & V_POOL_STATS) != 0) if (family == V_POOL_STATS) return launch_pool(render_pool_kernel_pstats<v.lens, v.exact, v.nl, v.c>, p, v.lens, stream);
    if constexpr ((F & V_POOL_BVH) != 0) if (family == V_POOL_BVH) return launch_pool(render_pool_bvh_kernel<v.c>, p, false, stream);
    if constexpr ((F & V_TRACE) != 0) if (family == V_TRACE) {
        const size_t smem = render_smem_bytes(p);
        cudaError_t e = ensure_smem(trace_kernel<v.lens, v.exact, v.nl, v.bvh>, smem);
        if (e != cudaSuccess) return e;
        trace_kernel<v.lens, v.exact, v.nl, v.bvh><<<(t.n + 255) / 256, 256, smem, stream>>>(p, t.n, t.origins, t.dirs, t.out);
        return cudaGetLastError();
    }
    return cudaErrorNotSupported;
}

template <size_t... I>
cudaError_t launch_row(int row, int family, const RenderParams& p, const TraceArgs& t, cudaStream_t stream, std::index_sequence<I...>) {
    static constexpr cudaError_t (*rows[])(int, const RenderParams&, const TraceArgs&, cudaStream_t) = {&launch_variant<I>...};
    return rows[row](family, p, t, stream);
}

// a call no row serves is an error (bt_render_pool_stats: BT_ERR_UNSUPPORTED), never a fall-back to another family
cudaError_t launch_family(int family, const RenderParams& p, const TraceArgs& t, cudaStream_t stream, uint64_t* launches) {
    const int row = select_variant(p, family, kExactFlavour);
    if (row < 0) return cudaErrorNotSupported;
    ++*launches;
    return launch_row(row, family, p, t, stream, std::make_index_sequence<kNumVariants>());
}
}  // namespace

cudaError_t BT_SFX(launch_render)(const RenderParams& p, cudaStream_t stream, uint64_t* launches) {
    return launch_family(render_family(p), p, TraceArgs{}, stream, launches);
}

cudaError_t BT_SFX(launch_trace)(const RenderParams& p, uint32_t n, const float* origins, const float* dirs,
                         DeviceSegment* out, cudaStream_t stream, uint64_t* launches) {
    if (n == 0) return cudaSuccess;
    return launch_family(V_TRACE, p, TraceArgs{n, origins, dirs, out}, stream, launches);
}

cudaError_t BT_SFX(launch_camera_rays)(const RenderParams& p, uint32_t n, const uint32_t* xs, const uint32_t* ys,
                               const uint64_t* path_index, float* out, cudaStream_t stream, uint64_t* launches) {
    if (n == 0) return cudaSuccess;
    camera_rays_kernel<<<(n + 255) / 256, 256, 0, stream>>>(p, n, xs, ys, path_index, out);
    ++*launches;
    return cudaGetLastError();
}

#ifndef BT_EXACT_SCAN
cudaError_t launch_integrate(const IntegrateParams& p, cudaStream_t stream, uint64_t* launches) {
    if (p.n == 0) return cudaSuccess;
    size_t smem = (size_t)p.n_lens * LENS_STRIDE * sizeof(float4);
    // BT_INTEGRATE_SMEM_PAD=<bytes>: extra dynamic shared memory per CTA, i.e. fewer resident warps per SM
    // (tools/occupancy_probe.py: how many warps the FMA-dense stepper needs to stay issue-bound)
    if (const char* pad = std::getenv("BT_INTEGRATE_SMEM_PAD")) smem += (size_t)std::atol(pad);
    cudaError_t e;
    const unsigned grid = (p.n + 255) / 256;
#define BT_INTEGRATE(EXACT, NL)                                                                \
    do {                                                                                       \
        if ((e = ensure_smem(integrate_kernel<EXACT, NL>, smem)) != cudaSuccess) return e;     \
        integrate_kernel<EXACT, NL><<<grid, 256, smem, stream>>>(p);                           \
    } while (0)
    if (p.exact) BT_INTEGRATE(true, 0);
    else if (p.n_lens == 1) BT_INTEGRATE(false, 1);
    else if (p.n_lens == 2) BT_INTEGRATE(false, 2);
    else if (p.n_lens == 4) BT_INTEGRATE(false, 4);
    else BT_INTEGRATE(false, 0);
#undef BT_INTEGRATE
    ++*launches;
    return cudaGetLastError();
}

cudaError_t launch_resolve(const float4* fb, uint32_t n_pixels, uint64_t samples, int color_space, uchar4* out,
                           cudaStream_t stream, uint64_t* launches) {
    if (n_pixels == 0) return cudaSuccess;
    float samples_recip = 1.0f / (float)samples;  // buffer.rs:124
    resolve_kernel<<<(n_pixels + 255) / 256, 256, 0, stream>>>(fb, n_pixels, samples_recip, color_space, out);
    ++*launches;
    return cudaGetLastError();
}

cudaError_t launch_accumulate_frames(float4* dst, const PeerFrames& pf, uint32_t n_pixels, int sm_count, cudaStream_t stream, uint64_t* launches) {
    if (n_pixels == 0 || pf.n == 0) return cudaSuccess;
    const unsigned blocks = (unsigned)std::min<uint64_t>(((uint64_t)n_pixels + 255) / 256, (uint64_t)sm_count * 8);
    accumulate_frames_kernel<<<blocks, 256, 0, stream>>>(dst, pf, n_pixels);
    ++*launches;
    return cudaGetLastError();
}

cudaError_t launch_fp32_peak(float* out, uint32_t iters, int blocks, cudaStream_t stream, uint64_t* launches) {
    fp32_peak_kernel<<<blocks, FP32_PEAK_THREADS, 0, stream>>>(out, iters);
    ++*launches;
    return cudaGetLastError();
}

#endif  // !BT_EXACT_SCAN

}  // namespace bt
