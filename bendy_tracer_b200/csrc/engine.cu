// engine.cu -- implementation of the C ABI in include/bendy_b200.h.
//
// Host side of the drop-in boundary: owns the CUDA device/stream, the parsed Scene and its
// flattened device buffers, merges Config/RenderConfig exactly like ChunkConfig::with_configs
// (reference src/tracer/mod.rs:218-229) and launches the kernels.  No CPU fallback.
#include "../../include/bendy_b200.h"

#include <cuda_runtime.h>

#include <algorithm>
#include <cctype>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

#include "kernels.h"
#include "scene.hpp"

using namespace bt;

namespace {
thread_local std::string g_error;
int fail(int code, const std::string& msg) {
    g_error = msg;
    return code;
}
int cuda_fail(cudaError_t e, const char* what) {
    return fail(BT_ERR_CUDA, std::string(what) + ": " + cudaGetErrorString(e));
}
#define CK(call)                                          \
    do {                                                  \
        cudaError_t e_ = (call);                          \
        if (e_ != cudaSuccess) return cuda_fail(e_, #call); \
    } while (0)
}  // namespace

// Scheduling knobs of the kernels: none of them changes an image.  Read from the environment ONCE, when the
// engine is created (BT_<NAME>), and settable per engine with bt_engine_set_tuning; -1 = the built-in default.
struct Tuning {
    int64_t compact_lanes = -1, compact_patience = -1, regen_lanes = -1, regen_patience = -1, scan_lanes = -1, scan_patience = -1;
    int64_t steps_per_turn = -1, lens_no_skip = -1, lens_dist_grid = -1, host_bands = -1;
    int64_t pool_w = -1, pool_refill = -1, pool_step_min = -1, pool_threads = -1, bvh_stack_k = -1;
};
struct TuningName {
    const char* name;
    int64_t Tuning::*field;
};
static const TuningName kTuning[] = {
    {"compact_lanes", &Tuning::compact_lanes}, {"compact_patience", &Tuning::compact_patience},
    {"regen_lanes", &Tuning::regen_lanes},     {"regen_patience", &Tuning::regen_patience},
    {"scan_lanes", &Tuning::scan_lanes},       {"scan_patience", &Tuning::scan_patience},
    {"steps_per_turn", &Tuning::steps_per_turn}, {"lens_no_skip", &Tuning::lens_no_skip}, {"lens_dist_grid", &Tuning::lens_dist_grid},
    {"host_bands", &Tuning::host_bands},
    {"pool_w", &Tuning::pool_w},               {"pool_refill", &Tuning::pool_refill},
    {"pool_step_min", &Tuning::pool_step_min}, {"pool_threads", &Tuning::pool_threads},
    {"bvh_stack_k", &Tuning::bvh_stack_k},
};

struct bt_engine {
    int device;
    Tuning tune;
    cudaStream_t stream;
    cudaStream_t stream2;   // second lane of the host-buffer pipeline (bt_render, BT_MEM_HOST)
    cudaEvent_t ev_fork, ev_join;
    uint64_t launches;
    // scratch for host-memory calls (every user synchronises before it returns)
    void* d_scratch;
    size_t scratch_bytes;
    // lens tables too large for the kernel parameters (bt_geodesic_integrate): their own buffer, guarded by an event
    // recorded after the kernel that reads it, because the device-memory flavour of that call does not synchronise
    float4* d_lens;
    size_t lens_cap;
    cudaEvent_t ev_lens;
    // path-state arenas of the pooled render kernel (render_pool.cuh), one per pipeline lane of bt_render: two launches
    // that may overlap (neighbouring row bands on the two streams) never share one
    char* d_pool_q[2];
    size_t pool_q_cap[2];
    int sm_count;
    int clock_khz;
    // ---- multi-device engine (bt_engine_create_multi): this engine is device 0 and owns the others ----
    std::vector<bt_engine*> peers;     // devices 1 .. n-1 (each a complete engine: stream, scratch frame, arenas)
    std::vector<char> peer_direct;     // its slice is readable from device 0 through a peer mapping (or lives on device 0)
    cudaEvent_t ev_slice;              // (on a peer) its slice of the frame is rendered
    cudaEvent_t ev_reduced;            // (on device 0) the last framebuffer reduce has read the peers' slices
    float4* d_stage;                   // (on device 0) staging frame for peers without a peer mapping
    size_t stage_cap;
};

struct bt_scene;
static bool use_exact(const bt_engine* e, const bt_scene* s);

// the device copy of a scene on one GPU (a multi-device engine keeps one per device)
struct SceneDev {
    int device;
    uint64_t version;   // FlatScene version this copy holds (0: none)
    cudaEvent_t ev_use; // recorded after every kernel that reads the copy: a re-upload waits for it
    float4* d_blob;
    size_t blob_cap;
    float* d_grids;
    size_t grids_cap;
    uint8_t* d_dist;    // free-distance grid (FlatScene::dist)
    size_t dist_cap;
    uint64_t env_version;  // bt_scene::env_version this copy's environment map holds
    float4* d_env;
    size_t env_cap;
};

struct bt_scene {
    bt_engine* engine;  // identity of the engine the scene is bound to (compared, never dereferenced: the engine may die first)
    Scene scene;
    FlatScene flat;
    uint64_t flat_version;  // bumped by every re-flatten
    int accel;          // ACCEL_AUTO / ACCEL_LINEAR / ACCEL_BVH
    int precision;      // BT_PRECISION_AUTO / _FAST / _EXACT
    bool flat_dirty;    // host flattening out of date: flatten from scratch
    // transform edits not yet applied to `flat` (bt_scene_apply_transform; applied by bt_scene_commit or the next render):
    // the objects whose world transform changed (the edited object and its descendants)
    std::vector<uint64_t> pending;
    // blob ranges (float4 offset, count) rewritten in place since the flattening of version patch_base: a device copy that is
    // at least that recent is brought up to date by uploading just these
    std::vector<std::pair<uint32_t, uint32_t> > patch;
    uint64_t patch_base;
    bool patch_dist;    // ... and the free-distance grid too
    // environment map (bt_scene_set_environment): env_w x env_h float4 texels (.w = 0), uploaded on its own -- setting or
    // clearing it never re-flattens the scene.  env_version is bumped by every set / clear (0: never set).
    std::vector<float4> env;
    uint32_t env_w, env_h;
    uint64_t env_version;
    std::vector<SceneDev> devs;
};

// Which arithmetic flavour of the kernels renders this scene.  AUTO: volumetric scenes are chaotic
// in their rounding (steep density gradients turn a 1-ulp position difference into a flipped
// scatter decision on ~5e-4 of the paths), so they get the bit-exact flavour; surface-only scenes
// get the fast one (image MAE vs the oracle ~1e-8 .. 1e-5).
static bool use_exact(const bt_engine*, const bt_scene* s) {
    if (s->precision == BT_PRECISION_AUTO) return s->flat.header.has_volume_prims != 0;
    return s->precision == BT_PRECISION_EXACT;
}

// The cells of the free-distance grid (layout.h: SceneHeader::dist_*; scene.cpp: build_dist_grid lays the grid out and holds
// the host version of exactly this arithmetic -- this file is compiled -fmad=false, so the two agree bit for bit).  One thread
// per cell: the lower bound, over all points of the cell, of the distance to the nearest primitive surface (spheres exactly,
// everything else through its world AABB -- the bound records of the blob), minus the rounding margins of the hit tests,
// in quanta of dist_q, rounded down.
__global__ void __launch_bounds__(256) dist_grid_kernel(const float4* __restrict__ blob, const SceneHeader h, uint8_t* __restrict__ out) {
    const uint64_t n_cells = (uint64_t)h.dist_nx * h.dist_ny * h.dist_nz;
    const uint64_t idx = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= n_cells) return;
    const uint32_t x = (uint32_t)(idx % h.dist_nx), y = (uint32_t)((idx / h.dist_nx) % h.dist_ny), z = (uint32_t)(idx / ((uint64_t)h.dist_nx * h.dist_ny));
    const double cell = (double)h.dist_cell;
    const double half_diag = 0.5 * sqrt(3.0) * cell * 1.01 + 1e-5;
    const double c[3] = {h.dist_lo[0] + (x + 0.5) * cell, h.dist_lo[1] + (y + 0.5) * cell, h.dist_lo[2] + (z + 0.5) * cell};
    const double l1 = fabs(c[0]) + fabs(c[1]) + fabs(c[2]) + 3.0 * half_diag;
    double best = 1e30;
    for (uint32_t i = 0; i < h.n_prims; ++i) {
        const float4* rec = blob + h.prim_off + (size_t)i * PRIM_STRIDE;
        double b;
        if ((__float_as_uint(rec[4].x) & 3u) == PRIM_SPHERE) {
            const float4 q0 = rec[0];
            const double dx = c[0] - q0.x, dy = c[1] - q0.y, dz = c[2] - q0.z, r = q0.w;
            const double dc = sqrt(dx * dx + dy * dy + dz * dz), dmax = dc + half_diag;
            b = fabs(dc - r) - (dmax * dmax * (double)rec[1].z + 2e-5 * (dmax + r) + 1e-6);
        } else {
            const float4 lo = blob[h.bound_off + (size_t)i * BOUND_STRIDE], hi = blob[h.bound_off + (size_t)i * BOUND_STRIDE + 1];
            const float blo[3] = {lo.x, lo.y, lo.z}, bhi[3] = {hi.x, hi.y, hi.z};
            double d2 = 0.0, ext = 0.0;
            for (int k = 0; k < 3; ++k) {
                const double d = fmax(fmax((double)blo[k] - c[k], c[k] - (double)bhi[k]), 0.0);
                d2 += d * d;
                ext += fabs((double)bhi[k] - (double)blo[k]);
            }
            b = sqrt(d2) - (1e-4 * (l1 + ext + sqrt(d2)) + 1e-4);
        }
        best = fmin(best, b);
    }
    const double v = floor((best - half_diag) / (double)h.dist_q);
    out[idx] = (uint8_t)fmin(fmax(v, 0.0), 255.0);
}

namespace {

int ensure_scratch(bt_engine* e, size_t bytes) {
    if (bytes <= e->scratch_bytes) return BT_OK;
    if (e->d_scratch) cudaFree(e->d_scratch);
    e->d_scratch = 0;
    e->scratch_bytes = 0;
    CK(cudaMalloc(&e->d_scratch, bytes));
    e->scratch_bytes = bytes;
    return BT_OK;
}

// Brings the scene's copy on the CURRENT device (cudaSetDevice done by the caller) up to date; *out = that copy.
// the free-distance grid of this device copy: filled by dist_grid_kernel from the blob just uploaded (or copied, when the host
// filled it: BT_DIST_GRID_HOST)
int upload_dist_grid(bt_scene* s, SceneDev* d, cudaStream_t stream) {
    const SceneHeader& h = s->flat.header;
    if (h.lens_skip != 3) return BT_OK;
    const size_t db = (size_t)h.dist_nx * h.dist_ny * h.dist_nz;
    if (db > d->dist_cap) {
        if (d->d_dist) cudaFree(d->d_dist);
        d->d_dist = 0;
        d->dist_cap = 0;
        CK(cudaMalloc((void**)&d->d_dist, db));
        d->dist_cap = db;
    }
    if (!s->flat.dist.empty()) {
        CK(cudaMemcpyAsync(d->d_dist, s->flat.dist.data(), db, cudaMemcpyHostToDevice, stream));
    } else {
        dist_grid_kernel<<<(unsigned)((db + 255) / 256), 256, 0, stream>>>(d->d_blob, h, d->d_dist);
        CK(cudaGetLastError());
    }
    return BT_OK;
}

// the host half of a scene update: from scratch, or -- for transform edits -- in place (update_flat: records rewritten, BVH refit)
void commit_scene(bt_scene* s) {
    if (!s->flat_dirty && !s->pending.empty()) {
        std::sort(s->pending.begin(), s->pending.end());
        s->pending.erase(std::unique(s->pending.begin(), s->pending.end()), s->pending.end());
        bool dist = false;
        std::vector<std::pair<uint32_t, uint32_t> > dirty;
        if (update_flat(s->flat, s->scene, s->pending, &dirty, &dist)) {
            s->patch.insert(s->patch.end(), dirty.begin(), dirty.end());
            s->patch_dist |= dist;
            ++s->flat_version;
            if (s->patch.size() > 4096) {  // so many small ranges that a full upload is cheaper: older copies take that path
                s->patch.clear();
                s->patch_base = s->flat_version;
            }
        } else {
            s->flat_dirty = true;
        }
    }
    s->pending.clear();
    if (s->flat_dirty) {
        s->flat = flatten(s->scene, s->accel);
        s->flat_dirty = false;
        ++s->flat_version;
        s->patch.clear();
        s->patch_dist = false;
        s->patch_base = s->flat_version;
    }
}

// Brings the scene's copy on the CURRENT device (cudaSetDevice done by the caller) up to date; *out = that copy.
int refresh_scene(bt_scene* s, int device, cudaStream_t stream, SceneDev** out) {
    commit_scene(s);
    SceneDev* d = 0;
    for (SceneDev& c : s->devs)
        if (c.device == device) d = &c;
    if (!d) {
        SceneDev c;
        std::memset(&c, 0, sizeof c);
        c.device = device;
        s->devs.push_back(c);
        d = &s->devs.back();
    }
    if (d->version != s->flat_version && d->version >= s->patch_base && d->version != 0) {
        // only in-place edits since this copy was made: upload the rewritten ranges (a moved object's records, the refitted
        // BVH nodes) instead of the whole scene
        if (d->ev_use) CK(cudaEventSynchronize(d->ev_use));
        for (const std::pair<uint32_t, uint32_t>& r : s->patch)
            CK(cudaMemcpyAsync(d->d_blob + r.first, s->flat.blob.data() + r.first, (size_t)r.second * sizeof(float4), cudaMemcpyHostToDevice, stream));
        if (s->patch_dist) {
            int rc = upload_dist_grid(s, d, stream);
            if (rc != BT_OK) return rc;
        }
        CK(cudaStreamSynchronize(stream));
        d->version = s->flat_version;
    }
    if (d->version != s->flat_version) {
        // a render enqueued without synchronising (bt_render_async) may still be reading the old copy
        if (d->ev_use) CK(cudaEventSynchronize(d->ev_use));
        size_t bb = s->flat.blob.size() * sizeof(float4), gb = s->flat.grids.size() * sizeof(float);
        if (bb > d->blob_cap) {
            if (d->d_blob) cudaFree(d->d_blob);
            d->d_blob = 0;
            d->blob_cap = 0;
            CK(cudaMalloc((void**)&d->d_blob, bb));
            d->blob_cap = bb;
        }
        if (gb > d->grids_cap) {
            if (d->d_grids) cudaFree(d->d_grids);
            d->d_grids = 0;
            d->grids_cap = 0;
            CK(cudaMalloc((void**)&d->d_grids, gb));
            d->grids_cap = gb;
        }
        CK(cudaMemcpyAsync(d->d_blob, s->flat.blob.data(), bb, cudaMemcpyHostToDevice, stream));
        CK(cudaMemcpyAsync(d->d_grids, s->flat.grids.data(), gb, cudaMemcpyHostToDevice, stream));
        {
            int rc = upload_dist_grid(s, d, stream);
            if (rc != BT_OK) return rc;
        }
        CK(cudaStreamSynchronize(stream));  // the host vectors may change after we return
        d->version = s->flat_version;
    }
    if (d->env_version != s->env_version) {
        // the environment map on its own (the flattened scene does not depend on it); a render enqueued without
        // synchronising may still be reading the old texels
        if (d->ev_use) CK(cudaEventSynchronize(d->ev_use));
        const size_t eb = s->env.size() * sizeof(float4);
        if (eb > d->env_cap) {
            if (d->d_env) cudaFree(d->d_env);
            d->d_env = 0;
            d->env_cap = 0;
            CK(cudaMalloc((void**)&d->d_env, eb));
            d->env_cap = eb;
        }
        if (eb) {
            CK(cudaMemcpyAsync(d->d_env, s->env.data(), eb, cudaMemcpyHostToDevice, stream));
            CK(cudaStreamSynchronize(stream));
        }
        d->env_version = s->env_version;
    }
    *out = d;
    return BT_OK;
}

// ChunkConfig::with_configs, reference src/tracer/mod.rs:218-229
struct Merged {
    int32_t output;
    uint32_t subsample;
    uint64_t samples, max_bounces, max_volume_bounces;
    float clip_min, clip_max, volume_step;
};
Merged merge(const bt_config& c, const bt_render_config& r) {
    Merged m;
    m.output = r.has_output ? r.output : c.output;
    m.subsample = r.subsample;
    m.samples = r.samples;
    m.max_bounces = r.has_max_bounces ? r.max_bounces : c.max_bounces;
    // mod.rs:224: max_volume_bounces takes render.max_BOUNCES (reference quirk, preserved)
    m.max_volume_bounces = r.has_max_bounces ? r.max_bounces : c.max_volume_bounces;
    m.clip_min = c.clip_min;
    m.clip_max = c.clip_max;
    m.volume_step = r.has_volume_step ? r.volume_step : c.volume_step;
    return m;
}

uint32_t clamp_u32(uint64_t v) { return v > 0xfffffffeULL ? 0xfffffffeu : (uint32_t)v; }

uint32_t knob(int64_t v, uint32_t dflt) { return v < 0 ? dflt : (uint32_t)v; }

int build_params(const bt_engine* en, bt_scene* s, const SceneDev* dev, uint64_t camera_ref, bool need_camera, const bt_config* config,
                 const bt_render_config* rc, uint64_t seed, uint64_t sample_base, uint32_t width, uint32_t height, RenderParams* out) {
    const Tuning& tn = en->tune;
    Merged m = merge(*config, *rc);
    RenderParams p;
    std::memset(&p, 0, sizeof p);
    p.scene = s->flat.header;
    uint32_t sub_n = m.subsample == 0 ? 1u : m.subsample;
    if ((uint64_t)sub_n * sub_n > 0xffffffffULL) return fail(BT_ERR_INVALID_ARG, "subsample too large");
    p.sub_count = sub_n * sub_n;
    if (need_camera) p.cam = make_camera_block(s->scene, camera_ref, width, height, m.subsample);
    p.cam.sub_n = sub_n;
    p.blob = dev->d_blob;
    p.grids = dev->d_grids;
    p.dist = dev->d_dist;
    p.env = dev->d_env;
    p.env_w = s->env.empty() ? 0u : s->env_w;
    p.env_h = s->env_h;
    p.width = width;
    p.height = height;
    if (m.samples * p.sub_count > 0xffffffffULL) return fail(BT_ERR_INVALID_ARG, "samples * subpixel_count exceeds 2^32 per call");
    p.paths_per_pixel = (uint32_t)(m.samples * p.sub_count);
    p.seed = seed;
    p.path_base = sample_base * p.sub_count;
    p.row0 = 0;
    p.row_end = height;
    {   // UniformInt<usize>::new(0, n).sample: zone = MAX - (MAX - n + 1) % n, hoisted out of the kernel
        const uint64_t range = p.scene.n_lights;
        p.light_zone = range ? 0xffffffffffffffffULL - (0xffffffffffffffffULL - range + 1) % range : 0;
    }
    p.output = m.output;
    p.max_bounces = clamp_u32(m.max_bounces);
    p.max_volume_bounces = clamp_u32(m.max_volume_bounces);
    p.clip_min = m.clip_min;
    p.clip_max = m.clip_max;
    p.volume_step = m.volume_step;
    // Scheduling thresholds of the per-warp phase machine (kernels.cu), tuned per kernel family on the
    // shipped scenes (profiles/r1_sweep_*.log).  Long flights through a surface-only scene end a path
    // every ~50 turns per lane: small batches keep lanes flying; a marching volume wants larger ones.
    const bool long_flights = p.scene.n_lens != 0 && !p.scene.has_volume_prims;
    p.compact_lanes = knob(tn.compact_lanes, long_flights ? 12 : 16);
    const bool bvh_rays = p.scene.n_bvh != 0 && p.scene.n_lens == 0;  // (patience counts node / leaf units there; profiles/r2_sweep_bvh.md)
    p.compact_patience = knob(tn.compact_patience, long_flights ? 8 : (bvh_rays ? 32 : 16));
    // A scan over a handful of surface primitives costs less than half a ray generation: such a warp
    // is better off collecting more idle lanes first (scene.json.gz: +4.6 %, profiles/r1_sweep_regen2.log).
    const bool cheap_scans = p.scene.n_lens == 0 && !p.scene.has_volume_prims && p.scene.n_bvh == 0 && p.scene.n_prims <= 8;
    p.regen_lanes = knob(tn.regen_lanes, long_flights || bvh_rays ? 4 : (cheap_scans ? 24 : 12));
    p.regen_patience = knob(tn.regen_patience, long_flights ? 8 : (cheap_scans ? 32 : 16));
    p.scan_lanes = knob(tn.scan_lanes, 8);      // (profiles/r1_sweep_nearest_sphere_bound.log: flat within 1 % from 6/2 to 8/4)
    p.scan_patience = knob(tn.scan_patience, 3);
    // The exact arithmetic flavour means EVERY operation of the path is the oracle's, the stepper's 1 / |d| included: a scene that
    // AUTO renders exactly (volumetric spheres: a 1e-5 position error flips scatter decisions of the 33-step march at a visible
    // rate -- cloud + lens at 64 spp: MAE 1.2e-3 .. 2.3e-3 with MUFU.RSQ, ~1e-7 with the rounded rsqrt) gets the exact stepper too.
    if (use_exact(en, s) && p.scene.n_lens != 0) p.scene.lens_exact = 1;
    if (tn.lens_no_skip > 0) p.scene.lens_skip = 0;
    if (tn.lens_dist_grid == 0 && p.scene.lens_skip == 3) p.scene.lens_skip = 1;  // (A/B: the per-flight bookkeeping)
    p.steps_per_turn = std::max(1u, knob(tn.steps_per_turn, long_flights || bvh_rays ? 3 : 2));  // (pooled traversal: node visits in a row)
    // the pooled kernel (render_pool.cuh): 32 W path slots per warp; 0 = one path per lane (render_body)
    // default: on for lens fields (long flights: C3 +22 %, cornell2 + lens +60 %, cloud + lens +16 % over the lane kernel), off for
    // flat ones, whose scan -> shade ping-pong gains nothing from compaction and pays for the state traffic (C2 -12 %)
    // -- except BVH scenes, whose traversal runs as pooled NODE / LEAF phases (32 k primitives: 238 against 221 Msamples/s; W = 3 of {1, 2, 3, 4})
    p.pool_w = std::min(knob(tn.pool_w, p.scene.n_lens != 0 ? 4 : (bvh_rays ? 3 : 0)), 8u);
    p.pool_refill = std::max(1u, knob(tn.pool_refill, 3));   // (profiles/r2_sweep_pool_C3.log: 3 / 32 best of {3, 6, 9} x {24, 28, 32})
    p.pool_step_min = knob(tn.pool_step_min, 32);
    p.pool_threads = knob(tn.pool_threads, 0) & ~31u;  // 0: the kernel's own CTA size (launch_pool)
    p.bvh_stack_k = std::max(1u, knob(tn.bvh_stack_k, 0xffffu));  // (tests: force the traversal stack's tail)
    p.tau_scale = uniform_scale_inclusive(0.0f, 6.28318530717958647692f);
    p.one_scale = uniform_scale_inclusive(0.0f, 1.0f);
    *out = p;
    return BT_OK;
}

// a scene created without an engine binds to the first engine that uses it
int bind_scene(bt_engine* engine, bt_scene* scene) {
    if (!scene->engine) scene->engine = engine;
    if (scene->engine != engine) return fail(BT_ERR_INVALID_ARG, "scene belongs to another engine");
    return BT_OK;
}
// every kernel that reads the scene's device copy is followed by this (refresh_scene / bt_scene_destroy wait for it)
int mark_scene_use(SceneDev* d, cudaStream_t stream) {
    if (!d->ev_use) CK(cudaEventCreateWithFlags(&d->ev_use, cudaEventDisableTiming));
    CK(cudaEventRecord(d->ev_use, stream));
    return BT_OK;
}

int check_renderable(const bt_scene* s) {
    if (s->flat.diffuse_without_light)
        return fail(BT_ERR_SCENE, "Uniform::new called with `low >= high` (a Diffuse surface needs at least one LIGHT object)");
    if (s->flat.cuboid_light_without_area)
        return fail(BT_ERR_SCENE, "called `Result::unwrap()` on an `Err` value: AllWeightsZero (a LIGHT Cuboid without face area)");
    if (render_smem_bytes(RenderParams{s->flat.header}) > 200 * 1024)
        return fail(BT_ERR_UNSUPPORTED, "scene does not fit the shared-memory staging buffer (use BT_ACCEL_BVH / BT_ACCEL_AUTO)");
    return BT_OK;
}

}  // namespace

#define GUARD_BEGIN try {
#define GUARD_END                                                  \
    }                                                              \
    catch (const ParseError& e) { return fail(BT_ERR_PARSE, e.what()); }  \
    catch (const SceneError& e) { return fail(BT_ERR_SCENE, e.what()); }  \
    catch (const std::exception& e) { return fail(BT_ERR_INVALID_ARG, e.what()); }

extern "C" {

const char* bt_last_error(void) { return g_error.c_str(); }

int bt_engine_create(int device, bt_engine** out) {
    if (!out) return fail(BT_ERR_INVALID_ARG, "out is NULL");
    int count = 0;
    cudaError_t e = cudaGetDeviceCount(&count);
    if (e != cudaSuccess || count == 0)
        return fail(BT_ERR_CUDA, std::string("no CUDA device available (the engine has no CPU fallback): ") + cudaGetErrorString(e));
    if (device < 0 || device >= count) return fail(BT_ERR_INVALID_ARG, "device index out of range");
    CK(cudaSetDevice(device));
    cudaDeviceProp prop;
    CK(cudaGetDeviceProperties(&prop, device));
    if (prop.major < 10) return fail(BT_ERR_CUDA, std::string("device is not sm_100 class: ") + prop.name);
    bt_engine* en = new bt_engine();
    en->device = device;
    for (const TuningName& t : kTuning) {  // BT_COMPACT_LANES, BT_POOL_W, ...: read once, here
        std::string env = "BT_";
        for (const char* c = t.name; *c; ++c) env += (char)std::toupper((unsigned char)*c);
        if (const char* v = std::getenv(env.c_str())) en->tune.*(t.field) = std::atoll(v);
    }
    en->launches = 0;
    en->d_scratch = 0;
    en->scratch_bytes = 0;
    en->d_lens = 0;
    en->lens_cap = 0;
    en->ev_lens = 0;
    en->d_pool_q[0] = en->d_pool_q[1] = 0;
    en->pool_q_cap[0] = en->pool_q_cap[1] = 0;
    en->ev_slice = en->ev_reduced = 0;
    en->d_stage = 0;
    en->stage_cap = 0;
    en->sm_count = prop.multiProcessorCount;
    int khz = 0;
    cudaDeviceGetAttribute(&khz, cudaDevAttrClockRate, device);
    en->clock_khz = khz;
    en->stream = en->stream2 = 0;
    en->ev_fork = en->ev_join = 0;
    e = cudaStreamCreateWithFlags(&en->stream, cudaStreamNonBlocking);
    if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&en->stream2, cudaStreamNonBlocking);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&en->ev_fork, cudaEventDisableTiming);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&en->ev_join, cudaEventDisableTiming);
    if (e != cudaSuccess) {
        bt_engine_destroy(en);
        return cuda_fail(e, "cudaStreamCreate");
    }
    *out = en;
    return BT_OK;
}

void bt_engine_destroy(bt_engine* engine) {
    if (!engine) return;
    for (bt_engine* peer : engine->peers) bt_engine_destroy(peer);
    cudaSetDevice(engine->device);
    if (engine->ev_slice) cudaEventDestroy(engine->ev_slice);
    if (engine->ev_reduced) cudaEventDestroy(engine->ev_reduced);
    if (engine->d_stage) cudaFree(engine->d_stage);
    if (engine->d_scratch) cudaFree(engine->d_scratch);
    if (engine->d_lens) cudaFree(engine->d_lens);
    for (int i = 0; i < 2; ++i)
        if (engine->d_pool_q[i]) cudaFree(engine->d_pool_q[i]);
    if (engine->ev_lens) cudaEventDestroy(engine->ev_lens);
    if (engine->ev_fork) cudaEventDestroy(engine->ev_fork);
    if (engine->ev_join) cudaEventDestroy(engine->ev_join);
    if (engine->stream2) cudaStreamDestroy(engine->stream2);
    if (engine->stream) cudaStreamDestroy(engine->stream);
    delete engine;
}

uint64_t bt_engine_launch_count(const bt_engine* engine) {
    if (!engine) return 0;
    uint64_t n = engine->launches;
    for (const bt_engine* peer : engine->peers) n += peer->launches;
    return n;
}

int bt_engine_create_multi(const int* devices, int n_devices, bt_engine** out) {
    if (!devices || !out || n_devices < 1) return fail(BT_ERR_INVALID_ARG, "need at least one device");
    if (n_devices > MAX_PEER_FRAMES + 1) return fail(BT_ERR_INVALID_ARG, "too many devices");
    bt_engine* head = 0;
    int r = bt_engine_create(devices[0], &head);
    if (r != BT_OK) return r;
    for (int i = 1; i < n_devices; ++i) {
        bt_engine* peer = 0;
        if ((r = bt_engine_create(devices[i], &peer)) != BT_OK) {
            bt_engine_destroy(head);
            return r;
        }
        head->peers.push_back(peer);
        cudaError_t e = cudaEventCreateWithFlags(&peer->ev_slice, cudaEventDisableTiming);
        int can = devices[i] == devices[0];
        if (e == cudaSuccess && !can) {
            // read the peer's slice in place over NVLink where the topology allows it
            if (cudaDeviceCanAccessPeer(&can, devices[0], devices[i]) != cudaSuccess) can = 0;
            if (can) {
                cudaSetDevice(devices[0]);
                cudaError_t pe = cudaDeviceEnablePeerAccess(devices[i], 0);
                if (pe == cudaErrorPeerAccessAlreadyEnabled) (void)cudaGetLastError();
                else if (pe != cudaSuccess) {
                    (void)cudaGetLastError();
                    can = 0;
                }
            }
        }
        head->peer_direct.push_back((char)can);
        if (e != cudaSuccess) {
            bt_engine_destroy(head);
            return cuda_fail(e, "cudaEventCreate");
        }
    }
    cudaSetDevice(devices[0]);
    if (!head->peers.empty()) {
        cudaError_t e = cudaEventCreateWithFlags(&head->ev_reduced, cudaEventDisableTiming);
        if (e != cudaSuccess) {
            bt_engine_destroy(head);
            return cuda_fail(e, "cudaEventCreate");
        }
    }
    *out = head;
    return BT_OK;
}

int bt_engine_device_count(const bt_engine* engine) { return engine ? 1 + (int)engine->peers.size() : 0; }

int bt_engine_set_tuning(bt_engine* engine, const char* name, int64_t value) {
    if (!engine || !name) return fail(BT_ERR_INVALID_ARG, "NULL argument");
    for (const TuningName& t : kTuning)
        if (!std::strcmp(t.name, name)) {
            engine->tune.*(t.field) = value;
            for (bt_engine* peer : engine->peers) peer->tune.*(t.field) = value;
            return BT_OK;
        }
    return fail(BT_ERR_INVALID_ARG, std::string("unknown tuning knob `") + name + "`");
}

int bt_scene_create_json(bt_engine* engine, const void* bytes, size_t n, bt_scene** out) {
    if (!bytes || !out) return fail(BT_ERR_INVALID_ARG, "NULL argument");
    GUARD_BEGIN
    bt_scene* s = new bt_scene();
    s->engine = engine;
    s->flat_version = 1;
    s->patch_base = 1;
    s->patch_dist = false;
    try {
        s->accel = ACCEL_AUTO;
        s->precision = BT_PRECISION_AUTO;
        if (const char* e = std::getenv("BT_PRECISION"))
            s->precision = !std::strcmp(e, "fast") ? BT_PRECISION_FAST : (!std::strcmp(e, "exact") ? BT_PRECISION_EXACT : BT_PRECISION_AUTO);
        s->scene = Scene::from_json(bytes, n);
        s->flat = flatten(s->scene, s->accel);
    } catch (...) {
        delete s;
        throw;
    }
    s->flat_dirty = false;
    *out = s;
    return BT_OK;
    GUARD_END
}

int bt_scene_to_json(const bt_scene* scene, char** out, size_t* n) {
    if (!scene || !out || !n) return fail(BT_ERR_INVALID_ARG, "NULL argument");
    GUARD_BEGIN
    std::string s = scene->scene.to_json();
    char* buf = (char*)std::malloc(s.size() + 1);
    if (!buf) return fail(BT_ERR_INVALID_ARG, "out of memory");
    std::memcpy(buf, s.data(), s.size());
    buf[s.size()] = 0;
    *out = buf;
    *n = s.size();
    return BT_OK;
    GUARD_END
}

void bt_free(void* p) { std::free(p); }

void bt_scene_destroy(bt_scene* scene) {
    if (!scene) return;
    for (SceneDev& d : scene->devs) {
        cudaSetDevice(d.device);
        if (d.ev_use) {
            cudaEventSynchronize(d.ev_use);
            cudaEventDestroy(d.ev_use);
        }
        if (d.d_blob) cudaFree(d.d_blob);
        if (d.d_grids) cudaFree(d.d_grids);
        if (d.d_dist) cudaFree(d.d_dist);
        if (d.d_env) cudaFree(d.d_env);
    }
    delete scene;
}

int bt_scene_find_by_tag(const bt_scene* scene, const char* tag, uint64_t* object_ref) {
    if (!scene || !tag || !object_ref) return fail(BT_ERR_INVALID_ARG, "NULL argument");
    if (!scene->scene.find_by_tag(tag, object_ref)) return fail(BT_ERR_SCENE, std::string("no object tagged `") + tag + "`");
    return BT_OK;
}

int bt_scene_set_camera_aspect(bt_scene* scene, uint64_t camera_ref, float aspect_ratio) {
    if (!scene) return fail(BT_ERR_INVALID_ARG, "NULL argument");
    GUARD_BEGIN
    Object& o = scene->scene.get_object(camera_ref);
    if (o.kind != OBJ_CAMERA) return fail(BT_ERR_SCENE, "called `Option::unwrap()` on a `None` value (object is not a camera)");
    o.camera.aspect_ratio = aspect_ratio;  // read per call by make_camera_block; no re-flatten needed
    return BT_OK;
    GUARD_END
}

int bt_scene_set_camera_projection(bt_scene* scene, uint64_t camera_ref, int projection) {
    if (!scene) return fail(BT_ERR_INVALID_ARG, "NULL argument");
    GUARD_BEGIN
    Object& o = scene->scene.get_object(camera_ref);
    if (o.kind != OBJ_CAMERA) return fail(BT_ERR_SCENE, "called `Option::unwrap()` on a `None` value (object is not a camera)");
    if (projection != BT_PROJECTION_PERSPECTIVE && projection != BT_PROJECTION_EQUIRECTANGULAR)
        return fail(BT_ERR_INVALID_ARG, "projection must be BT_PROJECTION_PERSPECTIVE or BT_PROJECTION_EQUIRECTANGULAR");
    o.camera.projection = projection == BT_PROJECTION_EQUIRECTANGULAR ? PROJ_EQUIRECTANGULAR : PROJ_PERSPECTIVE;  // read per call, like the aspect
    return BT_OK;
    GUARD_END
}

int bt_scene_apply_transform(bt_scene* scene, uint64_t object_ref, const float affine[12]) {
    if (!scene || !affine) return fail(BT_ERR_INVALID_ARG, "NULL argument");
    GUARD_BEGIN
    Affine a;
    std::memcpy(a.f, affine, sizeof a.f);
    scene->scene.apply_transform(object_ref, a);
    // the edited object and every descendant get a new world transform (object/mod.rs:212-223)
    std::vector<uint64_t> todo(1, object_ref);
    while (!todo.empty()) {
        const uint64_t r = todo.back();
        todo.pop_back();
        scene->pending.push_back(r);
        const Object& o = scene->scene.get_object(r);
        todo.insert(todo.end(), o.children.begin(), o.children.end());
    }
    return BT_OK;
    GUARD_END
}

int bt_scene_commit(bt_scene* scene) {
    if (!scene) return fail(BT_ERR_INVALID_ARG, "NULL argument");
    GUARD_BEGIN
    commit_scene(scene);
    return BT_OK;
    GUARD_END
}

void bt_lens_config_default(bt_lens_config* cfg) {
    if (!cfg) return;
    cfg->kappa = 0.05f;
    cfg->h_min = 0.02f;
    cfg->h_max = 5.0f;
    cfg->r_far = 500.0f;
    cfg->max_steps = 4096;
    cfg->flags = 0;
}

int bt_scene_set_lenses(bt_scene* scene, const float* xyzr, uint32_t n, const bt_lens_config* cfg) {
    if (!scene || (n && !xyzr)) return fail(BT_ERR_INVALID_ARG, "NULL argument");
    bt_lens_config c;
    if (cfg) c = *cfg; else bt_lens_config_default(&c);
    if (!(c.kappa > 0.0f) || !(c.h_min > 0.0f) || !(c.h_max >= c.h_min) || c.max_steps == 0)
        return fail(BT_ERR_INVALID_ARG, "lens config: need kappa > 0, 0 < h_min <= h_max, max_steps > 0");
    scene->scene.lenses.clear();
    for (uint32_t i = 0; i < n; ++i) {
        Lens l = {{xyzr[4 * i], xyzr[4 * i + 1], xyzr[4 * i + 2]}, xyzr[4 * i + 3]};
        scene->scene.lenses.push_back(l);
    }
    scene->scene.lens_config.kappa = c.kappa;
    scene->scene.lens_config.h_min = c.h_min;
    scene->scene.lens_config.h_max = c.h_max;
    scene->scene.lens_config.r_far = c.r_far;
    scene->scene.lens_config.max_steps = c.max_steps;
    scene->scene.lens_config.flags = c.flags;
    scene->flat_dirty = true;
    return BT_OK;
}

int bt_scene_set_environment(bt_scene* scene, const float* rgb, uint32_t width, uint32_t height) {
    if (!scene) return fail(BT_ERR_INVALID_ARG, "NULL argument");
    if (!rgb) {
        if (width != 0 || height != 0) return fail(BT_ERR_INVALID_ARG, "environment map: NULL texels need width = height = 0 (clear)");
        std::vector<float4>().swap(scene->env);
        scene->env_w = scene->env_h = 0;
        ++scene->env_version;
        return BT_OK;
    }
    if (width == 0 || height == 0) return fail(BT_ERR_INVALID_ARG, "environment map: width and height must be positive");
    if ((uint64_t)width * height >= (1ull << 31)) return fail(BT_ERR_INVALID_ARG, "environment map: width * height must be below 2^31");
    const size_t n = (size_t)width * height;
    for (size_t i = 0; i < 3 * n; ++i)
        if (!(rgb[i] >= 0.0f && rgb[i] <= 3.402823466e38f))
            return fail(BT_ERR_INVALID_ARG, "environment map: texel " + std::to_string(i / 3) + " is negative or not finite");
    GUARD_BEGIN
    std::vector<float4> texels(n);
    for (size_t i = 0; i < n; ++i) texels[i] = make_float4(rgb[3 * i], rgb[3 * i + 1], rgb[3 * i + 2], 0.0f);
    scene->env.swap(texels);
    scene->env_w = width;
    scene->env_h = height;
    ++scene->env_version;
    return BT_OK;
    GUARD_END
}

int bt_scene_set_accel(bt_scene* scene, int accel) {
    if (!scene) return fail(BT_ERR_INVALID_ARG, "NULL argument");
    if (accel < ACCEL_AUTO || accel > ACCEL_LINEAR_FACES) return fail(BT_ERR_INVALID_ARG, "accel must be BT_ACCEL_AUTO, _LINEAR, _BVH or _LINEAR_FACES");
    scene->accel = accel;
    scene->flat_dirty = true;
    return BT_OK;
}

int bt_scene_set_precision(bt_scene* scene, int precision) {
    if (!scene) return fail(BT_ERR_INVALID_ARG, "NULL argument");
    if (precision < BT_PRECISION_AUTO || precision > BT_PRECISION_EXACT)
        return fail(BT_ERR_INVALID_ARG, "precision must be BT_PRECISION_AUTO, _FAST or _EXACT");
    scene->precision = precision;
    return BT_OK;
}

int bt_scene_get_info(const bt_scene* scene, bt_scene_info* info) {
    if (!scene || !info) return fail(BT_ERR_INVALID_ARG, "NULL argument");
    GUARD_BEGIN
    FlatScene tmp;
    const FlatScene* f = &scene->flat;
    if (scene->flat_dirty) {
        tmp = flatten(scene->scene, scene->accel);
        f = &tmp;
    }
    info->n_objects = (uint32_t)scene->scene.objects.size();
    info->n_data = (uint32_t)scene->scene.data.size();
    info->n_primitives = f->header.n_prims;
    info->n_lights = f->header.n_lights;
    info->n_volumes = f->header.n_vols;
    info->n_lenses = f->header.n_lens;
    info->n_bvh_nodes = f->header.n_bvh;
    info->n_boxes = f->header.n_boxes;
    info->root_material = scene->scene.root_material;
    return BT_OK;
    GUARD_END
}

int bt_scene_copy_bvh(const bt_scene* scene, float* nodes, uint64_t nodes_cap, uint32_t* order, float* bounds, uint64_t prims_cap) {
    if (!scene) return fail(BT_ERR_INVALID_ARG, "NULL argument");
    GUARD_BEGIN
    FlatScene tmp;
    const FlatScene* f = &scene->flat;
    if (scene->flat_dirty) {
        tmp = flatten(scene->scene, scene->accel);
        f = &tmp;
    }
    const SceneHeader& h = f->header;
    if ((nodes && nodes_cap < h.n_bvh) || ((order || bounds) && prims_cap < h.n_prims)) return fail(BT_ERR_INVALID_ARG, "buffer too small");
    if (nodes && h.n_bvh) std::memcpy(nodes, &f->blob[h.bvh_off], (size_t)h.n_bvh * BVH_STRIDE * sizeof(float4));
    if (order)
        for (uint32_t i = 0; i < h.n_prims; ++i) order[i] = f->prim_order[i];
    if (bounds)
        for (uint32_t i = 0; i < h.n_prims; ++i)
            for (int k = 0; k < 3; ++k) {
                bounds[i * 6 + k] = f->prim_bounds[i].lo[k];
                bounds[i * 6 + 3 + k] = f->prim_bounds[i].hi[k];
            }
    return BT_OK;
    GUARD_END
}

void bt_config_default(bt_config* c) {
    if (!c) return;
    c->max_bounces = 8;
    c->max_volume_bounces = 32;
    c->clip_min = 0.01f;
    c->clip_max = 1000.0f;
    c->volume_step = 0.1f;
    c->chunks_x = 4;
    c->chunks_y = 2;
    c->output = BT_OUTPUT_FULL;
}

void bt_render_config_default(bt_render_config* c) {
    if (!c) return;
    std::memset(c, 0, sizeof *c);
    c->subsample = 0;
    c->samples = 64;
}

namespace {
// The body of Tracer::render for pixel rows [row0, row_end) of the frame at `fb` (device memory):
// checks, per-call constants, ONE kernel launch on `stream`.  bt_render_async renders the whole
// frame with it; bt_render pipelines a host frame through it in bands.
int ensure_pool_arena(bt_engine* e, int lane, RenderParams* p) {
    if (p->pool_w == 0) return BT_OK;
    const size_t bytes = render_pool_arena_bytes(p->pool_w, e->sm_count, p->scene.n_bvh != 0 && p->scene.n_lens == 0);
    if (bytes > e->pool_q_cap[lane]) {
        // (only ever grows; a kernel that may still read the old arena was launched on this lane's stream, and
        // cudaFree synchronises the device)
        if (e->d_pool_q[lane]) cudaFree(e->d_pool_q[lane]);
        e->d_pool_q[lane] = 0;
        e->pool_q_cap[lane] = 0;
        CK(cudaMalloc((void**)&e->d_pool_q[lane], bytes));
        e->pool_q_cap[lane] = bytes;
    }
    p->pool_counter = (unsigned long long*)e->d_pool_q[lane];
    p->pool_q = e->d_pool_q[lane] + 256;
    p->pool_q_cap = e->pool_q_cap[lane] - 256;
    return BT_OK;
}

int render_rows(bt_engine* engine, bt_scene* scene, uint64_t camera_ref, const bt_config* config, const bt_render_config* rc,
                uint64_t seed, uint64_t sample_base, float* fb, uint32_t width, uint32_t height, uint32_t row0, uint32_t row_end,
                cudaStream_t stream, int lane, uint32_t* sub_count_out) {
    SceneDev* sdev = 0;
    int rcode = refresh_scene(scene, engine->device, stream, &sdev);
    if (rcode != BT_OK) return rcode;
    if ((rcode = check_renderable(scene)) != BT_OK) return rcode;
    RenderParams p;
    if ((rcode = build_params(engine, scene, sdev, camera_ref, true, config, rc, seed, sample_base, width, height, &p)) != BT_OK) return rcode;
    p.fb = (float4*)fb;
    p.row0 = row0;
    p.row_end = row_end;
    if ((rcode = ensure_pool_arena(engine, lane, &p)) != BT_OK) return rcode;
    CK(use_exact(engine, scene) ? launch_render_exact(p, stream, &engine->launches) : launch_render_fast(p, stream, &engine->launches));
    if ((rcode = mark_scene_use(sdev, stream)) != BT_OK) return rcode;
    if (sub_count_out) *sub_count_out = p.sub_count;
    return BT_OK;
}
// Tracer::render on a multi-device engine.  The reference fans the tiles of one frame out over its thread pool INSIDE
// render (mod.rs:190-197); here the frame's passes [sample_base, sample_base + samples) are cut into one contiguous slice
// per device (SURVEY 8e: samples are i.i.d. and the buffer is a running sum).  Device 0 adds its slice straight into the
// caller's frame `fb` (device-0 memory) on `stream`; every other device renders its slice into a zeroed frame of its own on
// its own stream, and one kernel on device 0 then adds those frames to `fb`, reading them in place over NVLink
// (accumulate_frames_kernel).  One host thread drives all devices; the kernels of the different GPUs run concurrently.
int render_multi(bt_engine* engine, bt_scene* scene, uint64_t camera_ref, const bt_config* config, const bt_render_config* rc,
                 uint64_t seed, uint64_t sample_base, float* fb, uint32_t width, uint32_t height, cudaStream_t stream,
                 uint32_t* sub_count_out) {
    const uint64_t n = 1 + engine->peers.size(), total = rc->samples;
    const size_t bytes = (size_t)width * height * 4 * sizeof(float);
    bt_render_config part = *rc;
    PeerFrames direct;
    direct.n = 0;
    std::vector<size_t> staged;  // peers whose slice has to be copied to device 0 first
    int r = BT_OK;
    for (uint64_t g = 1; g < n && r == BT_OK; ++g) {
        const uint64_t lo = total * g / n, hi = total * (g + 1) / n;
        if (hi == lo) continue;
        bt_engine* peer = engine->peers[g - 1];
        CK(cudaSetDevice(peer->device));
        if ((r = ensure_scratch(peer, bytes)) != BT_OK) break;
        CK(cudaStreamWaitEvent(peer->stream, engine->ev_reduced, 0));  // the previous reduce is done with this frame
        CK(cudaMemsetAsync(peer->d_scratch, 0, bytes, peer->stream));
        part.samples = hi - lo;
        r = render_rows(peer, scene, camera_ref, config, &part, seed, sample_base + lo, (float*)peer->d_scratch, width, height, 0, height,
                        peer->stream, 0, nullptr);
        if (r != BT_OK) break;
        CK(cudaEventRecord(peer->ev_slice, peer->stream));
        if (engine->peer_direct[g - 1]) direct.src[direct.n++] = (const float4*)peer->d_scratch;
        else staged.push_back(g - 1);
    }
    CK(cudaSetDevice(engine->device));
    if (r != BT_OK) return r;
    part.samples = total / n;  // slice 0 = [0, total / n)
    if (part.samples) {
        if ((r = render_rows(engine, scene, camera_ref, config, &part, seed, sample_base, fb, width, height, 0, height, stream, 0,
                             sub_count_out)) != BT_OK)
            return r;
    } else if (sub_count_out) {
        *sub_count_out = rc->subsample == 0 ? 1u : rc->subsample * rc->subsample;
    }
    // ONE framebuffer reduce per call
    for (uint64_t g = 1; g < n; ++g)
        if (total * g / n != total * (g + 1) / n) CK(cudaStreamWaitEvent(stream, engine->peers[g - 1]->ev_slice, 0));
    CK(launch_accumulate_frames((float4*)fb, direct, width * height, engine->sm_count, stream, &engine->launches));
    for (size_t i : staged) {  // no peer mapping (not NVLink-connected): through a staging frame on device 0
        bt_engine* peer = engine->peers[i];
        if (bytes > engine->stage_cap) {
            if (engine->d_stage) cudaFree(engine->d_stage);
            engine->d_stage = 0;
            engine->stage_cap = 0;
            CK(cudaMalloc((void**)&engine->d_stage, bytes));
            engine->stage_cap = bytes;
        }
        CK(cudaMemcpyPeerAsync(engine->d_stage, engine->device, peer->d_scratch, peer->device, bytes, stream));
        PeerFrames one;
        one.n = 1;
        one.src[0] = engine->d_stage;
        CK(launch_accumulate_frames((float4*)fb, one, width * height, engine->sm_count, stream, &engine->launches));
    }
    CK(cudaEventRecord(engine->ev_reduced, stream));
    return BT_OK;
}
int check_render_args(bt_engine* engine, bt_scene* scene, const bt_config* config, const bt_render_config* rc, const float* fb,
                      uint32_t width, uint32_t height) {
    if (int b = bind_scene(engine, scene)) return b;
    if (!fb || width == 0 || height == 0) return fail(BT_ERR_INVALID_ARG, "empty buffer");
    if (config->output < 0 || config->output > 3 || (rc->has_output && (rc->output < 0 || rc->output > 3)))
        return fail(BT_ERR_INVALID_ARG, "invalid Output");
    return BT_OK;
}
}  // namespace

int bt_render_async(bt_engine* engine, bt_scene* scene, uint64_t camera_ref, const bt_config* config,
                    const bt_render_config* rc, uint64_t seed, uint64_t sample_base, float* rgba32f_device,
                    uint32_t width, uint32_t height, uint64_t* samples_inout, int32_t* status, void* cuda_stream) {
    if (!engine || !scene || !config || !rc || !status) return fail(BT_ERR_INVALID_ARG, "NULL argument");
    GUARD_BEGIN
    if (rc->samples == 0) {  // mod.rs:186-188
        *status = BT_STATUS_DONE;
        return BT_OK;
    }
    int rcode = check_render_args(engine, scene, config, rc, rgba32f_device, width, height);
    if (rcode != BT_OK) return rcode;
    CK(cudaSetDevice(engine->device));
    cudaStream_t stream = (cudaStream_t)cuda_stream;  // NULL is the CUDA default stream, taken literally
    uint32_t sub_count = 1;
    if (!engine->peers.empty())
        rcode = render_multi(engine, scene, camera_ref, config, rc, seed, sample_base, rgba32f_device, width, height, stream, &sub_count);
    else
        rcode = render_rows(engine, scene, camera_ref, config, rc, seed, sample_base, rgba32f_device, width, height, 0, height, stream, 0,
                            &sub_count);
    if (rcode != BT_OK) return rcode;
    if (samples_inout) *samples_inout += rc->samples * sub_count;  // mod.rs:199
    *status = BT_STATUS_IN_PROGRESS;
    return BT_OK;
    GUARD_END
}

int bt_render_stats(bt_engine* engine, bt_scene* scene, uint64_t camera_ref, const bt_config* config,
                    const bt_render_config* rc, uint64_t seed, uint64_t sample_base, uint32_t width, uint32_t height,
                    uint64_t stats_out[4]) {
    if (!engine || !scene || !config || !rc || !stats_out) return fail(BT_ERR_INVALID_ARG, "NULL argument");
    GUARD_BEGIN
    if (int b = bind_scene(engine, scene)) return b;
    for (int i = 0; i < 4; ++i) stats_out[i] = 0;
    if (rc->samples == 0) return BT_OK;
    CK(cudaSetDevice(engine->device));
    SceneDev* sdev = 0;
    int rcode = refresh_scene(scene, engine->device, engine->stream, &sdev);
    if (rcode != BT_OK) return rcode;
    if ((rcode = check_renderable(scene)) != BT_OK) return rcode;
    RenderParams p;
    if ((rcode = build_params(engine, scene, sdev, camera_ref, true, config, rc, seed, sample_base, width, height, &p)) != BT_OK) return rcode;
    size_t fb_bytes = (size_t)width * height * 16;
    if ((rcode = ensure_scratch(engine, fb_bytes + 64)) != BT_OK) return rcode;
    CK(cudaMemsetAsync(engine->d_scratch, 0, fb_bytes + 64, engine->stream));
    p.fb = (float4*)engine->d_scratch;
    p.stats = (unsigned long long*)((char*)engine->d_scratch + fb_bytes);
    CK(use_exact(engine, scene) ? launch_render_exact(p, engine->stream, &engine->launches) : launch_render_fast(p, engine->stream, &engine->launches));
    unsigned long long host[4];
    CK(cudaMemcpyAsync(host, p.stats, sizeof host, cudaMemcpyDeviceToHost, engine->stream));
    CK(cudaStreamSynchronize(engine->stream));
    for (int i = 0; i < 4; ++i) stats_out[i] = host[i];
    return BT_OK;
    GUARD_END
}

int bt_render_pool_stats(bt_engine* engine, bt_scene* scene, uint64_t camera_ref, const bt_config* config,
                         const bt_render_config* rc, uint64_t seed, uint64_t sample_base, uint32_t width, uint32_t height,
                         uint64_t stats_out[21]) {
    if (!engine || !scene || !config || !rc || !stats_out) return fail(BT_ERR_INVALID_ARG, "NULL argument");
    GUARD_BEGIN
    if (int b = bind_scene(engine, scene)) return b;
    for (int i = 0; i < 21; ++i) stats_out[i] = 0;
    if (rc->samples == 0) return BT_OK;
    CK(cudaSetDevice(engine->device));
    SceneDev* sdev = 0;
    int rcode = refresh_scene(scene, engine->device, engine->stream, &sdev);
    if (rcode != BT_OK) return rcode;
    if ((rcode = check_renderable(scene)) != BT_OK) return rcode;
    RenderParams p;
    if ((rcode = build_params(engine, scene, sdev, camera_ref, true, config, rc, seed, sample_base, width, height, &p)) != BT_OK) return rcode;
    if (p.pool_w == 0) return fail(BT_ERR_UNSUPPORTED, "the pooled kernel is switched off (tuning knob pool_w = 0)");
    size_t fb_bytes = (size_t)width * height * 16;
    if ((rcode = ensure_scratch(engine, fb_bytes + 256)) != BT_OK) return rcode;
    CK(cudaMemsetAsync(engine->d_scratch, 0, fb_bytes + 256, engine->stream));
    p.fb = (float4*)engine->d_scratch;
    p.stats = (unsigned long long*)((char*)engine->d_scratch + fb_bytes);
    p.pool_stats = 1;
    if ((rcode = ensure_pool_arena(engine, 0, &p)) != BT_OK) return rcode;
    cudaError_t ce = use_exact(engine, scene) ? launch_render_exact(p, engine->stream, &engine->launches) : launch_render_fast(p, engine->stream, &engine->launches);
    if (ce == cudaErrorNotSupported) return fail(BT_ERR_UNSUPPORTED, "scheduling counters exist for the content-specialised pooled kernels only");
    CK(ce);
    unsigned long long host[21];
    CK(cudaMemcpyAsync(host, p.stats, sizeof host, cudaMemcpyDeviceToHost, engine->stream));
    CK(cudaStreamSynchronize(engine->stream));
    for (int i = 0; i < 21; ++i) stats_out[i] = host[i];
    return BT_OK;
    GUARD_END
}

int bt_render(bt_engine* engine, bt_scene* scene, uint64_t camera_ref, const bt_config* config,
              const bt_render_config* rc, uint64_t seed, uint64_t sample_base, float* rgba32f, int mem,
              uint32_t width, uint32_t height, uint64_t* samples_inout, int32_t* status) {
    if (!engine || !rc || !status) return fail(BT_ERR_INVALID_ARG, "NULL argument");
    if (rc->samples == 0) {
        *status = BT_STATUS_DONE;
        return BT_OK;
    }
    if (!rgba32f) return fail(BT_ERR_INVALID_ARG, "empty buffer");
    CK(cudaSetDevice(engine->device));
    if (mem == BT_MEM_DEVICE) {
        int r = bt_render_async(engine, scene, camera_ref, config, rc, seed, sample_base, rgba32f, width, height,
                                samples_inout, status, engine->stream);
        if (r != BT_OK) return r;
        CK(cudaStreamSynchronize(engine->stream));
        return BT_OK;
    }
    // Host buffer: the frame goes through the GPU in horizontal bands, each band's upload, kernel and
    // download queued on one of two streams, so that band i+1's upload and band i-1's download run
    // under band i's kernel; only the first upload and the last download are exposed.  Pixels are
    // independent and the RNG is keyed by pixel, so the image does not depend on the banding
    // (BT_HOST_BANDS=1 renders the frame in one piece; tests compare the two bit for bit).
    if (!scene || !config) return fail(BT_ERR_INVALID_ARG, "NULL argument");
    GUARD_BEGIN
    int r = check_render_args(engine, scene, config, rc, rgba32f, width, height);
    if (r != BT_OK) return r;
    const size_t row_bytes = (size_t)width * 4 * sizeof(float), bytes = row_bytes * height;
    if ((r = ensure_scratch(engine, bytes)) != BT_OK) return r;
    if (!engine->peers.empty()) {
        // multi-device engine: the caller's running sums go to device 0, every device adds its pass slice (render_multi:
        // one reduce over NVLink), the summed frame comes back
        uint32_t sub = 1;
        CK(cudaMemcpyAsync(engine->d_scratch, rgba32f, bytes, cudaMemcpyHostToDevice, engine->stream));
        r = render_multi(engine, scene, camera_ref, config, rc, seed, sample_base, (float*)engine->d_scratch, width, height, engine->stream, &sub);
        if (r == BT_OK) CK(cudaMemcpyAsync(rgba32f, engine->d_scratch, bytes, cudaMemcpyDeviceToHost, engine->stream));
        CK(cudaStreamSynchronize(engine->stream));
        if (r != BT_OK) return r;
        if (samples_inout) *samples_inout += rc->samples * sub;  // mod.rs:199
        *status = BT_STATUS_IN_PROGRESS;
        return BT_OK;
    }
    uint32_t bands = (uint32_t)std::min<size_t>(8, std::max<size_t>(1, bytes / (8u << 20)));
    if (engine->tune.host_bands > 0) bands = (uint32_t)engine->tune.host_bands;
    uint32_t band_rows = ((height + bands - 1) / bands + 15u) & ~15u;  // whole 16-row CTAs
    // the scene's device copy is refreshed on the first stream; the second one waits for it
    SceneDev* sdev0 = 0;
    if ((r = refresh_scene(scene, engine->device, engine->stream, &sdev0)) != BT_OK) return r;
    CK(cudaEventRecord(engine->ev_fork, engine->stream));
    CK(cudaStreamWaitEvent(engine->stream2, engine->ev_fork, 0));
    uint32_t sub_count = 1;
    int band = 0;
    for (uint32_t row0 = 0; row0 < height; row0 += band_rows, ++band) {
        const uint32_t row_end = std::min(height, row0 + band_rows);
        cudaStream_t st = (band & 1) ? engine->stream2 : engine->stream;
        char* dev = (char*)engine->d_scratch + (size_t)row0 * row_bytes;
        char* host = (char*)rgba32f + (size_t)row0 * row_bytes;
        const size_t n = (size_t)(row_end - row0) * row_bytes;
        cudaError_t ce = cudaMemcpyAsync(dev, host, n, cudaMemcpyHostToDevice, st);
        if (ce == cudaSuccess) {
            r = render_rows(engine, scene, camera_ref, config, rc, seed, sample_base, (float*)engine->d_scratch, width, height, row0,
                            row_end, st, band & 1, &sub_count);
            if (r == BT_OK) ce = cudaMemcpyAsync(host, dev, n, cudaMemcpyDeviceToHost, st);
        }
        if (ce != cudaSuccess || r != BT_OK) {  // drain both lanes before reporting
            cudaStreamSynchronize(engine->stream);
            cudaStreamSynchronize(engine->stream2);
            return ce != cudaSuccess ? cuda_fail(ce, "bt_render: band copy") : r;
        }
    }
    CK(cudaEventRecord(engine->ev_join, engine->stream2));
    CK(cudaStreamWaitEvent(engine->stream, engine->ev_join, 0));
    CK(cudaStreamSynchronize(engine->stream));
    if (samples_inout) *samples_inout += rc->samples * sub_count;  // mod.rs:199
    *status = BT_STATUS_IN_PROGRESS;
    return BT_OK;
    GUARD_END
}

int bt_resolve_u8(bt_engine* engine, const float* rgba32f, int mem, uint32_t width, uint32_t height,
                  uint64_t samples, int color_space, uint8_t* rgba8) {
    if (!engine || !rgba32f || !rgba8) return fail(BT_ERR_INVALID_ARG, "NULL argument");
    if (color_space < 0 || color_space > 3) return fail(BT_ERR_INVALID_ARG, "invalid ColorSpace");
    CK(cudaSetDevice(engine->device));
    uint32_t n = width * height;
    if (mem == BT_MEM_DEVICE) {
        CK(launch_resolve((const float4*)rgba32f, n, samples, color_space, (uchar4*)rgba8, engine->stream, &engine->launches));
        CK(cudaStreamSynchronize(engine->stream));
        return BT_OK;
    }
    size_t fb_bytes = (size_t)n * 16, out_bytes = (size_t)n * 4;
    int r = ensure_scratch(engine, fb_bytes + out_bytes);
    if (r != BT_OK) return r;
    char* base = (char*)engine->d_scratch;
    CK(cudaMemcpyAsync(base, rgba32f, fb_bytes, cudaMemcpyHostToDevice, engine->stream));
    CK(launch_resolve((const float4*)base, n, samples, color_space, (uchar4*)(base + fb_bytes), engine->stream, &engine->launches));
    CK(cudaMemcpyAsync(rgba8, base + fb_bytes, out_bytes, cudaMemcpyDeviceToHost, engine->stream));
    CK(cudaStreamSynchronize(engine->stream));
    return BT_OK;
}

int bt_trace_segments(bt_engine* engine, bt_scene* scene, const bt_config* config, uint32_t n,
                      const float* origins, const float* dirs, bt_segment* out) {
    if (!engine || !scene || !config || (n && (!origins || !dirs || !out))) return fail(BT_ERR_INVALID_ARG, "NULL argument");
    GUARD_BEGIN
    if (int b = bind_scene(engine, scene)) return b;
    CK(cudaSetDevice(engine->device));
    SceneDev* sdev = 0;
    int r = refresh_scene(scene, engine->device, engine->stream, &sdev);
    if (r != BT_OK) return r;
    if ((r = check_renderable(scene)) != BT_OK && r != BT_ERR_SCENE) return r;
    bt_render_config rc;
    bt_render_config_default(&rc);
    rc.samples = 1;
    RenderParams p;
    if ((r = build_params(engine, scene, sdev, 0, false, config, &rc, 0, 0, 1, 1, &p)) != BT_OK) return r;
    size_t in_bytes = (size_t)n * 3 * sizeof(float), out_bytes = (size_t)n * sizeof(DeviceSegment);
    size_t off_d = (in_bytes + 255) & ~(size_t)255, off_o = 2 * off_d;
    if ((r = ensure_scratch(engine, off_o + out_bytes + 256)) != BT_OK) return r;
    char* base = (char*)engine->d_scratch;
    CK(cudaMemcpyAsync(base, origins, in_bytes, cudaMemcpyHostToDevice, engine->stream));
    CK(cudaMemcpyAsync(base + off_d, dirs, in_bytes, cudaMemcpyHostToDevice, engine->stream));
    CK((use_exact(engine, scene) ? launch_trace_exact : launch_trace_fast)(p, n, (const float*)base, (const float*)(base + off_d), (DeviceSegment*)(base + off_o), engine->stream, &engine->launches));
    std::vector<DeviceSegment> host(n);
    CK(cudaMemcpyAsync(host.data(), base + off_o, out_bytes, cudaMemcpyDeviceToHost, engine->stream));
    CK(cudaStreamSynchronize(engine->stream));
    for (uint32_t i = 0; i < n; ++i) {
        const DeviceSegment& d = host[i];
        bt_segment& o = out[i];
        o.face = d.face;
        o.steps = d.steps;
        o.object_ref = d.obj >= 0 ? scene->flat.object_refs[d.obj] : 0;
        o.t = d.t;
        std::memcpy(o.position, d.position, sizeof o.position);
        std::memcpy(o.normal, d.normal, sizeof o.normal);
        std::memcpy(o.direction, d.direction, sizeof o.direction);
    }
    return BT_OK;
    GUARD_END
}

int bt_camera_rays(bt_engine* engine, bt_scene* scene, uint64_t camera_ref, const bt_config* config,
                   const bt_render_config* rc, uint64_t seed, uint64_t sample_base, uint32_t width, uint32_t height,
                   uint32_t n, const uint32_t* xs, const uint32_t* ys, const uint64_t* path_index, float* out) {
    if (!engine || !scene || !config || !rc || (n && (!xs || !ys || !path_index || !out))) return fail(BT_ERR_INVALID_ARG, "NULL argument");
    GUARD_BEGIN
    if (int b = bind_scene(engine, scene)) return b;
    CK(cudaSetDevice(engine->device));
    SceneDev* sdev = 0;
    int r = refresh_scene(scene, engine->device, engine->stream, &sdev);
    if (r != BT_OK) return r;
    RenderParams p;
    if ((r = build_params(engine, scene, sdev, camera_ref, true, config, rc, seed, sample_base, width, height, &p)) != BT_OK) return r;
    size_t b32 = ((size_t)n * 4 + 255) & ~(size_t)255, b64 = ((size_t)n * 8 + 255) & ~(size_t)255, bo = (size_t)n * 24;
    if ((r = ensure_scratch(engine, 2 * b32 + b64 + bo + 256)) != BT_OK) return r;
    char* base = (char*)engine->d_scratch;
    CK(cudaMemcpyAsync(base, xs, (size_t)n * 4, cudaMemcpyHostToDevice, engine->stream));
    CK(cudaMemcpyAsync(base + b32, ys, (size_t)n * 4, cudaMemcpyHostToDevice, engine->stream));
    CK(cudaMemcpyAsync(base + 2 * b32, path_index, (size_t)n * 8, cudaMemcpyHostToDevice, engine->stream));
    CK((use_exact(engine, scene) ? launch_camera_rays_exact : launch_camera_rays_fast)(p, n, (const uint32_t*)base, (const uint32_t*)(base + b32), (const uint64_t*)(base + 2 * b32),
                          (float*)(base + 2 * b32 + b64), engine->stream, &engine->launches));
    CK(cudaMemcpyAsync(out, base + 2 * b32 + b64, bo, cudaMemcpyDeviceToHost, engine->stream));
    CK(cudaStreamSynchronize(engine->stream));
    return BT_OK;
    GUARD_END
}

int bt_geodesic_integrate(bt_engine* engine, const float* xyzr, uint32_t n_lenses, const bt_lens_config* cfg,
                          uint32_t n, float* xv, int mem, uint32_t n_steps, void* cuda_stream) {
    if (!engine || (n_lenses && !xyzr) || (n && !xv)) return fail(BT_ERR_INVALID_ARG, "NULL argument");
    bt_lens_config c;
    if (cfg) c = *cfg; else bt_lens_config_default(&c);
    CK(cudaSetDevice(engine->device));
    cudaStream_t stream = mem == BT_MEM_HOST ? engine->stream : (cudaStream_t)cuda_stream;
    std::vector<float4> lens;
    for (uint32_t i = 0; i < n_lenses; ++i) {
        float rs = xyzr[4 * i + 3];
        if (!(rs > 0.0f)) continue;
        float4 e0 = {xyzr[4 * i], xyzr[4 * i + 1], xyzr[4 * i + 2], -1.5f * rs};
        float4 e1 = {rs, c.r_far * rs, 0.0f, 0.0f};
        lens.push_back(e0);
        lens.push_back(e1);
    }
    IntegrateParams p;
    std::memset(&p, 0, sizeof p);
    p.n_lens = (uint32_t)(lens.size() / LENS_STRIDE);
    if (p.n_lens <= INTEGRATE_INLINE_LENSES) {
        std::copy(lens.begin(), lens.end(), p.inline_lens);  // by value: nothing to upload, nothing to race with
    } else {
        // a table of its own, never shared with the scratch of the other entry points; the previous launch that read
        // it (possibly still running on the caller's stream) must be over before it is overwritten
        const size_t bytes = lens.size() * sizeof(float4);
        if (engine->ev_lens) CK(cudaEventSynchronize(engine->ev_lens));
        if (bytes > engine->lens_cap) {
            if (engine->d_lens) cudaFree(engine->d_lens);
    for (int i = 0; i < 2; ++i)
        if (engine->d_pool_q[i]) cudaFree(engine->d_pool_q[i]);
            engine->d_lens = 0;
            engine->lens_cap = 0;
            CK(cudaMalloc((void**)&engine->d_lens, bytes));
            engine->lens_cap = bytes;
        }
        CK(cudaMemcpyAsync(engine->d_lens, lens.data(), bytes, cudaMemcpyHostToDevice, stream));
        CK(cudaStreamSynchronize(stream));  // the upload reads a stack vector
        p.lens = engine->d_lens;
    }
    p.kappa = c.kappa;
    p.h_min = c.h_min;
    p.h_max = c.h_max;
    p.n = n;
    p.n_steps = n_steps;
    p.exact = c.flags & BT_LENS_EXACT_RSQRT;
    if (mem == BT_MEM_HOST) {
        size_t xv_bytes = (size_t)n * 6 * sizeof(float);
        int r = ensure_scratch(engine, xv_bytes + 256);
        if (r != BT_OK) return r;
        float* d_xv = (float*)engine->d_scratch;
        CK(cudaMemcpyAsync(d_xv, xv, xv_bytes, cudaMemcpyHostToDevice, stream));
        p.xv = d_xv;
        CK(launch_integrate(p, stream, &engine->launches));
        CK(cudaMemcpyAsync(xv, d_xv, xv_bytes, cudaMemcpyDeviceToHost, stream));
        CK(cudaStreamSynchronize(stream));
    } else {
        p.xv = xv;
        CK(launch_integrate(p, stream, &engine->launches));
        if (p.lens) {
            if (!engine->ev_lens) CK(cudaEventCreateWithFlags(&engine->ev_lens, cudaEventDisableTiming));
            CK(cudaEventRecord(engine->ev_lens, stream));
        }
    }
    return BT_OK;
}

int bt_fp32_peak(bt_engine* engine, uint32_t iters, double* tflops) {
    if (!engine || !tflops || iters == 0) return fail(BT_ERR_INVALID_ARG, "NULL argument");
    CK(cudaSetDevice(engine->device));
    int blocks = engine->sm_count * 8;
    int r = ensure_scratch(engine, (size_t)blocks * FP32_PEAK_THREADS * sizeof(float));
    if (r != BT_OK) return r;
    cudaEvent_t e0, e1;
    CK(cudaEventCreate(&e0));
    CK(cudaEventCreate(&e1));
    CK(launch_fp32_peak((float*)engine->d_scratch, iters / 4 + 1, blocks, engine->stream, &engine->launches));  // warm-up
    CK(cudaEventRecord(e0, engine->stream));
    CK(launch_fp32_peak((float*)engine->d_scratch, iters, blocks, engine->stream, &engine->launches));
    CK(cudaEventRecord(e1, engine->stream));
    CK(cudaStreamSynchronize(engine->stream));
    float ms = 0.0f;
    CK(cudaEventElapsedTime(&ms, e0, e1));
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    double flops = 2.0 * (double)blocks * FP32_PEAK_THREADS * FP32_PEAK_CHAINS * FP32_PEAK_UNROLL * (double)iters;
    *tflops = flops / (ms * 1e-3) / 1e12;
    return BT_OK;
}

}  // extern "C"
