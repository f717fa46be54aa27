/*
 * bendy_b200.h -- C ABI of the B200-native render engine for bendy-tracer's per-sample loop.
 *
 * This is the drop-in boundary: the reference has no FFI, its operator boundary is the Rust
 * method  Tracer::render(&self, &Scene, ObjectRef, &RenderConfig, &mut Buffer) -> Status
 * (reference src/tracer/mod.rs:179-202) plus the public types it touches.  A `bendy-b200-sys`
 * crate (build.rs + nvcc, see INTEGRATION.md) binds exactly these entry points; the Python
 * package `bendy_tracer_b200` binds them with ctypes.
 *
 * Conventions: plain pointers and sizes, no C++/torch types.  Every function returns BT_OK or a
 * negative BT_ERR_* code and never aborts; the message is available from bt_last_error() on the
 * calling thread.  Conditions on which the reference panics (invalid refs, wrong data kind, a
 * Diffuse surface in a scene without LIGHT objects, negative volume density) are reported as
 * BT_ERR_SCENE with the reference's panic text.  Handles are owned by the caller.  One render
 * call per engine at a time (the reference's `&mut Buffer` exclusivity, src/tracer/mod.rs:184).
 *
 * There is no CPU fallback: every compute entry point fails with BT_ERR_CUDA when no sm_100
 * device is available.
 */
#ifndef BENDY_B200_H
#define BENDY_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

enum {
    BT_OK = 0,
    BT_ERR_INVALID_ARG = -1,
    BT_ERR_PARSE = -2,       /* scene JSON / gzip could not be decoded (serde_json error in the reference) */
    BT_ERR_SCENE = -3,       /* the reference would panic on this scene / ref */
    BT_ERR_CUDA = -4,
    BT_ERR_UNSUPPORTED = -5
};

/* Output, reference src/tracer/mod.rs:108-115 */
enum { BT_OUTPUT_FULL = 0, BT_OUTPUT_ALBEDO = 1, BT_OUTPUT_NORMAL = 2, BT_OUTPUT_DEPTH = 3 };
/* Status, reference src/tracer/mod.rs:159-163 */
enum { BT_STATUS_DONE = 0, BT_STATUS_IN_PROGRESS = 1 };
/* ColorSpace, reference src/tracer/buffer.rs:11-17 */
enum { BT_CS_NONE = 0, BT_CS_NORMAL = 1, BT_CS_LINEAR = 2, BT_CS_SRGB = 3 };
/* Face, reference src/tracer/ray.rs:8-15, plus the two non-hit outcomes of a traced segment */
enum { BT_FACE_FRONT = 0, BT_FACE_BACK = 1, BT_FACE_VOLUME = 2, BT_FACE_VOLUME_FRONT = 3,
       BT_FACE_VOLUME_BACK = 4, BT_FACE_MISS = -1, BT_FACE_CAPTURED = -2 };
/* where a caller-owned buffer lives */
enum { BT_MEM_HOST = 0, BT_MEM_DEVICE = 1 };

typedef struct bt_engine bt_engine;   /* one CUDA device + its stream and scratch */
typedef struct bt_scene bt_scene;     /* a parsed Scene + its flattened SoA device buffers */

/* Config, reference src/tracer/mod.rs:16-45 (defaults: 8, 32, 0.01, 1000, 0.1, 4, 2, Full) */
typedef struct {
    uint64_t max_bounces;
    uint64_t max_volume_bounces;
    float clip_min, clip_max, volume_step;
    uint32_t chunks_x, chunks_y;   /* scheduling hint only, as in the reference (never changes the image) */
    int32_t output;
} bt_config;

/* RenderConfig, reference src/tracer/mod.rs:117-135; Option<T> fields are has_/value pairs */
typedef struct {
    uint32_t subsample;            /* 0 = Subsample::None, n = Subsample::Subpixel(n) (mod.rs:47-68) */
    uint64_t samples;
    int32_t has_output, output;
    int32_t has_max_bounces;
    uint64_t max_bounces;
    int32_t has_max_volume_bounces;
    uint64_t max_volume_bounces;
    int32_t has_volume_step;
    float volume_step;
} bt_render_config;

/* Lens-field stepping parameters (extension; DESIGN.md "Geodesic model").  Defaults via
 * bt_lens_config_default(): kappa 0.05, h_min 0.02, h_max 5, r_far 500, max_steps 4096, flags 0.
 * BT_LENS_EXACT_RSQRT: the stepper's 1/|d| is correctly rounded (__frsqrt_rn) instead of
 * MUFU.RSQ (<= 2 ulp); every other operation is already IEEE, so the lensed path becomes
 * bit-identical to the CPU oracle.  Costs ~18 extra instructions per mass per evaluation. */
/* BT_LENS_NO_SKIP: intersect every chord with the scene, as the spec's loop is written.  By default
 * a chord is intersected only when it is at least as long as a conservative lower bound on the
 * distance from its start to the nearest primitive (refreshed by every intersection pass), which
 * cannot change a result -- the flag exists so that tests can prove that. */
enum { BT_LENS_EXACT_RSQRT = 1, BT_LENS_NO_SKIP = 2 };
typedef struct {
    float kappa, h_min, h_max, r_far;
    uint32_t max_steps;
    uint32_t flags;
} bt_lens_config;

/* One traced ray segment: Manifold (reference src/tracer/ray.rs:36-47) reduced to plain data. */
typedef struct {
    int32_t face;                  /* BT_FACE_* */
    uint32_t steps;                /* RK4 steps taken (0 in a flat field) */
    uint64_t object_ref;
    float t;                       /* distance (accumulated chord length under lensing) */
    float position[3];
    float normal[3];
    float direction[3];            /* direction of the last chord, or the escape direction */
} bt_segment;

typedef struct {
    uint32_t n_objects, n_data, n_primitives /* flattened: spheres + rects + 6 per cuboid */,
             n_lights, n_volumes, n_lenses, n_bvh_nodes,
             n_boxes /* cuboids recognised as one rectangular box: one slab test instead of six rect tests */;
    uint64_t root_material;
} bt_scene_info;

/* ---- engine ---------------------------------------------------------------------------- */
/* Replaces Tracer::new / with_config's implicit "use the rayon global pool" (mod.rs:170-177,194). */
int bt_engine_create(int device, bt_engine** out);
/* One engine over n CUDA devices of this box: the counterpart of the rayon fan-out INSIDE Tracer::render (reference
 * src/tracer/mod.rs:190-197), so that a caller of bt_render / bt_render_async uses 8 GPUs without changing a line.
 * Every render call cuts its passes [sample_base, sample_base + samples) into one contiguous slice per device (the RNG
 * is keyed by the global pass index: the union of the slices IS the one-device sample set); devices[0] owns the caller's
 * frame (BT_MEM_DEVICE buffers live there) and adds its slice into it, the others render into frames of their own, and
 * ONE kernel on devices[0] sums those in place over NVLink peer mappings (through a staging copy where the topology has
 * none).  The image equals the one-device image up to f32 summation order.  One host thread drives all devices.  A device
 * may be listed more than once (its kernels then share that GPU).  Probes, resolve and the stepper run on devices[0]. */
int bt_engine_create_multi(const int* devices, int n_devices, bt_engine** out);
int bt_engine_device_count(const bt_engine* engine);
void bt_engine_destroy(bt_engine* engine);
/* number of kernels this engine has launched since creation (bench.py's gpu_launches) */
uint64_t bt_engine_launch_count(const bt_engine* engine);
/* Scheduling knobs of the kernels -- the counterpart of Config::chunks_x / chunks_y (reference
 * src/tracer/mod.rs:22-23): they decide how the work is laid out on the device and never change an
 * image.  Each knob is read ONCE from the environment when the engine is created (BT_<NAME>,
 * upper case) and can be set per engine here; value < 0 restores the built-in default.
 *   pool_w          path slots per warp / 32 of the pooled render kernel; 0 = one path per lane
 *   pool_refill, pool_step_min, pool_threads     refill batch, step-phase exit level, CTA size of that kernel
 *   host_bands      row bands a BT_MEM_HOST frame is pipelined in (bt_render)
 *   compact_lanes, compact_patience, regen_lanes, regen_patience, scan_lanes, scan_patience,
 *   steps_per_turn                               thresholds of the one-path-per-lane kernel
 *   bvh_stack_k     BVH traversal: stack levels kept in shared memory (fewer = more of the stack in its slow tail; tests)
 *   lens_no_skip    1: as BT_LENS_NO_SKIP for every scene */
int bt_engine_set_tuning(bt_engine* engine, const char* name, int64_t value);

/* ---- scene ----------------------------------------------------------------------------- */
/* serde_json::from_reader(GzDecoder|BufReader) -> Scene, reference src/main.rs:93-102.
 * gzip is detected from the magic bytes.  The optional top-level "lenses" key
 * ([[x,y,z,r_s],...]) is an extension the reference's loader ignores.  `engine` may be NULL:
 * the scene is then host-only until its first render, which binds it to that engine. */
int bt_scene_create_json(bt_engine* engine, const void* bytes, size_t n, bt_scene** out);
/* serde_json::to_writer(&Scene), reference src/main.rs:299-313.  *out is malloc'd; free with bt_free. */
int bt_scene_to_json(const bt_scene* scene, char** out, size_t* n);
void bt_free(void* p);
void bt_scene_destroy(bt_scene* scene);
/* Scene::find_by_tag, reference src/scene/mod.rs:124-129.  BT_ERR_SCENE when no object has the tag. */
int bt_scene_find_by_tag(const bt_scene* scene, const char* tag, uint64_t* object_ref);
/* The one scene update main issues: camera.aspect_ratio = w/h through an UpdateQueue
 * (reference src/main.rs:218-223, 337-350). */
int bt_scene_set_camera_aspect(bt_scene* scene, uint64_t camera_ref, float aspect_ratio);
/* Camera projection (extension; DESIGN.md §3.6).  PERSPECTIVE (the default) is the reference's frustum.  EQUIRECTANGULAR
 * renders the whole sphere around the camera in the environment map's convention (bt_scene_set_environment), so a panorama
 * of an empty scene reproduces its map: with the jittered NDC u, v formed as for PERSPECTIVE (the same two draws and
 * sub-pixel offsets), u' = u + pixel_width / 2, v' = v + pixel_height / 2 (pixel_width = 2 / width, ...),
 * phi = PI_F * u', theta = -(PI_F / 2) * v', and the camera-space direction is
 * (cos theta * sin phi, sin theta, -(cos theta * cos phi)), each product and sum rounded on its own and sin / cos from the
 * engine's own polynomial in both arithmetic flavours (DESIGN.md §3.6 spells out the order): pixel (x, y) with zero
 * jitter looks at the centre of texel (x, y) of a width x height map, the centre column along camera -z, columns towards
 * camera +x, row 0 at the +y pole.  Directions past a pole (sub-pixel offsets on the last row) are used as computed.  The
 * direction then goes through the camera's world transform as for PERSPECTIVE and the origin is the camera's position.
 * An equirectangular camera is a pinhole: focus and fstop are ignored and no unit-disk numbers are drawn, so every path
 * draws exactly two numbers for its camera ray.  sensor_size, focal_length and aspect_ratio do not apply; any width x height
 * is allowed (width = 2 height gives square pixels).  Host-only: read per render call, never re-flattens or uploads, and
 * not part of the wire format (bt_scene_to_json is unchanged).  BT_ERR_SCENE for a reference that is not a camera,
 * BT_ERR_INVALID_ARG for an unknown projection (scene unchanged). */
enum { BT_PROJECTION_PERSPECTIVE = 0, BT_PROJECTION_EQUIRECTANGULAR = 1 };
int bt_scene_set_camera_projection(bt_scene* scene, uint64_t camera_ref, int projection);
/* Object::apply_transform on one object followed by UpdateQueue::commit (reference
 * src/scene/object/mod.rs:212-223, src/scene/mod.rs:204-213): local = local * affine, world and
 * the children's parent transforms are re-derived, device buffers are re-flattened lazily. */
int bt_scene_apply_transform(bt_scene* scene, uint64_t object_ref, const float affine[12]);
/* UpdateQueue::commit (reference src/scene/mod.rs:204-213): applies the edits queued since the last render to the flattened
 * scene on the host.  Transform edits are applied IN PLACE -- the records of the moved objects are rewritten, the BVH is refit
 * (same topology, new boxes), and the next render uploads only those ranges -- unless an edit changes the layout (then, as for
 * every other kind of edit, the scene is flattened from scratch).  Optional: the next render call commits what is pending. */
int bt_scene_commit(bt_scene* scene);
/* lens field: n point masses (x, y, z, r_s); cfg may be NULL for the defaults */
int bt_scene_set_lenses(bt_scene* scene, const float* xyzr, uint32_t n, const bt_lens_config* cfg);
void bt_lens_config_default(bt_lens_config* cfg);
/* Environment map (extension; DESIGN.md "Environment map"): an equirectangular RGB image the colour of every escaping
 * path is multiplied by, looked up in its escape direction d (the straight ray, the last chord / final velocity of a
 * bent flight, the march direction of a volume escape): colour = sample_root's colour * env(d).  Albedo, normal and
 * depth outputs, captured flights, paths and RNG draws are unchanged; with the root Emissive{white, k} the sky shows
 * k * map, with a Flat{black} root nothing.  rgb = width * height * 3 floats in host memory, row-major: row 0 is the +y
 * pole, row height-1 the -y pole, the centre column looks along -z (the default camera's view) and columns grow
 * towards +x.  Lookup: phi = atan2(d.x, -d.z), theta = atan2(d.y, sqrt(d.x^2 + d.z^2)), u = 0.5 + phi / 2pi,
 * v = 0.5 - theta / pi, texel coordinates (u W - 0.5, v H - 0.5), bilinear, columns wrap, rows clamp.  The texels are
 * copied (the caller may free rgb); rgb = NULL with width = height = 0 clears the map.  BT_ERR_INVALID_ARG (scene
 * unchanged) for zero or inconsistent sizes, width * height >= 2^31, negative or non-finite values.  Like the lens
 * field it is not part of the wire format (bt_scene_to_json is unchanged), and setting it never re-flattens the scene. */
int bt_scene_set_environment(bt_scene* scene, const float* rgb, uint32_t width, uint32_t height);
/* Closest-hit structure.  AUTO: the reference's linear scan (try_hit, src/tracer/mod.rs:389-402)
 * over shared memory up to 64 flattened primitives, a BVH (global-memory nodes, shared-memory
 * traversal stack) beyond.  Both give the same hits, exact-distance ties included.  Scenes with
 * volumetric spheres always use the scan (hit_volumetric depends on the scan order, :414-424). */
enum { BT_ACCEL_AUTO = 0, BT_ACCEL_LINEAR = 1, BT_ACCEL_BVH = 2,
       BT_ACCEL_LINEAR_FACES = 3 /* the scan with every Cuboid as its six Rect::hit tests (cuboid.rs:83-105, literally);
                                    the other modes test a box-shaped cuboid with one slab test and an
                                    axis-aligned Rect with a component-picking test that rounds identically) */ };
int bt_scene_set_accel(bt_scene* scene, int accel);
/* Arithmetic flavour of the render / trace / camera-ray kernels for this scene.  EXACT: every
 * division, square root and dot product is the IEEE operation sequence of the reference (values
 * bit-identical to the CPU oracle up to libm's sin/cos/pow).  FAST: MUFU reciprocal / square
 * roots and FMA-contracted rect tests, each within ~1 ulp (image MAE vs the oracle 1e-8 .. 1e-5 on
 * surface scenes).  AUTO (default): EXACT for scenes with volumetric spheres -- their steep density
 * gradients turn ulp-level differences into flipped scatter decisions -- FAST otherwise.  Under a lens
 * field EXACT implies BT_LENS_EXACT_RSQRT (the whole path is then bit-identical to the oracle).
 * Environment override for new scenes: BT_PRECISION=fast|exact|auto. */
enum { BT_PRECISION_AUTO = 0, BT_PRECISION_FAST = 1, BT_PRECISION_EXACT = 2 };
int bt_scene_set_precision(bt_scene* scene, int precision);
int bt_scene_get_info(const bt_scene* scene, bt_scene_info* info);
/* Introspection of the acceleration structure (tests, tools; an extension like the BVH itself): copies the 4-wide nodes
 * (32 floats per node: min.x[4] max.x[4] min.y[4] max.y[4] min.z[4] max.z[4], four child references as raw 32-bit
 * patterns, four unused -- child: inner node index, 0x80000000 | kind << 29 | count << 24 | first record (kind 1: all
 * spheres, 2: no sphere, 0: mixed; count <= 31), or 0xfffffffe = empty), the
 * record order (tree position -> canonical primitive index) and the primitives' bounds (6 floats each: min xyz, max
 * xyz, canonical order) as of the last flatten / commit.  Any pointer may be NULL; capacities in nodes / primitives;
 * BT_ERR_INVALID_ARG when one is too small (bt_scene_get_info gives the counts). */
int bt_scene_copy_bvh(const bt_scene* scene, float* nodes, uint64_t nodes_cap, uint32_t* order, float* bounds, uint64_t prims_cap);

/* ---- the hot path ---------------------------------------------------------------------- */
void bt_config_default(bt_config* cfg);                /* Config::DEFAULT, mod.rs:29-38 */
void bt_render_config_default(bt_render_config* cfg);  /* RenderConfig::DEFAULT, mod.rs:128-135 */

/* Tracer::render, reference src/tracer/mod.rs:179-202.
 *   samples == 0           -> *status = BT_STATUS_DONE, nothing touched.
 *   otherwise              -> adds samples * subpixel_count radiance samples per pixel into
 *                             rgba32f (row-major, y down, 4 f32 per pixel, alpha untouched:
 *                             buffer.rs:159-178), *samples_inout += samples * subpixel_count
 *                             (mod.rs:199), *status = BT_STATUS_IN_PROGRESS.
 * seed / sample_base key the per-path RNG stream (replaces SmallRng::from_entropy, mod.rs:240):
 * pass s of this call uses global pass index sample_base + s, so disjoint [sample_base,
 * sample_base + samples) ranges on different GPUs render disjoint sample sets of one image.
 * Blocking.  mem = BT_MEM_HOST copies the buffer to the device and back inside the call: the frame
 * is pipelined through the GPU in row bands over two streams (upload and download of a band run
 * under its neighbours' kernels; pin the buffer -- cudaHostAlloc / cudaHostRegister -- for the
 * overlap to be real).  The image does not depend on the banding (tuning knob host_bands). */
int bt_render(bt_engine* engine, bt_scene* scene, uint64_t camera_ref, const bt_config* config,
              const bt_render_config* render_config, uint64_t seed, uint64_t sample_base,
              float* rgba32f, int mem, uint32_t width, uint32_t height, uint64_t* samples_inout,
              int32_t* status);
/* Same, device buffer only, enqueued on `cuda_stream` (a cudaStream_t, taken literally: NULL is
 * the CUDA default stream) without synchronising: the caller orders it with its own events. */
int bt_render_async(bt_engine* engine, bt_scene* scene, uint64_t camera_ref, const bt_config* config,
                    const bt_render_config* render_config, uint64_t seed, uint64_t sample_base,
                    float* rgba32f_device, uint32_t width, uint32_t height, uint64_t* samples_inout,
                    int32_t* status, void* cuda_stream);

/* Work counters of one bt_render call (same scene, config, seeds => same deterministic paths),
 * rendered into a scratch buffer by an instrumented copy of the render kernel; never timed.
 * stats_out = {camera paths, segment-intersection scans (each tests every primitive once), RK4
 * steps, shading events}.  bench.py turns them into the algorithmic flops of SURVEY 8d. */
int bt_render_stats(bt_engine* engine, bt_scene* scene, uint64_t camera_ref, const bt_config* config,
                    const bt_render_config* render_config, uint64_t seed, uint64_t sample_base,
                    uint32_t width, uint32_t height, uint64_t stats_out[4]);

/* Scheduling counters of the pooled render kernel for the same call (an instrumented copy, never timed):
 * stats_out = {STEP iterations, flying lanes summed over them, refill rounds, STEP entries, SCAN passes,
 * slots scanned, SHADE passes, slots shaded, REGEN passes, paths issued, paths retired, turns, SM clocks the
 * warps spent in STEP, SCAN, SHADE, REGEN, SM clocks of the warps' whole lives, STEP iterations in which a lane
 * refreshed its free distance from the lensed grid, those in which lanes inside and outside the grid's box both did,
 * lanes refreshed from a cell of the grid, lanes refreshed outside its box} summed over all warps -- lanes
 * per pass = slots / passes.  BT_ERR_UNSUPPORTED when no content-specialised pooled kernel renders the
 * call: pool_w = 0, a BVH scene, max bounces above 254, more than 126 primitives, or a scene or output
 * that only a generic kernel serves. */
int bt_render_pool_stats(bt_engine* engine, bt_scene* scene, uint64_t camera_ref, const bt_config* config,
                         const bt_render_config* render_config, uint64_t seed, uint64_t sample_base,
                         uint32_t width, uint32_t height, uint64_t stats_out[21]);

/* Buffer::preview, reference src/tracer/buffer.rs:117-138 (+ ColorSpace::convert_linear :19-30,
 * linear_to_srgb / f32_to_u8 src/color.rs:14-24).  rgba8 lives where rgba32f lives. */
int bt_resolve_u8(bt_engine* engine, const float* rgba32f, int mem, uint32_t width, uint32_t height,
                  uint64_t samples, int color_space, uint8_t* rgba8);

/* ---- probes used by the parity tests and the stepper roofline benchmark ---------------- */
/* ChunkState::try_hit (reference src/tracer/mod.rs:389-402) for n rays; under a lens field the
 * geodesic segment that replaces it.  origins / dirs = n*3 floats, host memory. */
int bt_trace_segments(bt_engine* engine, bt_scene* scene, const bt_config* config, uint32_t n,
                      const float* origins, const float* dirs, bt_segment* out);
/* The camera rays render_samples generates (reference src/tracer/mod.rs:272-302) for n
 * (x, y, path index within this call) triples; out = n*6 floats (origin, direction), host memory. */
int bt_camera_rays(bt_engine* engine, bt_scene* scene, uint64_t camera_ref, const bt_config* config,
                   const bt_render_config* render_config, uint64_t seed, uint64_t sample_base,
                   uint32_t width, uint32_t height, uint32_t n, const uint32_t* xs, const uint32_t* ys,
                   const uint64_t* path_index, float* out);
/* Exactly n_steps RK4 steps of n rays through the lens field with the adaptive step rule and no
 * intersection / capture test: the geodesic stepper in isolation (the FP32-roofline kernel).
 * xv = n*6 floats (x, v) updated in place; mem says where xv lives.  BT_MEM_DEVICE: enqueued on
 * cuda_stream (as above), not synchronised.  BT_MEM_HOST: blocking, cuda_stream ignored. */
int bt_geodesic_integrate(bt_engine* engine, const float* xyzr, uint32_t n_lenses,
                          const bt_lens_config* cfg, uint32_t n, float* xv, int mem, uint32_t n_steps,
                          void* cuda_stream);
/* FP32 FMA-chain microbenchmark kernel: the measured FP32 peak the roofline is quoted against.
 * Returns the achieved TFLOP/s (FMA = 2 flops) over `iters` dependent-chain iterations. */
int bt_fp32_peak(bt_engine* engine, uint32_t iters, double* tflops);

const char* bt_last_error(void);

#ifdef __cplusplus
}
#endif
#endif
