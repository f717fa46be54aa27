/*
 * bendy_oracle.h -- C interface of the CPU ORACLE for the bendy-tracer per-sample render loop.
 *
 * THIS IS TEST INFRASTRUCTURE, NOT PRODUCT CODE.  Only tests/, __graft_entry__.smoke() and the
 * cpu_baseline / --impl reference legs of bench.py may load it.  The CUDA engine
 * (bendy_tracer_b200/csrc) never includes, links or calls anything in oracle/.
 *
 * PARITY UNPINNED: the reference (soycan-sim/bendy-tracer) ships no golden vectors, no known
 * answer tests and cannot be compiled here (no Rust toolchain).  The oracle is a line-by-line
 * restatement of the reference sources (each function cites file:line) plus restatements of the
 * published third-party arithmetic it calls (glam 0.21.2, rand 0.8.5 -- versions from
 * Cargo.lock).  The only third-party golden vector available (the xoshiro256++ reference
 * outputs that rand's own test-suite uses) is checked in tests/test_oracle_kat.py.
 */
#ifndef BENDY_ORACLE_H
#define BENDY_ORACLE_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* ObjectKind, reference src/scene/object/mod.rs:247-256 */
enum { ORC_EMPTY = 0, ORC_CAMERA = 1, ORC_SPHERE = 2, ORC_RECT = 3, ORC_CUBOID = 4 };
/* Material, reference src/scene/data/material.rs:22-44 */
enum { ORC_FLAT = 0, ORC_DIFFUSE = 1, ORC_METALLIC = 2, ORC_GLASS = 3, ORC_EMISSIVE = 4 };
/* Output, reference src/tracer/mod.rs:108-115 */
enum { ORC_OUT_FULL = 0, ORC_OUT_ALBEDO = 1, ORC_OUT_NORMAL = 2, ORC_OUT_DEPTH = 3 };
/* ColorSpace, reference src/tracer/buffer.rs:11-17 */
enum { ORC_CS_NONE = 0, ORC_CS_NORMAL = 1, ORC_CS_LINEAR = 2, ORC_CS_SRGB = 3 };
/* Face, reference src/tracer/ray.rs:8-15 (+ miss / capture codes used by the probe) */
enum { ORC_FACE_FRONT = 0, ORC_FACE_BACK = 1, ORC_FACE_VOLUME = 2, ORC_FACE_VOLUME_FRONT = 3,
       ORC_FACE_VOLUME_BACK = 4, ORC_FACE_MISS = -1, ORC_FACE_CAPTURED = -2 };
/* camera projection extension (NOT in the reference): the engine's BT_PROJECTION_* values */
enum { ORC_PROJECTION_PERSPECTIVE = 0, ORC_PROJECTION_EQUIRECTANGULAR = 1 };

typedef struct {            /* Rect, reference src/scene/object/rect.rs:11-19 */
    uint64_t material;
    float half_width, half_height;
    float x[3], y[3], z[3];
} orc_rect;

typedef struct {            /* Object, reference src/scene/object/mod.rs:33-41 */
    uint64_t object_ref;
    uint32_t kind;
    uint32_t flags;         /* ObjectFlags bits, LIGHT = 1 */
    float transform[12];    /* transform_world: x_axis, y_axis, z_axis, translation (glam Affine3A) */
    /* Sphere (sphere.rs:11-16) */
    uint64_t material;
    int64_t volume;         /* -1 = None */
    float radius;
    /* Camera (camera.rs:3-10) */
    float sensor_size, focal_length, aspect_ratio, fstop, focus;
    int32_t has_focus;
    /* Rect */
    orc_rect rect;
    /* Cuboid (cuboid.rs:12-15): faces[i] = (offset, rect) */
    float face_offset[6][3];
    orc_rect faces[6];
} orc_object;

typedef struct {            /* Data, reference src/scene/data/mod.rs:9-51 */
    uint64_t data_ref;
    uint32_t kind;          /* 0 material, 1 volume */
    uint32_t mat_kind;
    float albedo[3];
    float roughness, ior, intensity;
    uint32_t width, height, depth;   /* DensityMap, volume.rs:75-82 */
    float size[3];
    const float* buffer;    /* copied by orc_scene_create */
} orc_data;

typedef struct {            /* Config + RenderConfig, reference src/tracer/mod.rs:16-45,117-135 */
    uint64_t max_bounces, max_volume_bounces;
    float clip_min, clip_max, volume_step;
    uint32_t chunks_x, chunks_y;
    int32_t output;
    /* RenderConfig */
    uint64_t samples;
    uint32_t subsample;                 /* 0 = Subsample::None, n = Subpixel(n) */
    int32_t has_output, r_output;
    int32_t has_max_bounces; uint64_t r_max_bounces;
    int32_t has_max_volume_bounces; uint64_t r_max_volume_bounces;
    int32_t has_volume_step; float r_volume_step;
} orc_config;

typedef struct {            /* lensing extension (NOT in the reference; DESIGN.md "Geodesic model") */
    float kappa, h_min, h_max, r_far;
    uint32_t max_steps;
} orc_lens_config;

typedef struct {            /* result of one traced segment (try_hit or geodesic) */
    int32_t face;           /* ORC_FACE_* */
    uint32_t steps;         /* RK4 steps taken (0 in a flat field) */
    uint64_t object_ref;
    double t;               /* accumulated chord length to the hit */
    double position[3];
    double normal[3];
    double direction[3];    /* unit direction of the last chord / escape direction */
} orc_probe_result;

void* orc_scene_create(const orc_object* objects, int n_objects, const orc_data* data, int n_data,
                       uint64_t root_material);
void orc_scene_set_lenses(void* scene, const float* xyzr, int n, const orc_lens_config* cfg);
int orc_scene_set_camera_aspect(void* scene, uint64_t camera_ref, float aspect);
/* environment map extension (NOT in the reference; DESIGN.md §3.5): width * height RGB texels,
 * row 0 = +y pole, copied; rgb = NULL or a zero size clears the map.  Returns 0. */
int orc_scene_set_environment(void* scene, const float* rgb, uint32_t width, uint32_t height);
/* camera projection extension (NOT in the reference; DESIGN.md §3.6): ORC_PROJECTION_*.
 * returns 0, or -1 (message via orc_last_error, scene unchanged) for a reference that is not a
 * camera or an unknown projection */
int orc_scene_set_camera_projection(void* scene, uint64_t camera_ref, int projection);
void orc_scene_destroy(void* scene);

/* Tracer::render (src/tracer/mod.rs:179-202) with the keyed RNG stream of DESIGN.md.
 * returns 0 = Status::Done, 1 = Status::InProgress, <0 = a reference panic (message via orc_last_error) */
int orc_render(void* scene, uint64_t camera_ref, const orc_config* cfg, uint64_t seed,
               uint64_t sample_base, float* rgba32f, uint32_t width, uint32_t height, int n_threads,
               uint64_t* samples_inout);
/* Buffer::preview (src/tracer/buffer.rs:117-138) */
void orc_resolve_u8(const float* rgba32f, uint32_t width, uint32_t height, uint64_t samples,
                    int color_space, uint8_t* rgba8);
/* first segment only: try_hit (flat field) or the geodesic trace; f32 or f64 arithmetic */
int orc_probe(void* scene, const orc_config* cfg, int n, const float* origins, const float* dirs,
              int use_f64, orc_probe_result* out);
/* camera rays exactly as render_samples generates them (for ray-gen parity): out = n*6 floats */
int orc_camera_rays(void* scene, uint64_t camera_ref, const orc_config* cfg, uint64_t seed,
                    uint64_t sample_base, uint32_t width, uint32_t height, int n,
                    const uint32_t* xs, const uint32_t* ys, const uint64_t* path_index, float* out);
/* exactly n_steps RK4 steps with the adaptive step rule, no intersection / capture test.
 * xv = n * 6 (x, v), updated in place as f32 (use_f64: integrated in double from the f32 input,
 * written to out64 = n * 6 doubles). */
void orc_integrate(const float* xyzr, int n_lens, const orc_lens_config* cfg, int n, const float* xv,
                   uint32_t n_steps, int use_f64, float* out32, double* out64);
const char* orc_last_error(void);

/* ---- unit-level exports for known-answer tests ---- */
void orc_xoshiro_from_seed(const uint64_t s[4], uint64_t* out, int n);       /* raw next_u64 stream */
void orc_xoshiro_seed_from_u64(uint64_t seed, uint64_t state_out[4]);
uint64_t orc_path_seed(uint64_t seed, uint64_t pixel, uint64_t path_index);
void orc_uniform_f32(uint64_t seed, float lo, float hi, int inclusive, float* out, int n, float* scale_out);
void orc_standard_f32(uint64_t seed, float* out, int n);
int orc_gen_bool(uint64_t seed, double p, uint8_t* out, int n);
int orc_uniform_usize(uint64_t seed, uint64_t n_range, uint64_t* out, int n);
void orc_with_frustum(float yfov, float xfov, float u, float v, float dir_out[3]);
/* the environment map's factor for one direction (any d: non-unit, zero, NaN / inf components) */
void orc_environment_lookup(const float* rgb, uint32_t width, uint32_t height, const float d[3], float out[3]);
/* the equirectangular camera-space direction for the NDC (u, v) before the half-pixel offset */
void orc_equirect_dir(float u, float v, float pixel_width, float pixel_height, float out[3]);
void orc_any_orthonormal_pair(const float n[3], float a_out[3], float b_out[3]);
void orc_distr(int which /*0 sphere,1 hemisphere,2 cosine,3 disk*/, uint64_t seed, const float n[3],
               float* out, int count);
int orc_sphere_hit(const float center[3], float radius, const float o[3], const float d[3],
                   float clip_min, float clip_max, float* t_out, float normal_out[3], int* face_out);
int orc_rect_hit(const orc_rect* rect, const float transform[12], const float o[3], const float d[3],
                 float clip_min, float clip_max, float* t_out, float normal_out[3], int* face_out);
float orc_density_sample(const orc_data* vol, const float coord[3]);
void orc_reflect(const float d[3], const float n[3], float out[3]);
void orc_refract(const float d[3], const float n[3], float ior, float out[3]);
float orc_fresnel(const float d[3], const float n[3], float ior);
float orc_linear_to_srgb(float x);
/* one RK4 step of the lens field; state = x[3], v[3]; returns in place */
void orc_rk4_step_f32(const float* xyzr, int n_lens, float* x, float* v, float h);
void orc_rk4_step_f64(const float* xyzr, int n_lens, double* x, double* v, double h);

#ifdef __cplusplus
}
#endif
#endif
