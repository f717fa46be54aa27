// oracle_camera.cpp -- TEST INFRASTRUCTURE: the CPU oracle with the environment map (tests/oracle_env.cpp, which compiles
// oracle/bendy_oracle.cpp unchanged) and the engine's equirectangular camera projection (DESIGN.md §3.6).  Built and loaded
// by tests/oracle_camera.py.
//
// The oracle has ONE definition of camera_ray (mod.rs:272-302) and two calls: the render loop and orc_camera_rays.  As in
// oracle_env.cpp, the macro below tells them apart by the first token of the argument list: the definition's is `const` and
// keeps its body under the name camera_ray_plain; a call -- first argument `cs` -- becomes camera_ray_projected(cs, ...),
// which renders a panorama when the camera (keyed on cs.cam_obj) has been switched to it and otherwise calls
// camera_ray_plain (without a projection set, this library renders exactly what oracle_env renders).
#include <cmath>
#include <cstdint>
#include <map>

template <class CS, class R>
auto camera_ray_projected(const CS& cs, R& rng, uint32_t x, uint32_t y, uint32_t sub_index)
    -> decltype(camera_ray_plain(cs, rng, x, y, sub_index));

#define camera_ray(x, ...) CAM_RAY_##x, __VA_ARGS__)
#define CAM_RAY_const camera_ray_plain(const
#define CAM_RAY_cs camera_ray_projected(cs
#include "oracle_env.cpp"
#undef camera_ray

namespace {

enum { PROJ_PERSPECTIVE = 0, PROJ_EQUIRECTANGULAR = 1 };
std::map<const void*, int> g_projection;  // per camera object (orc_object*) that is not PERSPECTIVE; written only between renders

// device.cuh's sincos_poly, operation for operation: Cody-Waite reduction by pi/2 and the Cephes polynomials in explicit FMAs
void sincos_poly(float x, float* sn, float* cs) {
    const float k = std::rint(x * 0.636619772367581343f);
    float y = std::fma(k, -1.5703125f, x);
    y = std::fma(k, -4.837512969970703125e-4f, y);
    y = std::fma(k, -7.549789954891882e-8f, y);
    const int q = (int)k;
    const float y2 = y * y;
    float s = std::fma(-1.9515295891e-4f, y2, 8.3321608736e-3f);
    s = std::fma(s, y2, -1.6666654611e-1f);
    s = std::fma(s * y2, y, y);
    float c = std::fma(2.443315711809948e-5f, y2, -1.388731625493765e-3f);
    c = std::fma(c, y2, 4.166664568298827e-2f);
    c = std::fma(c * y2, y2, std::fma(-0.5f, y2, 1.0f));
    const float a = (q & 1) ? c : s, b = (q & 1) ? s : c;
    *sn = (q & 2) ? -a : a;
    *cs = ((q + 1) & 2) ? -b : b;
}

// device.cuh camera_ray's equirectangular branch, operation for operation (this file is compiled -ffp-contract=off):
// (u, v) are the jittered NDC coordinates before the half-pixel offset
V3f equirect_dir(float u, float v, float pixel_width, float pixel_height) {
    const float phi = 3.14159274101257324f * (u + pixel_width * 0.5f);
    const float theta = -1.57079637050628662f * (v + pixel_height * 0.5f);
    float sp, cp, st, ct;
    sincos_poly(phi, &sp, &cp);
    sincos_poly(theta, &st, &ct);
    return mk<float>(ct * sp, st, -(ct * cp));
}

}  // namespace

template <class CS, class R>
auto camera_ray_projected(const CS& cs, R& rng, uint32_t x, uint32_t y, uint32_t sub_index)
    -> decltype(camera_ray_plain(cs, rng, x, y, sub_index)) {
    if (g_projection.find(cs.cam_obj) == g_projection.end()) return camera_ray_plain(cs, rng, x, y, sub_index);
    // (u, v) exactly as camera_ray_plain forms them: the same two draws, no unit-disk draws after them (a pinhole)
    float v = (float)y * cs.pixel_height - 1.0f;
    float u = (float)x * cs.pixel_width - 1.0f;
    float u_sub = 0.0f, v_sub = 0.0f;
    if (cs.sub_width != 0.0f) {
        uint32_t i = sub_index % cs.sub_n, j = sub_index / cs.sub_n;
        u_sub = (float)i * cs.sub_width;
        v_sub = (float)j * cs.sub_width;
    }
    float u_offset = u_sub * cs.pixel_width + cs.scatter_u.sample(rng);
    float v_offset = v_sub * cs.pixel_height + cs.scatter_v.sample(rng);
    u = u + u_offset;
    v = v + v_offset;
    const V3f dir_cam = equirect_dir(u, v, cs.pixel_width, cs.pixel_height);
    V3f origin = cs.tf.translation + mk<float>(0, 0, 0);  // Affine3A * Ray, ray.rs:126-137
    V3f direction = normalize_or_zero_s(transform_vector(cs.tf, dir_cam));
    return ray_new(origin, direction);
}

extern "C" {

// 0: PERSPECTIVE, 1: EQUIRECTANGULAR; -1 (and the scene unchanged) for a reference that is not a camera or another value
int orc_cam_set_projection(void* scene, uint64_t camera_ref, int projection) {
    Scene* s = (Scene*)scene;
    std::map<uint64_t, int>::iterator it = s->object_index.find(camera_ref);
    if (it == s->object_index.end() || s->objects[it->second].kind != ORC_CAMERA) {
        g_last_error = g_last_error_shared = "expected a camera object";
        return -1;
    }
    if (projection != PROJ_PERSPECTIVE && projection != PROJ_EQUIRECTANGULAR) {
        g_last_error = g_last_error_shared = "unknown projection";
        return -1;
    }
    const void* key = &s->objects[it->second];
    if (projection == PROJ_PERSPECTIVE) g_projection.erase(key);
    else g_projection[key] = projection;
    return 0;
}

// orc_env_scene_destroy that also forgets the scene's projections (a later scene may get the same addresses)
void orc_cam_scene_destroy(void* scene) {
    Scene* s = (Scene*)scene;
    for (size_t i = 0; i < s->objects.size(); ++i) g_projection.erase(&s->objects[i]);
    orc_env_scene_destroy(scene);
}

// the camera-space direction of an equirectangular camera for the NDC (u, v) before the half-pixel offset
void orc_cam_equirect_dir(float u, float v, float pixel_width, float pixel_height, float out[3]) {
    const V3f d = equirect_dir(u, v, pixel_width, pixel_height);
    out[0] = d.x;
    out[1] = d.y;
    out[2] = d.z;
}

}  // extern "C"
