// oracle_env.cpp -- TEST INFRASTRUCTURE: the CPU oracle (oracle/bendy_oracle.cpp, compiled here unchanged) with the
// environment-map extension of the engine (DESIGN.md §3.5): sample_root's colour times the bilinear lookup of an
// equirectangular map in the escape direction.  Built and loaded by tests/oracle_env.py.
//
// The oracle has ONE definition of sample_root (mod.rs:429-452) and three calls, all inside ChunkState.  The macro below
// tells them apart by the first token of the argument: the definition's is `const` and keeps its body under the name
// sample_root_plain; a call -- `ray` or `seg.escape` -- becomes env_root(this, <arg>), which calls sample_root_plain and
// multiplies the colour when the scene has a map (without one, this library renders exactly what
// oracle/libbendy_oracle.so renders).
#include <cmath>
#include <cstdint>
#include <map>
#include <mutex>
#include <vector>

template <class CS, class R>
auto env_root(CS* cs, const R& ray) -> decltype(cs->sample_root_plain(ray));

#define sample_root(x) ENV_ROOT_##x)
#define ENV_ROOT_const sample_root_plain(const
#define ENV_ROOT_ray env_root(this, ray
#define ENV_ROOT_seg env_root(this, seg
#include "../oracle/bendy_oracle.cpp"
#undef sample_root

namespace {

struct EnvMap {
    std::vector<float> rgb;  // w * h RGB texels, row 0 = +y pole
    uint32_t w = 0, h = 0;
};
std::mutex g_env_lock;
std::map<const void*, EnvMap> g_env;  // per oracle scene; written only between renders

// The lookup of device.cuh (env_lookup), operation for operation: every product and sum rounded on its own (this file
// is compiled -ffp-contract=off), atan2 / sqrt from libm.
V3f lookup(const float* rgb, uint32_t w, uint32_t h, V3f d) {
    const float phi = std::atan2(d.x, -d.z), theta = std::atan2(d.y, std::sqrt(d.x * d.x + d.z * d.z));
    const float u = 0.5f + phi * 0.159154943091895335769f, v = 0.5f - theta * 0.318309886183790671538f;  // 1/(2 pi), 1/pi
    const float x = std::fmin(std::fmax(u * (float)w - 0.5f, -1.0f), (float)w);
    const float y = std::fmin(std::fmax(v * (float)h - 0.5f, -1.0f), (float)h);
    const float fx = std::floor(x), fy = std::floor(y), tx = x - fx, ty = y - fy;
    const uint32_t c0 = fx < 0.0f ? w - 1 : std::min((uint32_t)fx, w - 1), c1 = c0 + 1 == w ? 0 : c0 + 1;
    const uint32_t r0 = fy < 0.0f ? 0 : std::min((uint32_t)fy, h - 1), r1 = fy < 0.0f ? 0 : std::min((uint32_t)fy + 1, h - 1);
    const float *a = rgb + 3 * ((size_t)r0 * w + c0), *b = rgb + 3 * ((size_t)r0 * w + c1);
    const float *c = rgb + 3 * ((size_t)r1 * w + c0), *e = rgb + 3 * ((size_t)r1 * w + c1);
    float out[3];
    for (int k = 0; k < 3; ++k) out[k] = lerp(lerp(a[k], b[k], tx), lerp(c[k], e[k], tx), ty);
    return mk<float>(out[0], out[1], out[2]);
}

}  // namespace

template <class CS, class R>
auto env_root(CS* cs, const R& ray) -> decltype(cs->sample_root_plain(ray)) {
    auto cd = cs->sample_root_plain(ray);
    std::map<const void*, EnvMap>::const_iterator it = g_env.find(cs->scene);
    if (it != g_env.end()) cd.color = cd.color * lookup(it->second.rgb.data(), it->second.w, it->second.h, ray.direction);
    return cd;
}

extern "C" {

// rgb = NULL (or a zero size) clears the scene's map; the texels are copied
void orc_env_set(void* scene, const float* rgb, uint32_t width, uint32_t height) {
    std::lock_guard<std::mutex> g(g_env_lock);
    if (!rgb || width == 0 || height == 0) {
        g_env.erase(scene);
        return;
    }
    EnvMap& m = g_env[scene];
    m.rgb.assign(rgb, rgb + (size_t)width * height * 3);
    m.w = width;
    m.h = height;
}

// orc_scene_destroy that also forgets the scene's map (a later scene may get the same address)
void orc_env_scene_destroy(void* scene) {
    orc_env_set(scene, nullptr, 0, 0);
    orc_scene_destroy(scene);
}

// the lookup for one direction (any d: non-unit, zero, NaN / inf components)
void orc_env_lookup(const float* rgb, uint32_t width, uint32_t height, const float d[3], float out[3]) {
    const V3f c = lookup(rgb, width, height, mk<float>(d[0], d[1], d[2]));
    out[0] = c.x;
    out[1] = c.y;
    out[2] = c.z;
}

}  // extern "C"
