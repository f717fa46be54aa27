/*
 * bendy_oracle.cpp -- CPU ORACLE: a restatement of soycan-sim/bendy-tracer's per-sample render
 * loop in scalar C++ (IEEE f32, no FMA contraction; build with -ffp-contract=off).
 *
 * THIS IS TEST INFRASTRUCTURE, NOT PRODUCT CODE (see bendy_oracle.h).  PARITY UNPINNED: the
 * reference holds no golden vectors and cannot be built here; every function cites the
 * reference file:line it follows.  Third-party arithmetic (glam 0.21.2, rand 0.8.5) is restated
 * from the published crates; where the exact operation order of a crate matters it is written
 * out explicitly and marked [glam] / [rand].
 *
 * Deliberate deviations from the reference (DESIGN.md):
 *   - RNG: one xoshiro256++ stream per camera path, keyed by (seed, pixel, path index), instead
 *     of SmallRng::from_entropy() per tile (src/tracer/mod.rs:239-242).
 *   - Object iteration order: ascending ObjectRef instead of hashbrown's per-process order.
 *   - Lensing (geodesic segments) exists only when lenses are set; with none the code path is
 *     the reference's try_hit.
 *   - The environment map and the equirectangular camera exist only when set; with neither the
 *     code paths are the reference's sample_root and camera_ray.
 */
#include "bendy_oracle.h"

#include <algorithm>
#include <atomic>
#include <cmath>
#include <cstring>
#include <limits>
#include <map>
#include <stdexcept>
#include <string>
#include <thread>
#include <vector>

namespace {

struct Panic : std::runtime_error {
    explicit Panic(const std::string& m) : std::runtime_error(m) {}
};
thread_local std::string g_last_error;
std::string g_last_error_shared;

// ------------------------------------------------------------------------------------------
// [glam] vector arithmetic.  T = float for the render path, double for the f64 probe.
// ------------------------------------------------------------------------------------------
template <class T>
struct V3 {
    T x, y, z;
};
typedef V3<float> V3f;

template <class T> inline V3<T> mk(T x, T y, T z) { V3<T> r = {x, y, z}; return r; }
template <class T> inline V3<T> operator+(V3<T> a, V3<T> b) { return mk<T>(a.x + b.x, a.y + b.y, a.z + b.z); }
template <class T> inline V3<T> operator-(V3<T> a, V3<T> b) { return mk<T>(a.x - b.x, a.y - b.y, a.z - b.z); }
template <class T> inline V3<T> operator-(V3<T> a) { return mk<T>(-a.x, -a.y, -a.z); }
template <class T> inline V3<T> operator*(V3<T> a, T s) { return mk<T>(a.x * s, a.y * s, a.z * s); }
template <class T> inline V3<T> operator*(T s, V3<T> a) { return mk<T>(s * a.x, s * a.y, s * a.z); }
template <class T> inline V3<T> operator*(V3<T> a, V3<T> b) { return mk<T>(a.x * b.x, a.y * b.y, a.z * b.z); }
template <class T> inline V3<T> operator/(V3<T> a, T s) { return mk<T>(a.x / s, a.y / s, a.z / s); }
template <class T> inline V3<T> operator/(V3<T> a, V3<T> b) { return mk<T>(a.x / b.x, a.y / b.y, a.z / b.z); }
// [glam] dot3: (x*x' + y*y') + z*z'
template <class T> inline T dot(V3<T> a, V3<T> b) { return (a.x * b.x + a.y * b.y) + a.z * b.z; }
template <class T> inline V3<T> cross(V3<T> a, V3<T> b) {
    return mk<T>(a.y * b.z - b.y * a.z, a.z * b.x - b.z * a.x, a.x * b.y - b.x * a.y);
}
template <class T> inline T length_squared(V3<T> a) { return dot(a, a); }
template <class T> inline T length(V3<T> a) { return std::sqrt(dot(a, a)); }
// [glam] Vec3A::normalize (sse2): v / sqrt(dot)
template <class T> inline V3<T> normalize_a(V3<T> a) { return a / length(a); }
// [glam] Vec3::normalize (scalar): v * (1 / sqrt(dot))
template <class T> inline V3<T> normalize_s(V3<T> a) { return a * (T(1) / length(a)); }
template <class T> inline V3<T> normalize_or_zero_s(V3<T> a) {
    T rcp = T(1) / length(a);
    if (std::isfinite(rcp) && rcp > T(0)) return a * rcp;
    return mk<T>(0, 0, 0);
}
template <class T> inline V3<T> vmin(V3<T> a, V3<T> b) { return mk<T>(std::min(a.x, b.x), std::min(a.y, b.y), std::min(a.z, b.z)); }
template <class T> inline V3<T> vmax(V3<T> a, V3<T> b) { return mk<T>(std::max(a.x, b.x), std::max(a.y, b.y), std::max(a.z, b.z)); }
template <class T> inline V3<T> splat(T s) { return mk<T>(s, s, s); }

// [glam] Affine3A: matrix3 columns + translation (serialised as 12 floats in this order)
template <class T>
struct Affine {
    V3<T> x_axis, y_axis, z_axis, translation;
};
template <class T> inline V3<T> transform_vector(const Affine<T>& m, V3<T> v) {
    V3<T> r = m.x_axis * v.x;
    r = r + m.y_axis * v.y;
    r = r + m.z_axis * v.z;
    return r;
}
template <class T> inline V3<T> transform_point(const Affine<T>& m, V3<T> v) {
    return transform_vector(m, v) + m.translation;
}
// Affine3A * Affine3A::from_translation(offset)  (cuboid.rs:39,52,68,95)
template <class T> inline Affine<T> mul_translation(const Affine<T>& m, V3<T> offset) {
    Affine<T> r = m;
    r.translation = transform_vector(m, offset) + m.translation;
    return r;
}
// [glam] Affine3A::inverse = Mat3A::inverse (cross products / determinant, transposed) + -(inv * t)
template <class T> inline Affine<T> inverse(const Affine<T>& m) {
    V3<T> tmp0 = cross(m.y_axis, m.z_axis);
    V3<T> tmp1 = cross(m.z_axis, m.x_axis);
    V3<T> tmp2 = cross(m.x_axis, m.y_axis);
    T det = dot(m.z_axis, tmp2);
    T inv_det = T(1) / det;
    V3<T> c0 = tmp0 * inv_det, c1 = tmp1 * inv_det, c2 = tmp2 * inv_det;
    Affine<T> r;
    r.x_axis = mk<T>(c0.x, c1.x, c2.x);
    r.y_axis = mk<T>(c0.y, c1.y, c2.y);
    r.z_axis = mk<T>(c0.z, c1.z, c2.z);
    r.translation = -transform_vector(r, m.translation);
    return r;
}
template <class T> inline Affine<T> affine_from(const float* f) {
    Affine<T> a;
    a.x_axis = mk<T>(f[0], f[1], f[2]);
    a.y_axis = mk<T>(f[3], f[4], f[5]);
    a.z_axis = mk<T>(f[6], f[7], f[8]);
    a.translation = mk<T>(f[9], f[10], f[11]);
    return a;
}
template <class T> inline V3<T> v3_from(const float* f) { return mk<T>(f[0], f[1], f[2]); }

// [glam] Vec3::any_orthonormal_pair (branch-free ONB)
inline void any_orthonormal_pair(V3f n, V3f* a_out, V3f* b_out) {
    float sign = std::copysign(1.0f, n.z);
    float a = -1.0f / (sign + n.z);
    float b = n.x * n.y * a;
    *a_out = mk<float>(1.0f + sign * n.x * n.x * a, sign * b, -sign * n.x);
    *b_out = mk<float>(b, sign + n.y * n.y * a, -n.y);
}

// src/math/mod.rs:5-25
inline float lerp(float a, float b, float f) { return a + (b - a) * f; }
// src/math/mod.rs:39-41
inline V3f reflect(V3f d, V3f n) { return d - (2.0f * dot(d, n)) * n; }
// src/math/mod.rs:43-48
inline V3f refract(V3f d, V3f n, float ior) {
    float cos_theta = std::min(dot(-d, n), 1.0f);
    V3f perp = (n * cos_theta + d) * ior;
    V3f parallel = n * -std::sqrt(std::fabs(1.0f - length_squared(perp)));
    return perp + parallel;
}
// src/math/mod.rs:50-55; powi(5) = x * ((x*x)*(x*x)) (compiler-rt __powisf2 order)
inline float fresnel(V3f d, V3f n, float ior) {
    float cos_theta = std::min(dot(-d, n), 1.0f);
    float r0 = (1.0f - ior) / (1.0f + ior);
    r0 = r0 * r0;
    float x = 1.0f - cos_theta;
    float x2 = x * x;
    float x4 = x2 * x2;
    return r0 + (1.0f - r0) * (x * x4);
}

// ------------------------------------------------------------------------------------------
// [rand] SmallRng = xoshiro256++ (64-bit targets), Uniform<f32>, Standard, Bernoulli, Uniform<usize>
// ------------------------------------------------------------------------------------------
inline uint64_t rotl64(uint64_t x, int k) { return (x << k) | (x >> (64 - k)); }
inline uint64_t splitmix_mix(uint64_t z) {
    z = (z ^ (z >> 30)) * 0xbf58476d1ce4e5b9ULL;
    z = (z ^ (z >> 27)) * 0x94d049bb133111ebULL;
    return z ^ (z >> 31);
}
struct Rng {
    uint64_t s[4];
    uint64_t next_u64() {
        uint64_t result = rotl64(s[0] + s[3], 23) + s[0];
        uint64_t t = s[1] << 17;
        s[2] ^= s[0];
        s[3] ^= s[1];
        s[1] ^= s[2];
        s[0] ^= s[3];
        s[2] ^= t;
        s[3] = rotl64(s[3], 45);
        return result;
    }
    // [rand] xoshiro256plusplus.rs: next_u32 = upper half of next_u64
    uint32_t next_u32() { return (uint32_t)(next_u64() >> 32); }
    // [rand] Xoshiro256PlusPlus::seed_from_u64: SplitMix64 x 4
    static Rng seed_from_u64(uint64_t state) {
        Rng r;
        for (int i = 0; i < 4; ++i) {
            state += 0x9e3779b97f4a7c15ULL;
            r.s[i] = splitmix_mix(state);
        }
        if ((r.s[0] | r.s[1] | r.s[2] | r.s[3]) == 0) return seed_from_u64(0);
        return r;
    }
};

// keyed stream (replaces from_entropy, src/tracer/mod.rs:239-242) -- DESIGN.md "RNG keying"
inline uint64_t path_seed(uint64_t seed, uint64_t pixel, uint64_t path_index) {
    uint64_t k = splitmix_mix(seed + 0x9e3779b97f4a7c15ULL);
    k = splitmix_mix(k + 0x9e3779b97f4a7c15ULL * (pixel + 1));
    k = splitmix_mix(k + 0xd1342543de82ef95ULL * (path_index + 1));
    return k;
}

inline float f32_dec(float x) {
    uint32_t b;
    std::memcpy(&b, &x, 4);
    b -= 1;
    std::memcpy(&x, &b, 4);
    return x;
}
// [rand] UniformFloat<f32>::new / new_inclusive / sample
struct UniformF32 {
    float low, scale;
    static UniformF32 make(float low, float high) {
        if (!(low < high)) throw Panic("Uniform::new called with `low >= high`");
        const float max_rand = 1.0f - 1.1920929e-07f;
        float scale = high - low;
        while (scale * max_rand + low >= high) scale = f32_dec(scale);
        UniformF32 u = {low, scale};
        return u;
    }
    static UniformF32 make_inclusive(float low, float high) {
        if (!(low <= high)) throw Panic("Uniform::new_inclusive called with `low > high`");
        const float max_rand = 1.0f - 1.1920929e-07f;
        float scale = (high - low) / max_rand;
        while (scale * max_rand + low > high) scale = f32_dec(scale);
        UniformF32 u = {low, scale};
        return u;
    }
    float sample(Rng& rng) const {
        uint32_t bits = (rng.next_u32() >> 9) | 0x3f800000u;
        float value1_2;
        std::memcpy(&value1_2, &bits, 4);
        float value0_1 = value1_2 - 1.0f;
        return value0_1 * scale + low;
    }
};
// [rand] Standard for f32: 24 bits * 2^-24
inline float standard_f32(Rng& rng) { return (float)(rng.next_u32() >> 8) * (1.0f / 16777216.0f); }
// [rand] Rng::gen_bool -> Bernoulli::new(p).sample
inline bool gen_bool(Rng& rng, double p) {
    if (!(p >= 0.0 && p < 1.0)) {
        if (p == 1.0) return true;
        throw Panic("p is outside range [0.0, 1.0]");
    }
    uint64_t p_int = (uint64_t)(p * 18446744073709551616.0);
    uint64_t v = rng.next_u64();
    return v < p_int;
}
// [rand] UniformInt<usize>::new(0, n).sample  (widening multiply + rejection zone)
inline uint64_t uniform_usize(Rng& rng, uint64_t n) {
    if (n == 0) throw Panic("Uniform::new called with `low >= high`");
    uint64_t range = n;
    uint64_t ints_to_reject = (UINT64_MAX - range + 1) % range;
    uint64_t zone = UINT64_MAX - ints_to_reject;
    for (;;) {
        uint64_t v = rng.next_u64();
        unsigned __int128 m = (unsigned __int128)v * range;
        uint64_t hi = (uint64_t)(m >> 64), lo = (uint64_t)m;
        if (lo <= zone) return hi;
    }
}

const float TAU = 6.28318530717958647692f;

// src/math/distr.rs:7-27
inline V3f unit_sphere(Rng& rng) {
    float r1 = UniformF32::make_inclusive(0.0f, TAU).sample(rng);
    float r2 = UniformF32::make_inclusive(0.0f, 1.0f).sample(rng);
    float x = std::cos(r1) * 2.0f * std::sqrt(r2 * (1.0f - r2));
    float y = std::sin(r1) * 2.0f * std::sqrt(r2 * (1.0f - r2));
    float z = 1.0f - 2.0f * r2;
    return mk<float>(x, y, z);
}
struct Basis {
    V3f x_axis, y_axis, z_axis;
    explicit Basis(V3f normal) {
        z_axis = normalize_s(normal);
        any_orthonormal_pair(z_axis, &x_axis, &y_axis);
    }
};
// src/math/distr.rs:29-65  (not unit length: z = 1 - r2)
inline V3f unit_hemisphere(Rng& rng, const Basis& b) {
    float r1 = UniformF32::make_inclusive(0.0f, TAU).sample(rng);
    float r2 = UniformF32::make_inclusive(0.0f, 1.0f).sample(rng);
    float x = std::cos(r1) * 2.0f * std::sqrt(r2 * (1.0f - r2));
    float y = std::sin(r1) * 2.0f * std::sqrt(r2 * (1.0f - r2));
    float z = 1.0f - r2;
    return b.x_axis * x + b.y_axis * y + b.z_axis * z;
}
// src/math/distr.rs:67-103
inline V3f cosine(Rng& rng, const Basis& b) {
    float r1 = UniformF32::make_inclusive(0.0f, TAU).sample(rng);
    float r2 = UniformF32::make_inclusive(0.0f, 1.0f).sample(rng);
    float x = std::cos(r1) * std::sqrt(r2);
    float y = std::sin(r1) * std::sqrt(r2);
    float z = std::sqrt(1.0f - r2);
    return b.x_axis * x + b.y_axis * y + b.z_axis * z;
}
// src/math/distr.rs:105-138  (radius linear in U)
inline V3f unit_disk(Rng& rng, const Basis& b) {
    float angle = UniformF32::make_inclusive(0.0f, TAU).sample(rng);
    float r = UniformF32::make_inclusive(0.0f, 1.0f).sample(rng);
    float x = std::cos(angle);
    float y = std::sin(angle);
    return (b.x_axis * x + b.y_axis * y) * r;
}

// ------------------------------------------------------------------------------------------
// scene model
// ------------------------------------------------------------------------------------------
struct Data {
    orc_data d;
    std::vector<float> buffer;
};
struct Lens {
    float c[3];
    float rs;
};
struct Scene {
    std::vector<orc_object> objects;  // ascending object_ref: the canonical iteration order
    std::map<uint64_t, int> object_index;
    std::map<uint64_t, Data> data;
    uint64_t root_material;
    std::vector<Lens> lenses;
    orc_lens_config lens_cfg;
    std::vector<float> env_rgb;          // environment map: env_w * env_h RGB texels, row 0 = +y pole
    uint32_t env_w = 0, env_h = 0;       // env_w == 0: no map
    std::map<uint64_t, int> projection;  // camera object_ref -> ORC_PROJECTION_*, only for cameras that are not PERSPECTIVE

    const orc_object& get_object(uint64_t r) const {  // src/scene/mod.rs:131-133
        std::map<uint64_t, int>::const_iterator it = object_index.find(r);
        if (it == object_index.end()) throw Panic("invalid object ref");
        return objects[it->second];
    }
    const Data& get_data(uint64_t r) const {  // src/scene/mod.rs:135-137
        std::map<uint64_t, Data>::const_iterator it = data.find(r);
        if (it == data.end()) throw Panic("invalid data ref");
        return it->second;
    }
    const Data& get_material(uint64_t r, const char* what) const {
        const Data& d = get_data(r);
        if (d.d.kind != 0) throw Panic(what);
        return d;
    }
};

template <class T>
struct Ray {
    V3<T> origin, direction;
};
typedef Ray<float> Rayf;
// src/tracer/ray.rs:96-101
template <class T> inline Ray<T> ray_new(V3<T> o, V3<T> d) {
    Ray<T> r = {o, normalize_a(d)};
    return r;
}
template <class T> inline V3<T> ray_at(const Ray<T>& r, T t) { return r.origin + t * r.direction; }

template <class T>
struct Clip {
    T min, max;
};

template <class T>
struct Manifold {  // src/tracer/ray.rs:36-47
    V3<T> position, normal, bbox_min, bbox_max;
    int face;
    T t;
    Ray<T> ray;
    bool has_object;
    uint64_t object_ref;
    bool has_mat;
    uint64_t mat_ref;
    bool has_vol;
    uint64_t vol_ref;
};

struct ColorData {  // src/tracer/ray.rs:49-76
    V3f color, albedo, normal;
    float depth;
    ColorData() : color(mk<float>(0, 0, 0)), albedo(mk<float>(0, 0, 0)), normal(mk<float>(0, 0, 0)),
                  depth(std::numeric_limits<float>::infinity()) {}
    static ColorData from_emitted(V3f e) {
        ColorData c;
        c.color = e;
        c.albedo = e;
        return c;
    }
};

// ------------------------------------------------------------------------------------------
// primitives
// ------------------------------------------------------------------------------------------
// src/scene/object/sphere.rs:85-119
template <class T>
Manifold<T> sphere_surface_manifold(const orc_object& o, V3<T> translation, const Ray<T>& ray, T t) {
    bool volumetric = o.volume >= 0;
    V3<T> position = ray_at(ray, t);
    V3<T> normal = (position - translation) / T(o.radius);
    Manifold<T> m;
    if (dot(ray.direction, normal) < T(0)) {
        m.normal = normal;
        m.face = volumetric ? ORC_FACE_VOLUME_FRONT : ORC_FACE_FRONT;
    } else {
        m.normal = -normal;
        m.face = volumetric ? ORC_FACE_VOLUME_BACK : ORC_FACE_BACK;
    }
    m.position = position;
    m.bbox_min = translation - splat<T>(T(o.radius));  // sphere.rs:35-38
    m.bbox_max = translation + splat<T>(T(o.radius));
    m.t = t;
    m.ray = ray;
    m.has_object = true;
    m.object_ref = o.object_ref;
    m.has_mat = true;
    m.mat_ref = o.material;
    m.has_vol = volumetric;
    m.vol_ref = volumetric ? (uint64_t)o.volume : 0;
    return m;
}
// src/scene/object/sphere.rs:121-148
template <class T>
bool sphere_hit(const orc_object& o, const Ray<T>& ray, const Clip<T>& clip, Manifold<T>* out) {
    V3<T> translation = mk<T>(o.transform[9], o.transform[10], o.transform[11]);
    V3<T> oc = ray.origin - translation;
    T half_b = dot(oc, ray.direction);
    T c = length_squared(oc) - T(o.radius) * T(o.radius);
    T discriminant = half_b * half_b - c;
    if (std::signbit(discriminant)) return false;
    T sqrtd = std::sqrt(discriminant);
    T t = -half_b - sqrtd;
    if (t < clip.min || t > clip.max) {
        t = -half_b + sqrtd;
        if (t < clip.min || t > clip.max) return false;
    }
    *out = sphere_surface_manifold(o, translation, ray, t);
    return true;
}
// src/scene/object/sphere.rs:150-166
template <class T>
bool sphere_hit_volumetric(const orc_object& o, const Ray<T>& ray, const Clip<T>& clip, Manifold<T>* out) {
    V3<T> translation = mk<T>(o.transform[9], o.transform[10], o.transform[11]);
    T t = clip.max;
    T dist_sqr = length_squared(ray_at(ray, t) - translation);
    T r_sqr = T(o.radius) * T(o.radius);
    if (dist_sqr <= r_sqr) {
        Manifold<T> m;  // sphere.rs:63-83
        m.position = ray_at(ray, t);
        m.normal = mk<T>(0, 0, 0);
        m.bbox_min = translation - splat<T>(T(o.radius));
        m.bbox_max = translation + splat<T>(T(o.radius));
        m.face = ORC_FACE_VOLUME;
        m.t = t;
        m.ray = ray;
        m.has_object = true;
        m.object_ref = o.object_ref;
        m.has_mat = true;
        m.mat_ref = o.material;
        m.has_vol = o.volume >= 0;
        m.vol_ref = o.volume >= 0 ? (uint64_t)o.volume : 0;
        *out = m;
        return true;
    }
    return sphere_hit(o, ray, clip, out);
}
// src/scene/object/rect.rs:38-56
template <class T>
void rect_bounding_box(const orc_rect& r, const Affine<T>& tf, V3<T>* bmin, V3<T>* bmax) {
    V3<T> x = v3_from<T>(r.x), y = v3_from<T>(r.y);
    T hw = r.half_width, hh = r.half_height;
    V3<T> pts[4] = {
        transform_point(tf, x * hw + y * hh),
        transform_point(tf, x * hw - y * hh),
        transform_point(tf, (-x) * hw + y * hh),
        transform_point(tf, (-x) * hw - y * hh),
    };
    T inf = std::numeric_limits<T>::infinity();
    V3<T> mn = splat<T>(inf), mx = splat<T>(-inf);
    for (int i = 0; i < 4; ++i) {
        mn = vmin(mn, pts[i]);
        mx = vmax(mx, pts[i]);
    }
    *bmin = mn;
    *bmax = mx;
}
// src/scene/object/rect.rs:74-80
template <class T>
bool rect_contains_point(const orc_rect& r, V3<T> point) {
    V3<T> rx = v3_from<T>(r.x), ry = v3_from<T>(r.y);
    V3<T> x = rx * dot(point, rx);  // project_onto_normalized
    V3<T> y = ry * dot(point, ry);
    T w_sqr = T(r.half_width) * T(r.half_width);
    T h_sqr = T(r.half_height) * T(r.half_height);
    return length_squared(x) <= w_sqr && length_squared(y) <= h_sqr;
}
// src/scene/object/rect.rs:110-155
template <class T>
bool rect_hit(const orc_rect& r, uint64_t object_ref, const Affine<T>& tf, const Ray<T>& ray,
              const Clip<T>& clip, Manifold<T>* out) {
    V3<T> translation = tf.translation;
    V3<T> normal = transform_vector(tf, v3_from<T>(r.z));
    T q = dot(ray.direction, normal);
    if (std::fabs(q) <= T(1e-5f)) return false;
    T p = dot(translation - ray.origin, normal);
    T t = p / q;
    if (t < clip.min || t > clip.max) return false;
    V3<T> position = ray_at(ray, t);
    if (!rect_contains_point(r, transform_point(inverse(tf), position))) return false;
    Manifold<T> m;
    if (p < T(0)) {
        m.normal = normal;
        m.face = ORC_FACE_FRONT;
    } else {
        m.normal = -normal;
        m.face = ORC_FACE_BACK;
    }
    m.position = position;
    rect_bounding_box(r, tf, &m.bbox_min, &m.bbox_max);
    m.t = t;
    m.ray = ray;
    m.has_object = true;
    m.object_ref = object_ref;
    m.has_mat = true;
    m.mat_ref = r.material;
    m.has_vol = false;
    m.vol_ref = 0;
    *out = m;
    return true;
}
// src/scene/object/cuboid.rs:83-105  (strict '<' against clip.max)
template <class T>
bool cuboid_hit(const orc_object& o, const Affine<T>& tf, const Ray<T>& ray, const Clip<T>& clip,
                Manifold<T>* out, int* face_index = 0) {
    T t = clip.max;
    bool found = false;
    for (int i = 0; i < 6; ++i) {
        Affine<T> ftf = mul_translation(tf, v3_from<T>(o.face_offset[i]));
        Manifold<T> m;
        if (rect_hit(o.faces[i], o.object_ref, ftf, ray, clip, &m)) {
            if (m.t < t) {
                t = m.t;
                *out = m;
                found = true;
                if (face_index) *face_index = i;
            }
        }
    }
    return found;
}
// src/scene/object/mod.rs:168-180
template <class T>
bool object_hit(const orc_object& o, const Ray<T>& ray, const Clip<T>& clip, Manifold<T>* out) {
    switch (o.kind) {
        case ORC_SPHERE: return sphere_hit(o, ray, clip, out);
        case ORC_RECT: return rect_hit(o.rect, o.object_ref, affine_from<T>(o.transform), ray, clip, out);
        case ORC_CUBOID: return cuboid_hit(o, affine_from<T>(o.transform), ray, clip, out);
        default: return false;
    }
}
// src/scene/object/mod.rs:182-198
template <class T>
bool object_hit_volumetric(const orc_object& o, const Ray<T>& ray, const Clip<T>& clip, Manifold<T>* out) {
    if (o.kind == ORC_SPHERE) return sphere_hit_volumetric(o, ray, clip, out);
    return false;
}
// src/scene/object/mod.rs:154-166; sphere.rs:44-61; rect.rs:92-108; cuboid.rs:56-81
bool object_pdf(const orc_object& o, const Rayf& ray, const Clip<float>& clip, float* pdf_out) {
    Manifold<float> m;
    switch (o.kind) {
        case ORC_SPHERE: {
            if (!sphere_hit(o, ray, clip, &m)) return false;
            float r = o.radius;
            float shadow = 3.14159265358979323846f * r * r;
            float dist_sqr = m.t * m.t;
            *pdf_out = dist_sqr / shadow;
            return true;
        }
        case ORC_RECT: {
            if (!rect_hit(o.rect, o.object_ref, affine_from<float>(o.transform), ray, clip, &m)) return false;
            float area = 4.0f * o.rect.half_width * o.rect.half_height;
            float shadow = area * std::fabs(dot(ray.direction, m.normal));
            *pdf_out = (m.t * m.t) / shadow;
            return true;
        }
        case ORC_CUBOID: {
            int face = -1;
            Affine<float> tf = affine_from<float>(o.transform);
            if (!cuboid_hit(o, tf, ray, clip, &m, &face)) return false;
            // cuboid.rs:77-80: rect.pdf on the selected face (re-hit with the same clip)
            Affine<float> ftf = mul_translation(tf, v3_from<float>(o.face_offset[face]));
            if (!rect_hit(o.faces[face], o.object_ref, ftf, ray, clip, &m)) return false;
            const orc_rect& r = o.faces[face];
            float area = 4.0f * r.half_width * r.half_height;
            float shadow = area * std::fabs(dot(ray.direction, m.normal));
            *pdf_out = (m.t * m.t) / shadow;
            return true;
        }
        default: return false;
    }
}
// rect.rs:82-86
V3f rect_random_point(const orc_rect& r, Rng& rng, const Affine<float>& tf) {
    float x = UniformF32::make_inclusive(-r.half_width, r.half_width).sample(rng);
    float y = UniformF32::make_inclusive(-r.half_height, r.half_height).sample(rng);
    return transform_point(tf, v3_from<float>(r.x) * x + v3_from<float>(r.y) * y);
}
// src/scene/object/mod.rs:145-152; sphere.rs:40-42; cuboid.rs:48-54
V3f object_random_point(const orc_object& o, Rng& rng) {
    V3f translation = mk<float>(o.transform[9], o.transform[10], o.transform[11]);
    switch (o.kind) {
        case ORC_SPHERE: return translation + unit_sphere(rng) * o.radius;
        case ORC_RECT: return rect_random_point(o.rect, rng, affine_from<float>(o.transform));
        case ORC_CUBOID: {
            // [rand] WeightedIndex<f32>: cumulative sums without the last weight, Uniform::new(0,total)
            float cumulative[5];
            float total = 4.0f * o.faces[0].half_width * o.faces[0].half_height;
            for (int i = 1; i < 6; ++i) {
                cumulative[i - 1] = total;
                total += 4.0f * o.faces[i].half_width * o.faces[i].half_height;
            }
            if (!(total > 0.0f)) throw Panic("called `Result::unwrap()` on an `Err` value: AllWeightsZero");
            float chosen = UniformF32::make(0.0f, total).sample(rng);
            int index = 0;
            while (index < 5 && cumulative[index] <= chosen) ++index;
            Affine<float> tf = mul_translation(affine_from<float>(o.transform), v3_from<float>(o.face_offset[index]));
            return rect_random_point(o.faces[index], rng, tf);
        }
        default: return translation;
    }
}

// ------------------------------------------------------------------------------------------
// volume  (src/scene/data/volume.rs)
// ------------------------------------------------------------------------------------------
float density_index(const Data& v, int x, int y, int z) {  // volume.rs:119-134
    if (v.d.width == 0 || v.d.height == 0 || v.d.depth == 0) return 0.0f;
    size_t ux = (size_t)(int64_t)x, uy = (size_t)(int64_t)y, uz = (size_t)(int64_t)z;
    if (!(ux < v.d.width) || !(uy < v.d.height) || !(uz < v.d.depth)) throw Panic("volume index out of bounds");
    return v.buffer[uz * v.d.height * v.d.width + uy * v.d.width + ux];
}
inline int f2i_sat(float x) {  // Rust `as i32`: saturating, NaN -> 0
    if (x != x) return 0;
    if (x >= 2147483648.0f) return INT32_MAX;
    if (x <= -2147483648.0f) return INT32_MIN;
    return (int)x;
}
inline float sample_xyz(const Data& v, float x, float y, float z) {
    return density_index(v, f2i_sat(x), f2i_sat(y), f2i_sat(z));
}
inline float fract(float x) { return x - std::trunc(x); }
float density_trilinear(const Data& v, V3f coord) {  // volume.rs:140-167
    coord = vmin(vmax(coord, splat<float>(0.0f)), splat<float>(1.0f));
    V3f ic = coord * mk<float>(v.d.size[0], v.d.size[1], v.d.size[2]);
    float fx = std::floor(ic.x), cx = std::ceil(ic.x);
    float fy = std::floor(ic.y), cy = std::ceil(ic.y);
    float fz = std::floor(ic.z), cz = std::ceil(ic.z);
    float x0 = sample_xyz(v, fx, fy, fz);
    float x1 = sample_xyz(v, cx, fy, fz);
    float y0 = lerp(x0, x1, fract(ic.x));
    x0 = sample_xyz(v, fx, cy, fz);
    x1 = sample_xyz(v, cx, cy, fz);
    float y1 = lerp(x0, x1, fract(ic.x));
    float z0 = lerp(y0, y1, fract(ic.y));
    x0 = sample_xyz(v, fx, fy, cz);
    x1 = sample_xyz(v, cx, fy, cz);
    y0 = lerp(x0, x1, fract(ic.x));
    x0 = sample_xyz(v, fx, cy, cz);
    x1 = sample_xyz(v, cx, cy, cz);
    y1 = lerp(x0, x1, fract(ic.x));
    float z1 = lerp(y0, y1, fract(ic.y));
    return lerp(z0, z1, fract(ic.z));
}

// ------------------------------------------------------------------------------------------
// lens field + geodesic segments (NOT in the reference; DESIGN.md "Geodesic model")
// ------------------------------------------------------------------------------------------
template <class T> inline T fma_t(T a, T b, T c) { return std::fma(a, b, c); }
// the stepper's 1/sqrt: correctly rounded (f32: via f64, exact up to 2^-29-probability double
// rounding).  The device's BT_LENS_EXACT_RSQRT mode (__frsqrt_rn) computes the same value; its
// default mode uses MUFU.RSQ (<= 2 ulp).
inline float rsqrt_t(float x) { return (float)(1.0 / std::sqrt((double)x)); }
inline double rsqrt_t(double x) { return 1.0 / std::sqrt(x); }

template <class T>
struct LensT {
    T cx, cy, cz, rs, k /* -1.5 rs */, far_r /* r_far * rs */;
};
template <class T>
struct Field {
    std::vector<LensT<T> > l;
    T kappa, h_min, h_max;
    uint32_t max_steps;
};
template <class T>
Field<T> make_field(const float* xyzr, int n, const orc_lens_config& cfg) {
    Field<T> f;
    for (int i = 0; i < n; ++i) {
        float rs = xyzr[4 * i + 3];
        if (!(rs > 0.0f)) continue;  // r_s <= 0: no mass (exact flat limit)
        LensT<T> l;
        l.cx = xyzr[4 * i];
        l.cy = xyzr[4 * i + 1];
        l.cz = xyzr[4 * i + 2];
        l.rs = rs;
        l.k = T(-1.5) * T(rs);
        l.far_r = T(cfg.r_far) * T(rs);
        f.l.push_back(l);
    }
    f.kappa = cfg.kappa;
    f.h_min = cfg.h_min;
    f.h_max = cfg.h_max;
    f.max_steps = cfg.max_steps;
    return f;
}
struct AccelInfo {
    bool captured, far;
};
// a = sum_m -(3/2) rs |d x v|^2 d / |d|^5, written with the explicit FMA placement the device
// stepper uses.  With info != 0 also returns min_m |d| and the capture / far-field flags.
template <class T>
inline V3<T> accel(const Field<T>& f, V3<T> x, bool staged, T a, V3<T> w, V3<T> v, T* rmin_out, AccelInfo* info) {
    T ax = 0, ay = 0, az = 0;
    T rmin = std::numeric_limits<T>::infinity();
    bool captured = false, far = true;
    for (size_t m = 0; m < f.l.size(); ++m) {
        const LensT<T>& l = f.l[m];
        // evaluated at x + a*w as d = fma(a, w, x - c): the stage offset is applied after the subtraction
        T dx = x.x - l.cx, dy = x.y - l.cy, dz = x.z - l.cz;
        if (staged) {
            dx = fma_t(a, w.x, dx);
            dy = fma_t(a, w.y, dy);
            dz = fma_t(a, w.z, dz);
        }
        T r2 = fma_t(dz, dz, fma_t(dy, dy, dx * dx));
        T lx = fma_t(dy, v.z, -(dz * v.y));
        T ly = fma_t(dz, v.x, -(dx * v.z));
        T lz = fma_t(dx, v.y, -(dy * v.x));
        T h2 = fma_t(lz, lz, fma_t(ly, ly, lx * lx));
        T inv = rsqrt_t(r2);
        T inv2 = inv * inv;
        T inv5 = (inv2 * inv2) * inv;
        T s = (l.k * h2) * inv5;
        ax = fma_t(s, dx, ax);
        ay = fma_t(s, dy, ay);
        az = fma_t(s, dz, az);
        if (info) {
            T r = r2 * inv;
            if (r < l.rs) captured = true;
            rmin = std::min(rmin, r);
            T dv = fma_t(dz, v.z, fma_t(dy, v.y, dx * v.x));
            if (!(r > l.far_r && dv > T(0))) far = false;
        }
    }
    if (info) {
        info->captured = captured;
        info->far = far;
        *rmin_out = rmin;
    }
    return mk<T>(ax, ay, az);
}
template <class T> inline V3<T> axpy(T a, V3<T> x, V3<T> y) {
    return mk<T>(fma_t(a, x.x, y.x), fma_t(a, x.y, y.y), fma_t(a, x.z, y.z));
}
// classic RK4 given k1 = accel(x, v)
template <class T>
inline void rk4_from_k1(const Field<T>& f, V3<T>& x, V3<T>& v, V3<T> k1, T h) {
    T hh = T(0.5) * h, h6 = h * T(1.0 / 6.0);
    V3<T> v2 = axpy(hh, k1, v);
    V3<T> k2 = accel<T>(f, x, true, hh, v, v2, 0, 0);
    V3<T> v3 = axpy(hh, k2, v);
    V3<T> k3 = accel<T>(f, x, true, hh, v2, v3, 0, 0);
    V3<T> v4 = axpy(h, k3, v);
    V3<T> k4 = accel<T>(f, x, true, h, v3, v4, 0, 0);
    V3<T> sv = axpy(T(2), v2 + v3, v + v4);
    V3<T> sk = axpy(T(2), k2 + k3, k1 + k4);
    x = axpy(h6, sv, x);
    v = axpy(h6, sk, v);
}
template <class T> inline T step_size(const Field<T>& f, T rmin) {
    return std::min(std::max(f.kappa * rmin, f.h_min), f.h_max);
}

// reference try_hit with an explicit clip (src/tracer/mod.rs:389-402)
template <class T>
bool try_hit_clip(const Scene& scene, const Ray<T>& ray, Clip<T> clip, Manifold<T>* out) {
    bool found = false;
    for (size_t i = 0; i < scene.objects.size(); ++i) {
        Manifold<T> m;
        if (object_hit(scene.objects[i], ray, clip, &m)) {
            clip.max = m.t;
            *out = m;
            found = true;
        }
    }
    return found;
}

enum { SEG_HIT = 0, SEG_ESCAPED = 1, SEG_CAPTURED = 2 };
template <class T>
struct Segment {
    int status;
    uint32_t steps;
    Manifold<T> manifold;  // SEG_HIT; manifold.t = accumulated chord length
    Ray<T> escape;         // SEG_ESCAPED: last position + unit direction
};
template <class T> inline V3<T> normalize_fma(V3<T> a, T* len_out) {
    T l2 = fma_t(a.z, a.z, fma_t(a.y, a.y, a.x * a.x));
    T inv = T(1) / std::sqrt(l2);
    if (len_out) *len_out = l2 * inv;
    return a * inv;
}
// one "ray" of the render loop = a chain of chords through the lens field
template <class T>
Segment<T> trace_segment(const Scene& scene, const Field<T>& f, const Ray<T>& ray, T clip_min, T clip_max) {
    Segment<T> seg;
    seg.steps = 0;
    if (f.l.empty()) {  // flat field: exactly the reference
        Clip<T> clip = {clip_min, clip_max};
        if (try_hit_clip(scene, ray, clip, &seg.manifold)) {
            seg.status = SEG_HIT;
        } else {
            seg.status = SEG_ESCAPED;
            seg.escape = ray;
        }
        return seg;
    }
    V3<T> x = ray.origin, v = ray.direction;
    T travelled = 0;
    for (;;) {
        T rmin;
        AccelInfo info;
        V3<T> k1 = accel<T>(f, x, false, T(0), v, v, &rmin, &info);
        if (info.captured) {
            seg.status = SEG_CAPTURED;
            return seg;
        }
        T remaining = clip_max - travelled;
        Clip<T> clip;
        clip.min = std::max(clip_min - travelled, T(0));
        if (info.far) {
            Ray<T> chord = {x, normalize_fma<T>(v, 0)};
            clip.max = remaining;
            if (try_hit_clip(scene, chord, clip, &seg.manifold)) {
                seg.status = SEG_HIT;
                seg.manifold.t = travelled + seg.manifold.t;
            } else {
                seg.status = SEG_ESCAPED;
                seg.escape = chord;
            }
            return seg;
        }
        T h = step_size(f, rmin);
        V3<T> x1 = x, v1 = v;
        rk4_from_k1(f, x1, v1, k1, h);
        T len;
        Ray<T> chord = {x, normalize_fma<T>(x1 - x, &len)};
        clip.max = std::min(len, remaining);
        if (try_hit_clip(scene, chord, clip, &seg.manifold)) {
            seg.status = SEG_HIT;
            seg.manifold.t = travelled + seg.manifold.t;
            return seg;
        }
        travelled += len;
        x = x1;
        v = v1;
        seg.steps++;
        if (travelled >= clip_max || seg.steps >= f.max_steps) {
            seg.status = SEG_ESCAPED;
            seg.escape.origin = x;
            seg.escape.direction = normalize_fma<T>(v, 0);
            return seg;
        }
    }
}

// ------------------------------------------------------------------------------------------
// environment map + equirectangular camera (NOT in the reference; DESIGN.md §3.5, §3.6)
// ------------------------------------------------------------------------------------------
// Earlier revisions' test layers #include this file and define sincos_poly, equirect_dir and
// orc_env_lookup themselves: the names here differ so that their tests still build against it.
// The lookup of device.cuh (env_lookup), operation for operation: every product and sum rounded
// on its own (-ffp-contract=off), atan2 / sqrt from libm.  Any d, NaN included, reads a texel.
V3f env_lookup(const float* rgb, uint32_t w, uint32_t h, V3f d) {
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

// device.cuh's sincos_poly, operation for operation: Cody-Waite reduction by pi/2 and the Cephes polynomials in explicit FMAs
void panorama_sincos(float x, float* sn, float* cs) {
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

// device.cuh camera_ray's equirectangular branch, operation for operation: the camera-space
// direction for the jittered NDC (u, v) before the half-pixel offset
V3f panorama_dir(float u, float v, float pixel_width, float pixel_height) {
    const float phi = 3.14159274101257324f * (u + pixel_width * 0.5f);
    const float theta = -1.57079637050628662f * (v + pixel_height * 0.5f);
    float sp, cp, st, ct;
    panorama_sincos(phi, &sp, &cp);
    panorama_sincos(theta, &st, &ct);
    return mk<float>(ct * sp, st, -(ct * cp));
}

// ------------------------------------------------------------------------------------------
// tracer  (src/tracer/mod.rs)
// ------------------------------------------------------------------------------------------
struct ChunkConfig {  // mod.rs:205-230
    int output;
    uint32_t subsample;
    uint64_t samples, max_bounces, max_volume_bounces;
    float clip_min, clip_max, volume_step;
    static ChunkConfig with_configs(const orc_config& c) {
        ChunkConfig k;
        k.output = c.has_output ? c.r_output : c.output;
        k.subsample = c.subsample;
        k.samples = c.samples;
        k.max_bounces = c.has_max_bounces ? c.r_max_bounces : c.max_bounces;
        // mod.rs:224 -- reads render.max_bounces, not render.max_volume_bounces (preserved)
        k.max_volume_bounces = c.has_max_bounces ? c.r_max_bounces : c.max_volume_bounces;
        k.clip_min = c.clip_min;
        k.clip_max = c.clip_max;
        k.volume_step = c.has_volume_step ? c.r_volume_step : c.volume_step;
        return k;
    }
};

struct ShaderData {  // material.rs:15-20
    bool has_scatter;
    Rayf scatter;
    bool has_albedo;
    ColorData albedo;
    float pdf;
};

struct ChunkState {
    ChunkConfig config;
    Rng rng;
    const Scene* scene;
    Field<float> field;

    Clip<float> clip() const {
        Clip<float> c = {config.clip_min, config.clip_max};
        return c;
    }

    // material.rs:71-79
    V3f emitted(const orc_data& m) const {
        switch (m.mat_kind) {
            case ORC_FLAT: return v3_from<float>(m.albedo);
            case ORC_EMISSIVE: return v3_from<float>(m.albedo) * m.intensity;
            default: return mk<float>(0, 0, 0);
        }
    }
    // material.rs:201-210, 301-311
    float material_pdf(const orc_data& m, const Manifold<float>& manifold, const Rayf& ray) const {
        if (m.mat_kind == ORC_DIFFUSE) return dot(manifold.normal, ray.direction) * 0.318309886183790671538f;
        return 1.0f;
    }
    // Pdf::scatter, material.rs:222-277
    Rayf scatter_diffuse(const Manifold<float>& m) {
        Basis b(m.normal);
        return ray_new(m.position, cosine(rng, b));
    }
    Rayf scatter_metallic(const Manifold<float>& m, float roughness) {
        Basis b(m.normal);
        V3f direction = reflect(m.ray.direction, m.normal);
        V3f fuzz = unit_hemisphere(rng, b) * roughness;
        return ray_new(m.position, direction + fuzz);
    }
    Rayf scatter_glass(const Manifold<float>& m, float roughness, float ior) {
        Basis b(m.normal);
        bool front = m.face == ORC_FACE_FRONT || m.face == ORC_FACE_VOLUME_FRONT;
        if (front) ior = 1.0f / ior;
        float cos_theta = std::min(dot(-m.ray.direction, m.normal), 1.0f);
        float sin_theta = std::sqrt(1.0f - cos_theta * cos_theta);
        float fr = fresnel(m.ray.direction, m.normal, ior);
        V3f direction;
        if (ior * sin_theta > 1.0f || gen_bool(rng, (double)fr))
            direction = reflect(m.ray.direction, m.normal);
        else
            direction = refract(m.ray.direction, m.normal, ior);
        V3f fuzz = unit_hemisphere(rng, b) * roughness;
        return ray_new(m.position, direction + fuzz);
    }
    Rayf scatter_light(const Manifold<float>& m, const orc_object& light) {
        V3f direction = object_random_point(light, rng) - m.position;
        return ray_new(m.position, direction);
    }
    static bool pdf_some(float p) { return !(std::fabs(p - 0.0f) <= 1e-5f); }  // approx abs_diff_eq

    // Material::shade, material.rs:81-199
    ShaderData shade(const orc_data& mat, const Manifold<float>& manifold, const Clip<float>& clip) {
        ShaderData sd;
        sd.has_scatter = false;
        sd.pdf = 1.0f;
        ColorData cd;
        cd.normal = manifold.normal;
        cd.depth = manifold.t;
        switch (mat.mat_kind) {
            case ORC_FLAT:
                sd.has_albedo = true;
                sd.albedo = cd;  // colour and albedo BLACK
                return sd;
            case ORC_EMISSIVE:
                sd.has_albedo = false;
                return sd;
            default: break;
        }
        cd.color = v3_from<float>(mat.albedo);
        cd.albedo = cd.color;
        sd.has_albedo = true;
        sd.albedo = cd;
        Rayf ray;
        float p;
        if (mat.mat_kind == ORC_DIFFUSE) {
            uint64_t count = 0;
            for (size_t i = 0; i < scene->objects.size(); ++i)
                if (scene->objects[i].flags & 1u) ++count;
            uint64_t index = uniform_usize(rng, count);
            const orc_object* light = 0;
            for (size_t i = 0; i < scene->objects.size(); ++i)
                if (scene->objects[i].flags & 1u) {
                    if (index == 0) {
                        light = &scene->objects[i];
                        break;
                    }
                    --index;
                }
            // Pdf::Mix(Diffuse, Light, 0.5): true selects b = the light (material.rs:269-275)
            if (gen_bool(rng, (double)0.5f))
                ray = scatter_light(manifold, *light);
            else
                ray = scatter_diffuse(manifold);
            float pa = dot(manifold.normal, ray.direction) * 0.318309886183790671538f;
            float pb = 0.0f;
            if (!object_pdf(*light, ray, clip, &pb)) pb = 0.0f;  // light_pdf, material.rs:313-316
            p = lerp(pa, pb, 0.5f);
        } else if (mat.mat_kind == ORC_METALLIC) {
            ray = scatter_metallic(manifold, mat.roughness);
            p = 1.0f;
        } else {
            ray = scatter_glass(manifold, mat.roughness, mat.ior);
            p = 1.0f;
        }
        if (pdf_some(p)) {
            sd.has_scatter = true;
            sd.scatter = ray;
            sd.pdf = p;
        }
        return sd;
    }

    // mod.rs:389-402
    bool try_hit(const Rayf& ray, Manifold<float>* out) { return try_hit_clip(*scene, ray, clip(), out); }
    // mod.rs:404-427
    bool try_hit_volume(const Rayf& ray, uint64_t last_object, Manifold<float>* out) {
        bool found = false;
        Clip<float> c = {0.0f, config.volume_step};
        for (size_t i = 0; i < scene->objects.size(); ++i) {
            const orc_object& o = scene->objects[i];
            Manifold<float> m;
            bool hit = (o.object_ref == last_object) ? object_hit_volumetric(o, ray, c, &m) : object_hit(o, ray, c, &m);
            if (hit) {
                c.max = m.t;
                *out = m;
                found = true;
            }
        }
        return found;
    }

    // mod.rs:429-452 (+ the environment map's factor in the escape direction when the scene has a map)
    ColorData sample_root(const Rayf& ray) {
        const Data& d = scene->get_material(scene->root_material, "expected root material to be a material");
        Manifold<float> manifold;
        manifold.position = ray_at(ray, config.clip_max);
        manifold.normal = -ray.direction;
        manifold.bbox_min = splat<float>(-std::numeric_limits<float>::infinity());
        manifold.bbox_max = splat<float>(std::numeric_limits<float>::infinity());
        manifold.face = ORC_FACE_VOLUME;
        manifold.t = config.clip_max;
        manifold.ray = ray;
        manifold.has_object = manifold.has_mat = manifold.has_vol = false;
        manifold.object_ref = manifold.mat_ref = manifold.vol_ref = 0;
        V3f e = emitted(d.d);
        ShaderData data = shade(d.d, manifold, clip());
        ColorData cd = data.has_albedo ? data.albedo : ColorData();
        cd.color = cd.color + e;
        if (scene->env_w != 0) cd.color = cd.color * env_lookup(scene->env_rgb.data(), scene->env_w, scene->env_h, ray.direction);
        return cd;
    }

    // mod.rs:454-486
    ColorData sample_surface(const Manifold<float>& manifold, uint64_t mat_ref, uint64_t bounce) {
        const Data& d = scene->get_material(mat_ref, "expected material data");
        V3f e = emitted(d.d);
        ShaderData data = shade(d.d, manifold, clip());
        if (data.has_scatter) {
            ColorData reflected = sample(data.scatter, bounce + 1);
            ColorData cd;
            if (data.has_albedo) {
                cd = data.albedo;
                cd.color = cd.color * material_pdf(d.d, manifold, data.scatter);
                cd.color = cd.color * (reflected.color / data.pdf);
            } else {
                cd = reflected;
            }
            cd.color = cd.color + e;
            return cd;
        }
        return ColorData::from_emitted(e);
    }

    // Volume::shade, volume.rs:26-60
    void volume_shade(const Data& vol, const Manifold<float>& manifold, float step, Rayf* ray_out,
                      bool* has_atten, ColorData* atten) {
        V3f offset = manifold.bbox_min;
        V3f size = manifold.bbox_max - manifold.bbox_min;
        V3f coord = (manifold.position - offset) / size;
        float density = step * density_trilinear(vol, coord);
        if (density >= 1.0f || gen_bool(rng, (double)density)) {
            V3f origin = manifold.position;
            if (manifold.face == ORC_FACE_VOLUME)
                origin = origin - manifold.ray.direction * step * standard_f32(rng);
            V3f direction = unit_sphere(rng);
            *ray_out = ray_new(origin, direction);
            ColorData cd;
            cd.color = splat<float>(0.8f);
            cd.albedo = splat<float>(0.8f);
            cd.normal = manifold.normal;
            cd.depth = manifold.t;
            *has_atten = true;
            *atten = cd;
        } else {
            *ray_out = ray_new(manifold.position, manifold.ray.direction);
            *has_atten = false;
        }
    }

    // mod.rs:488-523
    ColorData sample_volume(const Manifold<float>& manifold, uint64_t vol_ref, uint64_t bounce, uint64_t volume_bounce) {
        const Data& d = scene->get_data(vol_ref);
        if (d.d.kind != 1) throw Panic("expected volume data");
        Rayf ray;
        bool has_atten;
        ColorData atten;
        volume_shade(d, manifold, config.volume_step, &ray, &has_atten, &atten);
        ColorData reflected;
        if (manifold.face == ORC_FACE_VOLUME_BACK)
            reflected = sample(ray, bounce + 1);
        else
            reflected = sample_volumetric(ray, manifold.object_ref, bounce, volume_bounce + 1);
        if (has_atten) {
            atten.color = atten.color * reflected.color;
            return atten;
        }
        return reflected;
    }

    ColorData dispatch(const Manifold<float>& m, uint64_t bounce, uint64_t volume_bounce) {
        bool surface = m.face == ORC_FACE_FRONT || m.face == ORC_FACE_BACK;
        if (surface) {
            if (m.has_mat) return sample_surface(m, m.mat_ref, bounce);
            return ColorData();
        }
        if (m.has_vol) return sample_volume(m, m.vol_ref, bounce, volume_bounce);
        return ColorData();
    }

    // mod.rs:322-342 (+ geodesic segments when a lens field is present)
    ColorData sample(const Rayf& ray, uint64_t bounce) {
        if (bounce > config.max_bounces) return ColorData();
        if (field.l.empty()) {
            Manifold<float> m;
            if (try_hit(ray, &m)) return dispatch(m, bounce, 0);
            return sample_root(ray);
        }
        Segment<float> seg = trace_segment<float>(*scene, field, ray, config.clip_min, config.clip_max);
        if (seg.status == SEG_HIT) return dispatch(seg.manifold, bounce, 0);
        if (seg.status == SEG_CAPTURED) return ColorData();
        return sample_root(seg.escape);
    }

    // mod.rs:344-373
    ColorData sample_volumetric(const Rayf& ray, uint64_t last_object, uint64_t bounce, uint64_t volume_bounce) {
        if (volume_bounce > config.max_volume_bounces) return ColorData();
        Manifold<float> m;
        if (try_hit_volume(ray, last_object, &m)) return dispatch(m, bounce, volume_bounce);
        return sample_root(ray);
    }
};

// [glam] Quat::from_euler(YXZ, yrot, xrot, 0) * NEG_Z   (src/tracer/ray.rs:103-113)
V3f with_frustum_dir(float yfov, float xfov, float u, float v) {
    float yrot = xfov * 0.5f * -u;
    float xrot = yfov * 0.5f * -v;
    float sy = std::sin(yrot * 0.5f), cy = std::cos(yrot * 0.5f);
    float sx = std::sin(xrot * 0.5f), cx = std::cos(xrot * 0.5f);
    // rot_y(yrot) * rot_x(xrot) * rot_z(0); every component is a single product
    float qx = cy * sx, qy = sy * cx, qz = -(sy * sx), qw = cy * cx;
    // Quat * Vec3A: v*(w*w - b.b) + b*(2*(v.b)) + (b x v)*(2w), v = (0,0,-1)
    V3f b = mk<float>(qx, qy, qz);
    V3f vv = mk<float>(0.0f, 0.0f, -1.0f);
    float b2 = dot(b, b);
    float s1 = qw * qw - b2;
    float s2 = dot(vv, b) * 2.0f;
    float s3 = qw * 2.0f;
    return vv * s1 + b * s2 + cross(b, vv) * s3;
}

struct CameraSetup {
    const orc_object* cam_obj;
    Affine<float> tf;
    float yfov, xfov, pixel_width, pixel_height;
    UniformF32 scatter_u, scatter_v;
    Basis defocus_basis;
    uint32_t sub_n;  // 1 for Subsample::None
    float sub_width;
    int projection;  // ORC_PROJECTION_*
    CameraSetup() : defocus_basis(mk<float>(0.0f, 0.0f, -1.0f)) {}
};

// mod.rs:244-267
CameraSetup camera_setup(const Scene& scene, uint64_t camera_ref, const ChunkConfig& cfg, uint32_t width, uint32_t height) {
    CameraSetup cs;
    const orc_object& o = scene.get_object(camera_ref);
    if (o.kind != ORC_CAMERA) throw Panic("expected a camera object");
    cs.cam_obj = &o;
    cs.tf = affine_from<float>(o.transform);
    cs.yfov = 2.0f * std::atan2(o.sensor_size, 2.0f * o.focal_length);
    cs.xfov = cs.yfov * o.aspect_ratio;
    cs.pixel_width = 2.0f * (1.0f / (float)width);    // buffer.rs:68-76
    cs.pixel_height = 2.0f * (1.0f / (float)height);
    float subpixel_scale = cfg.subsample == 0 ? 1.0f : 1.0f / (float)cfg.subsample;
    cs.scatter_u = UniformF32::make(-0.5f * cs.pixel_width * subpixel_scale, 0.5f * cs.pixel_width * subpixel_scale);
    cs.scatter_v = UniformF32::make(-0.5f * cs.pixel_height * subpixel_scale, 0.5f * cs.pixel_height * subpixel_scale);
    cs.sub_n = cfg.subsample == 0 ? 1 : cfg.subsample;
    cs.sub_width = cfg.subsample == 0 ? 0.0f : 1.0f / (float)cfg.subsample;
    std::map<uint64_t, int>::const_iterator p = scene.projection.find(camera_ref);
    cs.projection = p == scene.projection.end() ? ORC_PROJECTION_PERSPECTIVE : p->second;
    return cs;
}

// mod.rs:272-302: one camera ray; draws jitter-u, jitter-v, [disk angle, disk radius].
// The equirectangular camera forms (u, v) the same way and is a pinhole: no disk draws.
Rayf camera_ray(const CameraSetup& cs, Rng& rng, uint32_t x, uint32_t y, uint32_t sub_index) {
    float v = (float)y * cs.pixel_height - 1.0f;
    float u = (float)x * cs.pixel_width - 1.0f;
    float u_sub = 0.0f, v_sub = 0.0f;
    if (cs.sub_width != 0.0f) {  // mod.rs:96-101
        uint32_t i = sub_index % cs.sub_n, j = sub_index / cs.sub_n;
        u_sub = (float)i * cs.sub_width;
        v_sub = (float)j * cs.sub_width;
    }
    float u_offset = u_sub * cs.pixel_width + cs.scatter_u.sample(rng);
    float v_offset = v_sub * cs.pixel_height + cs.scatter_v.sample(rng);
    u = u + u_offset;
    v = v + v_offset;
    if (cs.projection == ORC_PROJECTION_EQUIRECTANGULAR) {
        const V3f dir_cam = panorama_dir(u, v, cs.pixel_width, cs.pixel_height);
        V3f origin = cs.tf.translation + mk<float>(0, 0, 0);  // Affine3A * Ray, ray.rs:126-137
        V3f direction = normalize_or_zero_s(transform_vector(cs.tf, dir_cam));
        return ray_new(origin, direction);
    }
    Rayf ray;
    ray.origin = mk<float>(0, 0, 0);
    ray.direction = with_frustum_dir(cs.yfov, cs.xfov, u, v);
    const orc_object& cam = *cs.cam_obj;
    // Affine3A * Ray, ray.rs:126-137
    V3f origin = cs.tf.translation + ray.origin;
    V3f direction = normalize_or_zero_s(transform_vector(cs.tf, ray.direction));
    if (cam.has_focus) {
        V3f defocus = unit_disk(rng, cs.defocus_basis);
        float aperture = 0.5f * cam.focal_length / cam.fstop;
        V3f defocus_offset = transform_vector(cs.tf, defocus * aperture);
        float frac_f_z = cam.focus / std::fabs(ray.direction.z);
        Rayf r = ray_new(origin, direction);
        r.origin = r.origin + defocus_offset;
        r.direction = normalize_a(r.direction * frac_f_z - defocus_offset);
        return r;
    }
    return ray_new(origin, direction);
}

}  // namespace

// ==========================================================================================
// C interface
// ==========================================================================================
extern "C" {

const char* orc_last_error(void) {
    if (g_last_error.empty()) g_last_error = g_last_error_shared;
    return g_last_error.c_str();
}

void* orc_scene_create(const orc_object* objects, int n_objects, const orc_data* data, int n_data,
                       uint64_t root_material) {
    Scene* s = new Scene();
    s->objects.assign(objects, objects + n_objects);
    std::sort(s->objects.begin(), s->objects.end(),
              [](const orc_object& a, const orc_object& b) { return a.object_ref < b.object_ref; });
    for (size_t i = 0; i < s->objects.size(); ++i) s->object_index[s->objects[i].object_ref] = (int)i;
    for (int i = 0; i < n_data; ++i) {
        Data d;
        d.d = data[i];
        if (data[i].kind == 1 && data[i].buffer) {
            size_t n = (size_t)data[i].width * data[i].height * data[i].depth;
            d.buffer.assign(data[i].buffer, data[i].buffer + n);
        }
        d.d.buffer = 0;
        s->data[data[i].data_ref] = d;
    }
    s->root_material = root_material;
    std::memset(&s->lens_cfg, 0, sizeof(s->lens_cfg));
    return s;
}

void orc_scene_set_lenses(void* scene, const float* xyzr, int n, const orc_lens_config* cfg) {
    Scene* s = (Scene*)scene;
    s->lenses.clear();
    for (int i = 0; i < n; ++i) {
        Lens l = {{xyzr[4 * i], xyzr[4 * i + 1], xyzr[4 * i + 2]}, xyzr[4 * i + 3]};
        s->lenses.push_back(l);
    }
    if (cfg) s->lens_cfg = *cfg;
}

int orc_scene_set_camera_aspect(void* scene, uint64_t camera_ref, float aspect) {
    Scene* s = (Scene*)scene;
    std::map<uint64_t, int>::iterator it = s->object_index.find(camera_ref);
    if (it == s->object_index.end() || s->objects[it->second].kind != ORC_CAMERA) {
        g_last_error = g_last_error_shared = "expected a camera object";
        return -1;
    }
    s->objects[it->second].aspect_ratio = aspect;
    return 0;
}

int orc_scene_set_environment(void* scene, const float* rgb, uint32_t width, uint32_t height) {
    Scene* s = (Scene*)scene;
    if (!rgb || width == 0 || height == 0) {
        s->env_rgb.clear();
        s->env_w = s->env_h = 0;
        return 0;
    }
    s->env_rgb.assign(rgb, rgb + (size_t)width * height * 3);
    s->env_w = width;
    s->env_h = height;
    return 0;
}

int orc_scene_set_camera_projection(void* scene, uint64_t camera_ref, int projection) {
    Scene* s = (Scene*)scene;
    std::map<uint64_t, int>::iterator it = s->object_index.find(camera_ref);
    if (it == s->object_index.end() || s->objects[it->second].kind != ORC_CAMERA) {
        g_last_error = g_last_error_shared = "expected a camera object";
        return -1;
    }
    if (projection != ORC_PROJECTION_PERSPECTIVE && projection != ORC_PROJECTION_EQUIRECTANGULAR) {
        g_last_error = g_last_error_shared = "unknown projection";
        return -1;
    }
    if (projection == ORC_PROJECTION_PERSPECTIVE) s->projection.erase(camera_ref);
    else s->projection[camera_ref] = projection;
    return 0;
}

void orc_scene_destroy(void* scene) { delete (Scene*)scene; }

static Field<float> scene_field32(const Scene& s) {
    std::vector<float> xyzr;
    for (size_t i = 0; i < s.lenses.size(); ++i) {
        xyzr.insert(xyzr.end(), s.lenses[i].c, s.lenses[i].c + 3);
        xyzr.push_back(s.lenses[i].rs);
    }
    return make_field<float>(xyzr.data(), (int)s.lenses.size(), s.lens_cfg);
}
static Field<double> scene_field64(const Scene& s) {
    std::vector<float> xyzr;
    for (size_t i = 0; i < s.lenses.size(); ++i) {
        xyzr.insert(xyzr.end(), s.lenses[i].c, s.lenses[i].c + 3);
        xyzr.push_back(s.lenses[i].rs);
    }
    return make_field<double>(xyzr.data(), (int)s.lenses.size(), s.lens_cfg);
}

int orc_render(void* scene_p, uint64_t camera_ref, const orc_config* cfg, uint64_t seed,
               uint64_t sample_base, float* rgba32f, uint32_t width, uint32_t height, int n_threads,
               uint64_t* samples_inout) {
    try {
        const Scene& scene = *(const Scene*)scene_p;
        if (cfg->samples == 0) return 0;  // Status::Done, mod.rs:186-188
        ChunkConfig cc = ChunkConfig::with_configs(*cfg);
        CameraSetup cs = camera_setup(scene, camera_ref, cc, width, height);
        Field<float> field = scene_field32(scene);
        uint32_t sub_count = cs.sub_n * cs.sub_n;

        // Buffer::chunks, buffer.rs:102-115, 293-326
        uint32_t cx = cfg->chunks_x ? cfg->chunks_x : 1, cy = cfg->chunks_y ? cfg->chunks_y : 1;
        uint32_t cw = width % cx == 0 ? width / cx : width / cx + 1;
        uint32_t ch = height % cy == 0 ? height / cy : height / cy + 1;
        struct Tile { uint32_t x0, y0, x1, y1; };
        std::vector<Tile> tiles;
        for (uint32_t y0 = 0; y0 < height; y0 += ch)
            for (uint32_t x0 = 0; x0 < width; x0 += cw) {
                Tile t = {x0, y0, std::min(x0 + cw, width), std::min(y0 + ch, height)};
                tiles.push_back(t);
            }
        std::atomic<size_t> next(0);
        std::atomic<int> failed(0);
        auto worker = [&]() {
            try {
                ChunkState st;
                st.config = cc;
                st.scene = &scene;
                st.field = field;
                for (;;) {
                    size_t ti = next.fetch_add(1);
                    if (ti >= tiles.size() || failed.load()) break;
                    const Tile& t = tiles[ti];
                    for (uint32_t y = t.y0; y < t.y1; ++y)
                        for (uint32_t x = t.x0; x < t.x1; ++x) {
                            float* px = rgba32f + 4 * ((size_t)y * width + x);
                            for (uint64_t s = 0; s < cc.samples; ++s)
                                for (uint32_t k = 0; k < sub_count; ++k) {
                                    uint64_t path_index = (sample_base + s) * sub_count + k;
                                    st.rng = Rng::seed_from_u64(path_seed(seed, (uint64_t)y * width + x, path_index));
                                    Rayf ray = camera_ray(cs, st.rng, x, y, k);
                                    ColorData sample = st.sample(ray, 0);
                                    float depth = (sample.depth - cc.clip_min) / (cc.clip_max - cc.clip_min);
                                    depth = std::min(std::max(depth, 0.0f), 1.0f);
                                    switch (cc.output) {  // mod.rs:310-315 -> buffer.rs:159-178
                                        case ORC_OUT_FULL: px[0] += sample.color.x; px[1] += sample.color.y; px[2] += sample.color.z; break;
                                        case ORC_OUT_ALBEDO: px[0] += sample.albedo.x; px[1] += sample.albedo.y; px[2] += sample.albedo.z; break;
                                        case ORC_OUT_NORMAL: px[0] += sample.normal.x; px[1] += sample.normal.y; px[2] += sample.normal.z; break;
                                        default: px[0] += depth; px[1] += depth; px[2] += depth; break;
                                    }
                                }
                        }
                }
            } catch (const std::exception& e) {
                g_last_error_shared = e.what();
                failed.store(1);
            }
        };
        if (n_threads <= 1) {
            worker();
        } else {
            std::vector<std::thread> th;
            for (int i = 0; i < n_threads; ++i) th.emplace_back(worker);
            for (size_t i = 0; i < th.size(); ++i) th[i].join();
        }
        if (failed.load()) {
            g_last_error = g_last_error_shared;
            return -1;
        }
        if (samples_inout) *samples_inout += cc.samples * sub_count;  // mod.rs:199
        return 1;  // Status::InProgress
    } catch (const std::exception& e) {
        g_last_error = g_last_error_shared = e.what();
        return -1;
    }
}

float orc_linear_to_srgb(float x) {  // color.rs:14-20
    if (x <= 0.0031308f) return 12.92f * x;
    return 1.055f * std::pow(x, 1.0f / 2.4f) - 0.055f;
}
static uint8_t f32_to_u8(float x) {  // color.rs:22-24 with Rust's saturating cast
    float v = x * 255.0f;
    if (v != v) return 0;
    if (v <= 0.0f) return 0;
    if (v >= 255.0f) return 255;
    return (uint8_t)v;
}
void orc_resolve_u8(const float* rgba32f, uint32_t width, uint32_t height, uint64_t samples,
                    int color_space, uint8_t* rgba8) {  // buffer.rs:117-138
    float samples_recip = 1.0f / (float)samples;
    for (size_t i = 0; i < (size_t)width * height; ++i) {
        V3f rgb = mk<float>(rgba32f[4 * i], rgba32f[4 * i + 1], rgba32f[4 * i + 2]) * samples_recip;
        V3f c;
        switch (color_space) {
            case ORC_CS_NORMAL: c = (normalize_s(rgb) + splat<float>(1.0f)) * 0.5f; break;
            case ORC_CS_SRGB: c = mk<float>(orc_linear_to_srgb(rgb.x), orc_linear_to_srgb(rgb.y), orc_linear_to_srgb(rgb.z)); break;
            default: c = rgb; break;
        }
        rgba8[4 * i] = f32_to_u8(c.x);
        rgba8[4 * i + 1] = f32_to_u8(c.y);
        rgba8[4 * i + 2] = f32_to_u8(c.z);
        rgba8[4 * i + 3] = f32_to_u8(rgba32f[4 * i + 3]);
    }
}

}  // extern "C"
template <class T>
static void probe_one(const Scene& scene, const Field<T>& f, const orc_config* cfg, const float* o, const float* d,
                      orc_probe_result* out) {
    Ray<T> ray = {mk<T>(o[0], o[1], o[2]), mk<T>(d[0], d[1], d[2])};
    Segment<T> seg = trace_segment<T>(scene, f, ray, T(cfg->clip_min), T(cfg->clip_max));
    std::memset(out, 0, sizeof(*out));
    out->steps = seg.steps;
    if (seg.status == SEG_HIT) {
        const Manifold<T>& m = seg.manifold;
        out->face = m.face;
        out->object_ref = m.object_ref;
        out->t = m.t;
        out->position[0] = m.position.x; out->position[1] = m.position.y; out->position[2] = m.position.z;
        out->normal[0] = m.normal.x; out->normal[1] = m.normal.y; out->normal[2] = m.normal.z;
        out->direction[0] = m.ray.direction.x; out->direction[1] = m.ray.direction.y; out->direction[2] = m.ray.direction.z;
    } else if (seg.status == SEG_ESCAPED) {
        out->face = ORC_FACE_MISS;
        out->position[0] = seg.escape.origin.x; out->position[1] = seg.escape.origin.y; out->position[2] = seg.escape.origin.z;
        out->direction[0] = seg.escape.direction.x; out->direction[1] = seg.escape.direction.y; out->direction[2] = seg.escape.direction.z;
    } else {
        out->face = ORC_FACE_CAPTURED;
    }
}

extern "C" {
int orc_probe(void* scene_p, const orc_config* cfg, int n, const float* origins, const float* dirs,
              int use_f64, orc_probe_result* out) {
    try {
        const Scene& scene = *(const Scene*)scene_p;
        if (use_f64) {
            Field<double> f = scene_field64(scene);
            for (int i = 0; i < n; ++i) probe_one<double>(scene, f, cfg, origins + 3 * i, dirs + 3 * i, out + i);
        } else {
            Field<float> f = scene_field32(scene);
            for (int i = 0; i < n; ++i) probe_one<float>(scene, f, cfg, origins + 3 * i, dirs + 3 * i, out + i);
        }
        return 0;
    } catch (const std::exception& e) {
        g_last_error = g_last_error_shared = e.what();
        return -1;
    }
}

int orc_camera_rays(void* scene_p, uint64_t camera_ref, const orc_config* cfg, uint64_t seed,
                    uint64_t sample_base, uint32_t width, uint32_t height, int n,
                    const uint32_t* xs, const uint32_t* ys, const uint64_t* path_index, float* out) {
    try {
        const Scene& scene = *(const Scene*)scene_p;
        ChunkConfig cc = ChunkConfig::with_configs(*cfg);
        CameraSetup cs = camera_setup(scene, camera_ref, cc, width, height);
        uint32_t sub_count = cs.sub_n * cs.sub_n;
        for (int i = 0; i < n; ++i) {
            uint64_t pi = sample_base * sub_count + path_index[i];
            Rng rng = Rng::seed_from_u64(path_seed(seed, (uint64_t)ys[i] * width + xs[i], pi));
            Rayf r = camera_ray(cs, rng, xs[i], ys[i], (uint32_t)(path_index[i] % sub_count));
            out[6 * i] = r.origin.x; out[6 * i + 1] = r.origin.y; out[6 * i + 2] = r.origin.z;
            out[6 * i + 3] = r.direction.x; out[6 * i + 4] = r.direction.y; out[6 * i + 5] = r.direction.z;
        }
        return 0;
    } catch (const std::exception& e) {
        g_last_error = g_last_error_shared = e.what();
        return -1;
    }
}

}  // extern "C"
template <class T>
static void integrate_one(const Field<T>& f, V3<T>& x, V3<T>& v, uint32_t n_steps) {
    for (uint32_t s = 0; s < n_steps; ++s) {
        T rmin;
        AccelInfo info;
        V3<T> k1 = accel<T>(f, x, false, T(0), v, v, &rmin, &info);
        rk4_from_k1(f, x, v, k1, step_size(f, rmin));
    }
}
extern "C" {
void orc_integrate(const float* xyzr, int n_lens, const orc_lens_config* cfg, int n, const float* xv,
                   uint32_t n_steps, int use_f64, float* out32, double* out64) {
    if (use_f64) {
        Field<double> f = make_field<double>(xyzr, n_lens, *cfg);
        for (int i = 0; i < n; ++i) {
            V3<double> x = mk<double>(xv[6 * i], xv[6 * i + 1], xv[6 * i + 2]);
            V3<double> v = mk<double>(xv[6 * i + 3], xv[6 * i + 4], xv[6 * i + 5]);
            integrate_one(f, x, v, n_steps);
            double* o = out64 + 6 * i;
            o[0] = x.x; o[1] = x.y; o[2] = x.z; o[3] = v.x; o[4] = v.y; o[5] = v.z;
        }
    } else {
        Field<float> f = make_field<float>(xyzr, n_lens, *cfg);
        for (int i = 0; i < n; ++i) {
            V3f x = mk<float>(xv[6 * i], xv[6 * i + 1], xv[6 * i + 2]);
            V3f v = mk<float>(xv[6 * i + 3], xv[6 * i + 4], xv[6 * i + 5]);
            integrate_one(f, x, v, n_steps);
            float* o = out32 + 6 * i;
            o[0] = x.x; o[1] = x.y; o[2] = x.z; o[3] = v.x; o[4] = v.y; o[5] = v.z;
        }
    }
}

// ---- unit-level exports ----
void orc_xoshiro_from_seed(const uint64_t s[4], uint64_t* out, int n) {
    Rng r;
    std::memcpy(r.s, s, 32);
    for (int i = 0; i < n; ++i) out[i] = r.next_u64();
}
void orc_xoshiro_seed_from_u64(uint64_t seed, uint64_t state_out[4]) {
    Rng r = Rng::seed_from_u64(seed);
    std::memcpy(state_out, r.s, 32);
}
uint64_t orc_path_seed(uint64_t seed, uint64_t pixel, uint64_t path_index) { return path_seed(seed, pixel, path_index); }
void orc_uniform_f32(uint64_t seed, float lo, float hi, int inclusive, float* out, int n, float* scale_out) {
    Rng r = Rng::seed_from_u64(seed);
    UniformF32 u = inclusive ? UniformF32::make_inclusive(lo, hi) : UniformF32::make(lo, hi);
    if (scale_out) *scale_out = u.scale;
    for (int i = 0; i < n; ++i) out[i] = u.sample(r);
}
void orc_standard_f32(uint64_t seed, float* out, int n) {
    Rng r = Rng::seed_from_u64(seed);
    for (int i = 0; i < n; ++i) out[i] = standard_f32(r);
}
int orc_gen_bool(uint64_t seed, double p, uint8_t* out, int n) {
    try {
        Rng r = Rng::seed_from_u64(seed);
        for (int i = 0; i < n; ++i) out[i] = gen_bool(r, p) ? 1 : 0;
        return 0;
    } catch (const std::exception& e) {
        g_last_error = g_last_error_shared = e.what();
        return -1;
    }
}
int orc_uniform_usize(uint64_t seed, uint64_t n_range, uint64_t* out, int n) {
    try {
        Rng r = Rng::seed_from_u64(seed);
        for (int i = 0; i < n; ++i) out[i] = uniform_usize(r, n_range);
        return 0;
    } catch (const std::exception& e) {
        g_last_error = g_last_error_shared = e.what();
        return -1;
    }
}
void orc_with_frustum(float yfov, float xfov, float u, float v, float dir_out[3]) {
    V3f d = with_frustum_dir(yfov, xfov, u, v);
    dir_out[0] = d.x; dir_out[1] = d.y; dir_out[2] = d.z;
}
void orc_environment_lookup(const float* rgb, uint32_t width, uint32_t height, const float d[3], float out[3]) {
    V3f c = env_lookup(rgb, width, height, mk<float>(d[0], d[1], d[2]));
    out[0] = c.x; out[1] = c.y; out[2] = c.z;
}
void orc_equirect_dir(float u, float v, float pixel_width, float pixel_height, float out[3]) {
    V3f d = panorama_dir(u, v, pixel_width, pixel_height);
    out[0] = d.x; out[1] = d.y; out[2] = d.z;
}
void orc_any_orthonormal_pair(const float n[3], float a_out[3], float b_out[3]) {
    V3f a, b;
    any_orthonormal_pair(mk<float>(n[0], n[1], n[2]), &a, &b);
    a_out[0] = a.x; a_out[1] = a.y; a_out[2] = a.z;
    b_out[0] = b.x; b_out[1] = b.y; b_out[2] = b.z;
}
void orc_distr(int which, uint64_t seed, const float n[3], float* out, int count) {
    Rng r = Rng::seed_from_u64(seed);
    Basis b(mk<float>(n[0], n[1], n[2]));
    for (int i = 0; i < count; ++i) {
        V3f v;
        switch (which) {
            case 0: v = unit_sphere(r); break;
            case 1: v = unit_hemisphere(r, b); break;
            case 2: v = cosine(r, b); break;
            default: v = unit_disk(r, b); break;
        }
        out[3 * i] = v.x; out[3 * i + 1] = v.y; out[3 * i + 2] = v.z;
    }
}
int orc_sphere_hit(const float center[3], float radius, const float o[3], const float d[3],
                   float clip_min, float clip_max, float* t_out, float normal_out[3], int* face_out) {
    orc_object obj;
    std::memset(&obj, 0, sizeof(obj));
    obj.kind = ORC_SPHERE;
    obj.volume = -1;
    obj.radius = radius;
    obj.transform[0] = obj.transform[4] = obj.transform[8] = 1.0f;
    obj.transform[9] = center[0]; obj.transform[10] = center[1]; obj.transform[11] = center[2];
    Rayf ray = {mk<float>(o[0], o[1], o[2]), mk<float>(d[0], d[1], d[2])};
    Clip<float> clip = {clip_min, clip_max};
    Manifold<float> m;
    if (!sphere_hit(obj, ray, clip, &m)) return 0;
    *t_out = m.t;
    normal_out[0] = m.normal.x; normal_out[1] = m.normal.y; normal_out[2] = m.normal.z;
    *face_out = m.face;
    return 1;
}
int orc_rect_hit(const orc_rect* rect, const float transform[12], const float o[3], const float d[3],
                 float clip_min, float clip_max, float* t_out, float normal_out[3], int* face_out) {
    Rayf ray = {mk<float>(o[0], o[1], o[2]), mk<float>(d[0], d[1], d[2])};
    Clip<float> clip = {clip_min, clip_max};
    Manifold<float> m;
    if (!rect_hit(*rect, 0, affine_from<float>(transform), ray, clip, &m)) return 0;
    *t_out = m.t;
    normal_out[0] = m.normal.x; normal_out[1] = m.normal.y; normal_out[2] = m.normal.z;
    *face_out = m.face;
    return 1;
}
float orc_density_sample(const orc_data* vol, const float coord[3]) {
    Data d;
    d.d = *vol;
    size_t n = (size_t)vol->width * vol->height * vol->depth;
    d.buffer.assign(vol->buffer, vol->buffer + n);
    return density_trilinear(d, mk<float>(coord[0], coord[1], coord[2]));
}
void orc_reflect(const float d[3], const float n[3], float out[3]) {
    V3f r = reflect(mk<float>(d[0], d[1], d[2]), mk<float>(n[0], n[1], n[2]));
    out[0] = r.x; out[1] = r.y; out[2] = r.z;
}
void orc_refract(const float d[3], const float n[3], float ior, float out[3]) {
    V3f r = refract(mk<float>(d[0], d[1], d[2]), mk<float>(n[0], n[1], n[2]), ior);
    out[0] = r.x; out[1] = r.y; out[2] = r.z;
}
float orc_fresnel(const float d[3], const float n[3], float ior) {
    return fresnel(mk<float>(d[0], d[1], d[2]), mk<float>(n[0], n[1], n[2]), ior);
}
void orc_rk4_step_f32(const float* xyzr, int n_lens, float* x, float* v, float h) {
    orc_lens_config cfg = {0.05f, 0.0f, 1e30f, 1e30f, 0};
    Field<float> f = make_field<float>(xyzr, n_lens, cfg);
    V3f X = mk<float>(x[0], x[1], x[2]), V = mk<float>(v[0], v[1], v[2]);
    V3f k1 = accel<float>(f, X, false, 0.0f, V, V, 0, 0);
    rk4_from_k1(f, X, V, k1, h);
    x[0] = X.x; x[1] = X.y; x[2] = X.z; v[0] = V.x; v[1] = V.y; v[2] = V.z;
}
void orc_rk4_step_f64(const float* xyzr, int n_lens, double* x, double* v, double h) {
    orc_lens_config cfg = {0.05f, 0.0f, 1e30f, 1e30f, 0};
    Field<double> f = make_field<double>(xyzr, n_lens, cfg);
    V3<double> X = mk<double>(x[0], x[1], x[2]), V = mk<double>(v[0], v[1], v[2]);
    V3<double> k1 = accel<double>(f, X, false, 0.0, V, V, 0, 0);
    rk4_from_k1(f, X, V, k1, h);
    x[0] = X.x; x[1] = X.y; x[2] = X.z; v[0] = V.x; v[1] = V.y; v[2] = V.z;
}

}  // extern "C"
