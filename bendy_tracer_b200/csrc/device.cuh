// device.cuh -- device-side math of the render loop: RNG + distributions, vector helpers,
// primitive intersection over the shared-memory SoA blob, shading, volume shading and the
// geodesic (RK4) stepper.  The exact flavour is compiled with -fmad=false: a*b+c is never
// contracted (the Rust reference never contracts either), FMAs appear only where written as fmaf()
// -- i.e. in the geodesic stepper, whose arithmetic is this project's own definition (DESIGN.md).
// The fast flavour lets the compiler contract everything except the x*() helpers below.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "layout.h"

namespace bt {

#define BT_DEV __device__ __forceinline__

// ------------------------------------------------------------------------------------------
// vectors (glam operation order: dot = (x*x' + y*y') + z*z')
// ------------------------------------------------------------------------------------------
struct V3 {
    float x, y, z;
};
BT_DEV V3 v3(float x, float y, float z) { V3 r = {x, y, z}; return r; }
BT_DEV V3 v3(float4 q) { V3 r = {q.x, q.y, q.z}; return r; }
BT_DEV V3 operator+(V3 a, V3 b) { return v3(a.x + b.x, a.y + b.y, a.z + b.z); }
BT_DEV V3 operator-(V3 a, V3 b) { return v3(a.x - b.x, a.y - b.y, a.z - b.z); }
BT_DEV V3 operator-(V3 a) { return v3(-a.x, -a.y, -a.z); }
BT_DEV V3 operator*(V3 a, float s) { return v3(a.x * s, a.y * s, a.z * s); }
BT_DEV V3 operator*(float s, V3 a) { return v3(s * a.x, s * a.y, s * a.z); }
BT_DEV V3 operator*(V3 a, V3 b) { return v3(a.x * b.x, a.y * b.y, a.z * b.z); }
BT_DEV V3 operator/(V3 a, float s) { return v3(a.x / s, a.y / s, a.z / s); }
BT_DEV V3 operator/(V3 a, V3 b) { return v3(a.x / b.x, a.y / b.y, a.z / b.z); }
BT_DEV float dot(V3 a, V3 b) { return (a.x * b.x + a.y * b.y) + a.z * b.z; }
// The same operations with every product and sum rounded separately whatever the compiler's FMA
// contraction setting (the fast flavour is built -fmad=true): used where a contraction would matter --
// the sphere quadratic (|oc|^2 - r^2 cancels catastrophically for large spheres) and the hit point,
// which the scan, the BVH and the oracle must all round the same way.
BT_DEV float xdot(V3 a, V3 b) { return __fadd_rn(__fadd_rn(__fmul_rn(a.x, b.x), __fmul_rn(a.y, b.y)), __fmul_rn(a.z, b.z)); }
BT_DEV V3 xat(V3 o, float t, V3 d) { return v3(__fadd_rn(o.x, __fmul_rn(t, d.x)), __fadd_rn(o.y, __fmul_rn(t, d.y)), __fadd_rn(o.z, __fmul_rn(t, d.z))); }
BT_DEV V3 cross(V3 a, V3 b) { return v3(a.y * b.z - b.y * a.z, a.z * b.x - b.z * a.x, a.x * b.y - b.x * a.y); }
// Two arithmetic flavours (compile time).  BT_EXACT_SCAN: every division / square root is the IEEE
// operation the Rust reference performs, so values are bit-identical to the CPU oracle.  Default:
// MUFU-based reciprocal / square root / reciprocal square root, each within ~1 ulp of the IEEE
// result (PTX rcp.approx / sqrt.approx: <= 1 ulp; rsqrt.approx + one Newton step), a fraction of
// the instructions.  The parity tests hold the default build to the north-star tolerances.
#ifdef BT_EXACT_SCAN
#define BT_X_RCP 1
#define BT_X_SQRT 1
#define BT_X_RSQRT 1
#define BT_X_DIV 1
#define BT_X_NORM 1
#endif
#ifdef BT_X_RCP
BT_DEV float m_rcp(float x) { return 1.0f / x; }
#else
BT_DEV float m_rcp(float x) {
    float r;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
    return r;
}
#endif
#ifdef BT_X_SQRT
BT_DEV float m_sqrt(float x) { return sqrtf(x); }
#else
BT_DEV float m_sqrt(float x) {
    float r;
    asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
    return r;
}
#endif
#ifdef BT_X_RSQRT
BT_DEV float m_rsqrt(float x) { return 1.0f / sqrtf(x); }
#else
BT_DEV float m_rsqrt(float x) {  // MUFU.RSQ + one Newton step
    float y;
    asm("rsqrt.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    const float e = fmaf(-(x * y), y, 1.0f);
    return fmaf(0.5f * y, e, y);
}
#endif
#ifdef BT_X_DIV
BT_DEV V3 m_div(V3 a, float s) { return v3(a.x / s, a.y / s, a.z / s); }
BT_DEV V3 m_div(V3 a, V3 b) { return v3(a.x / b.x, a.y / b.y, a.z / b.z); }
#else
BT_DEV V3 m_div(V3 a, float s) { return a * m_rcp(s); }
BT_DEV V3 m_div(V3 a, V3 b) { return v3(a.x * m_rcp(b.x), a.y * m_rcp(b.y), a.z * m_rcp(b.z)); }
#endif
#ifdef BT_X_NORM
BT_DEV V3 normalize_a(V3 a) { return a / sqrtf(dot(a, a)); }
#else
BT_DEV V3 normalize_a(V3 a) { return a * m_rsqrt(dot(a, a)); }
#endif
// Vec3A::normalize: v / sqrt(dot);  Vec3::normalize: v * (1 / sqrt(dot))
BT_DEV V3 normalize_s(V3 a) { return a * m_rsqrt(dot(a, a)); }
BT_DEV V3 normalize_or_zero_s(V3 a) {
    float rcp = m_rsqrt(dot(a, a));
    if (isfinite(rcp) && rcp > 0.0f) return a * rcp;
    return v3(0.0f, 0.0f, 0.0f);
}
// Mat3A * Vec3A with columns c0,c1,c2: ((c0*x) + c1*y) + c2*z
BT_DEV V3 mat_vec(V3 c0, V3 c1, V3 c2, V3 v) { return (c0 * v.x + c1 * v.y) + c2 * v.z; }

// Vec3::any_orthonormal_pair (glam)
BT_DEV void any_orthonormal_pair(V3 n, V3& a_out, V3& b_out) {
    float sign = copysignf(1.0f, n.z);
    float a = -m_rcp(sign + n.z);
    float b = n.x * n.y * a;
    a_out = v3(1.0f + sign * n.x * n.x * a, sign * b, -sign * n.x);
    b_out = v3(b, sign + n.y * n.y * a, -n.y);
}
BT_DEV float lerpf(float a, float b, float f) { return a + (b - a) * f; }          // math/mod.rs:5-25
BT_DEV V3 reflect(V3 d, V3 n) { return d - (2.0f * dot(d, n)) * n; }                // math/mod.rs:39-41
BT_DEV V3 refract(V3 d, V3 n, float ior) {                                          // math/mod.rs:43-48
    float cos_theta = fminf(dot(-d, n), 1.0f);
    V3 perp = (n * cos_theta + d) * ior;
    V3 parallel = n * -m_sqrt(fabsf(1.0f - dot(perp, perp)));
    return perp + parallel;
}
BT_DEV float fresnel(V3 d, V3 n, float ior) {                                       // math/mod.rs:50-55
    float cos_theta = fminf(dot(-d, n), 1.0f);
    float r0 = (1.0f - ior) * m_rcp(1.0f + ior);
    r0 = r0 * r0;
    float x = 1.0f - cos_theta;
    float x2 = x * x;
    float x4 = x2 * x2;
    return r0 + (1.0f - r0) * (x * x4);  // powi(5)
}

// ------------------------------------------------------------------------------------------
// RNG: xoshiro256++ (rand 0.8.5 SmallRng on 64-bit), keyed per camera path
// ------------------------------------------------------------------------------------------
BT_DEV uint64_t rotl64(uint64_t x, int k) { return (x << k) | (x >> (64 - k)); }
BT_DEV uint64_t splitmix_mix(uint64_t z) {
    z = (z ^ (z >> 30)) * 0xbf58476d1ce4e5b9ULL;
    z = (z ^ (z >> 27)) * 0x94d049bb133111ebULL;
    return z ^ (z >> 31);
}
struct Rng {
    uint64_t s0, s1, s2, s3;
    BT_DEV uint64_t next_u64() {
        uint64_t result = rotl64(s0 + s3, 23) + s0;
        uint64_t t = s1 << 17;
        s2 ^= s0;
        s3 ^= s1;
        s1 ^= s2;
        s0 ^= s3;
        s2 ^= t;
        s3 = rotl64(s3, 45);
        return result;
    }
    BT_DEV uint32_t next_u32() { return (uint32_t)(next_u64() >> 32); }
    BT_DEV void seed_from_u64(uint64_t state) {  // SplitMix64 x 4
        state += 0x9e3779b97f4a7c15ULL; s0 = splitmix_mix(state);
        state += 0x9e3779b97f4a7c15ULL; s1 = splitmix_mix(state);
        state += 0x9e3779b97f4a7c15ULL; s2 = splitmix_mix(state);
        state += 0x9e3779b97f4a7c15ULL; s3 = splitmix_mix(state);
        if ((s0 | s1 | s2 | s3) == 0) {  // from_seed(all zero) -> seed_from_u64(0)
            s0 = 0xe220a8397b1dcdafULL; s1 = 0x6e789e6aa1b965f4ULL; s2 = 0x06c45d188009454fULL; s3 = 0xf88bb8a8724c81ecULL;
        }
    }
};
BT_DEV uint64_t path_seed(uint64_t seed, uint64_t pixel, uint64_t path_index) {
    uint64_t k = splitmix_mix(seed + 0x9e3779b97f4a7c15ULL);
    k = splitmix_mix(k + 0x9e3779b97f4a7c15ULL * (pixel + 1));
    k = splitmix_mix(k + 0xd1342543de82ef95ULL * (path_index + 1));
    return k;
}
// Uniform<f32>::sample with a precomputed (low, scale)
BT_DEV float uniform_f32(Rng& rng, float low, float scale) {
    float value1_2 = __uint_as_float((rng.next_u32() >> 9) | 0x3f800000u);
    float value0_1 = value1_2 - 1.0f;
    return value0_1 * scale + low;
}
BT_DEV float standard_f32(Rng& rng) { return (float)(rng.next_u32() >> 8) * (1.0f / 16777216.0f); }
// Bernoulli::new(p as f64): p_int = (p * 2^64) as u64, exact in integer arithmetic for f32 p in [0, 1)
BT_DEV bool gen_bool(Rng& rng, float p) {
    if (p >= 1.0f) return true;  // ALWAYS_TRUE: no draw (p > 1 panics in the reference)
    uint32_t bits = __float_as_uint(p);
    int e = (int)((bits >> 23) & 0xff);
    uint64_t mant = bits & 0x7fffffu;
    if (e != 0) mant |= 0x800000u; else e = 1;
    int shift = e - 86;  // value = mant * 2^(e - 150); times 2^64
    uint64_t p_int = shift >= 0 ? (mant << shift) : (shift > -64 ? (mant >> (-shift)) : 0ULL);
    return rng.next_u64() < p_int;
}
// UniformInt<usize>::new(0, n).sample (rand 0.8.5: widening multiply, rejection above `zone`).
// zone = MAX - (MAX - n + 1) % n depends on n only: the host computes it once per call
// (RenderParams::light_zone) -- in the kernel the 64-bit modulo was a 70-instruction subroutine
// per Diffuse event.  n == 1: every draw is accepted and the index is 0 (the draw is still consumed).
BT_DEV uint32_t uniform_index(Rng& rng, uint32_t n, uint64_t zone) {
    if (n == 1) {
        (void)rng.next_u64();
        return 0;
    }
    const uint64_t range = n;
    for (;;) {
        uint64_t v = rng.next_u64();
        uint64_t lo = v * range;
        if (lo <= zone) return (uint32_t)__umul64hi(v, range);
    }
}

// sin and cos of one argument (|x| up to a few thousand): Cody-Waite reduction by pi/2 in three
// parts and the Cephes single-precision minimax polynomials on [-pi/4, pi/4], all in explicit FMAs.
// <= 1.5 ulp, like CUDA's sincosf, at a quarter of its code size (no Payne-Hanek path): the render
// kernel calls it from four places and its loop body has to stay inside the instruction cache.
BT_DEV void bt_sincos(float x, float* sn, float* cs) {
#ifdef BT_EXACT_SCAN
    sincosf(x, sn, cs);  // agrees with glibc's sinf / cosf (the oracle) on all but ~1e-4 of arguments
    return;
#endif
    const float k = rintf(x * 0.636619772367581343f);
    float y = fmaf(k, -1.5703125f, x);
    y = fmaf(k, -4.837512969970703125e-4f, y);
    y = fmaf(k, -7.549789954891882e-8f, y);
    const int q = (int)k;
    const float y2 = y * y;
    float s = fmaf(-1.9515295891e-4f, y2, 8.3321608736e-3f);
    s = fmaf(s, y2, -1.6666654611e-1f);
    s = fmaf(s * y2, y, y);
    float c = fmaf(2.443315711809948e-5f, y2, -1.388731625493765e-3f);
    c = fmaf(c, y2, 4.166664568298827e-2f);
    c = fmaf(c * y2, y2, fmaf(-0.5f, y2, 1.0f));
    const float a = (q & 1) ? c : s, b = (q & 1) ? s : c;
    *sn = (q & 2) ? -a : a;
    *cs = ((q + 1) & 2) ? -b : b;
}

struct Consts {  // Uniform::new_inclusive(0, TAU) / (0, 1): low = 0
    float tau_scale, one_scale;
};
// math/distr.rs:7-27
BT_DEV V3 unit_sphere(Rng& rng, const Consts& k) {
    float r1 = uniform_f32(rng, 0.0f, k.tau_scale);
    float r2 = uniform_f32(rng, 0.0f, k.one_scale);
    float s, c;
    bt_sincos(r1, &s, &c);
    float w = sqrtf(r2 * (1.0f - r2));
    return v3(c * 2.0f * w, s * 2.0f * w, 1.0f - 2.0f * r2);
}
// math/distr.rs:29-65 (z = 1 - r2: not unit length, as in the reference)
BT_DEV V3 unit_hemisphere(Rng& rng, const Consts& k, V3 normal) {
    V3 zx = normalize_s(normal), xa, ya;
    any_orthonormal_pair(zx, xa, ya);
    float r1 = uniform_f32(rng, 0.0f, k.tau_scale);
    float r2 = uniform_f32(rng, 0.0f, k.one_scale);
    float s, c;
    bt_sincos(r1, &s, &c);
    float w = sqrtf(r2 * (1.0f - r2));
    return (xa * (c * 2.0f * w) + ya * (s * 2.0f * w)) + zx * (1.0f - r2);
}
// math/distr.rs:67-103
BT_DEV V3 cosine_dir(Rng& rng, const Consts& k, V3 normal) {
    V3 zx = normalize_s(normal), xa, ya;
    any_orthonormal_pair(zx, xa, ya);
    float r1 = uniform_f32(rng, 0.0f, k.tau_scale);
    float r2 = uniform_f32(rng, 0.0f, k.one_scale);
    float s, c;
    bt_sincos(r1, &s, &c);
    float w = sqrtf(r2);
    return (xa * (c * w) + ya * (s * w)) + zx * sqrtf(1.0f - r2);
}

// ------------------------------------------------------------------------------------------
// intersection over the shared-memory blob
// ------------------------------------------------------------------------------------------
struct Hit {
    float t;       // clip.max while scanning; the hit distance afterwards
    int prim;      // -1: miss
    int face;      // BT_FACE_*-compatible (0 front, 1 back, 2 volume, 3 volume front, 4 volume back)
};

// Two arithmetic flavours of the per-primitive tests:
//  * BT_EXACT_SCAN: the reference's operation order with every product and sum rounded separately
//    and an IEEE division -- hit distances are bit-identical to the CPU oracle;
//  * default: the RECT test with its dot products contracted to FMA chains, t = p * rcp(q)
//    (MUFU.RCP, <= 2 ulp) and no divergent early-outs.  Rect hit distances differ from the
//    reference by a few ulp (well inside the 1e-3 image bar, see tests/test_gpu_parity.py); ~35 %
//    fewer instructions per test.  Sphere tests keep the reference's rounding in both flavours.
#ifdef BT_EXACT_SCAN
BT_DEV float sdot(V3 a, V3 b) { return dot(a, b); }
BT_DEV V3 sat(V3 o, float t, V3 d) { return o + t * d; }
BT_DEV float sdiv(float p, float q) { return p / q; }
#else
BT_DEV float sdot(V3 a, V3 b) { return fmaf(a.z, b.z, fmaf(a.y, b.y, a.x * b.x)); }
BT_DEV V3 sat(V3 o, float t, V3 d) { return v3(fmaf(t, d.x, o.x), fmaf(t, d.y, o.y), fmaf(t, d.z, o.z)); }
BT_DEV float sdiv(float p, float q) { return __fdividef(p, q); }
#endif

// Sphere::hit roots (sphere.rs:121-148).  Returns true and the accepted root.
// FLIGHT: a chord of a geodesic under the fast stepper -- positions already carry ~1e-5 of MUFU.RSQ
// error, so the root uses the flavour's square root (MUFU.SQRT in the fast flavour).
template <bool FLIGHT = false>
BT_DEV bool sphere_roots_oc(V3 oc, float l2, float r2, V3 d, float tmin, float tmax, float& t_out) {
    // always the reference's rounding: |oc|^2 - r^2 cancels catastrophically for large spheres, and
    // a 1e-5 shift of a volume entry point flips Bernoulli scatter decisions at a visible rate
    float half_b = xdot(oc, d);
    float c = __fsub_rn(l2, r2);
    float disc = __fsub_rn(__fmul_rn(half_b, half_b), c);
    if (signbit(disc)) return false;  // most rays miss most spheres: a (mostly warp-uniform) early-out
    float sqrtd = FLIGHT ? m_sqrt(disc) : sqrtf(disc);
    float t0 = __fsub_rn(-half_b, sqrtd), t1 = __fadd_rn(-half_b, sqrtd);
    bool in0 = !(t0 < tmin || t0 > tmax), in1 = !(t1 < tmin || t1 > tmax);
    t_out = in0 ? t0 : t1;
    return in0 || in1;
}
template <bool FLIGHT = false>
BT_DEV bool sphere_roots(float4 q0, float r2, V3 o, V3 d, float tmin, float tmax, float& t_out) {
    V3 oc = o - v3(q0);
    return sphere_roots_oc<FLIGHT>(oc, xdot(oc, oc), r2, d, tmin, tmax, t_out);
}
BT_DEV float sqrt_approx(float x) {
    float r;
    asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
    return r;
}
// Rect::hit (rect.rs:110-155) on a pre-transformed record.  strict: Cuboid::hit's `t < best`.
BT_DEV bool rect_test_q(float4 q0, float4 q1, float4 q2, float4 q3, V3 o, V3 d, float tmin, float tmax, bool strict, float& t_out, bool& front) {
    const V3 n = v3(q0);
    const float qq = sdot(d, n);
    const float p = sdot(v3(q1) - o, n);
    const float t = sdiv(p, qq);
    bool ok = fabsf(qq) > 1e-5f && !(t < tmin || t > tmax) && !(strict && !(t < tmax));
    const V3 pos = sat(o, t, d);
#ifdef BT_EXACT_SCAN
    const float lx = dot(pos, v3(q2)) + q2.w;
    const float ly = dot(pos, v3(q3)) + q3.w;
#else
    const float lx = fmaf(pos.x, q2.x, fmaf(pos.y, q2.y, fmaf(pos.z, q2.z, q2.w)));
    const float ly = fmaf(pos.x, q3.x, fmaf(pos.y, q3.y, fmaf(pos.z, q3.z, q3.w)));
#endif
    ok = ok && (lx * lx <= q0.w) && (ly * ly <= q1.w);
    t_out = t;
    front = p < 0.0f;
    return ok;
}
BT_DEV bool rect_test(const float4* q, V3 o, V3 d, float tmin, float tmax, bool strict, float& t_out, bool& front) {
    return rect_test_q(q[0], q[1], q[2], q[3], o, d, tmin, tmax, strict, t_out, front);
}

// Rect::hit for a PRIM_RECT_AA record (layout.h): normal on axis K, q2 on axis (K+1)%3, q3 on (K+2)%3,
// all exact +-1.  Every dot product of rect_test then has one non-zero term (the products with the
// zero components are +-0 and the sums with them exact), so picking the components gives the same
// bits in both flavours with 5 multiply-adds instead of 15.  K is uniform across the warp.
template <int K> BT_DEV float comp(float4 v) { return K == 0 ? v.x : (K == 1 ? v.y : v.z); }
template <int K> BT_DEV float comp(V3 v) { return K == 0 ? v.x : (K == 1 ? v.y : v.z); }
#ifdef BT_EXACT_SCAN
BT_DEV float sat1(float o, float t, float d) { return o + t * d; }
#else
BT_DEV float sat1(float o, float t, float d) { return fmaf(t, d, o); }
#endif
template <int K>
BT_DEV bool rect_test_aa(const float4* q, V3 o, V3 d, float tmin, float tmax, float& t_out, bool& front) {
    const float4 q0 = q[0], q1 = q[1], q2 = q[2], q3 = q[3];
    const float nk = comp<K>(q0);
    const float qq = comp<K>(d) * nk;
    const float p = (comp<K>(q1) - comp<K>(o)) * nk;
    const float t = sdiv(p, qq);
    bool ok = fabsf(qq) > 1e-5f && !(t < tmin || t > tmax);
    const float pu = sat1(comp<(K + 1) % 3>(o), t, comp<(K + 1) % 3>(d));
    const float pw = sat1(comp<(K + 2) % 3>(o), t, comp<(K + 2) % 3>(d));
    const float lx = fmaf(pu, comp<(K + 1) % 3>(q2), q2.w);
    const float ly = fmaf(pw, comp<(K + 2) % 3>(q3), q3.w);
    ok = ok && (lx * lx <= q0.w) && (ly * ly <= q1.w);
    t_out = t;
    front = p < 0.0f;
    return ok;
}

// Cuboid::hit (cuboid.rs:83-105) for a cuboid whose six faces form one box: the smallest face
// distance in [tmin, tmax) from one slab test.  The per-face t equals Rect::hit's p / q for that
// face up to rounding; the rect's inside test becomes the slab-interval test.  Returns the face
// (0..5, the reference's face order) and Rect::hit's `p < 0` (front) for it.
BT_DEV float rcp_approx(float x) {  // MUFU.RCP, <= 1 ulp; callers guarantee 1e-5 < |x| <= ~1
    float r;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
    return r;
}
// *dist_out (optional): |L-infinity distance| from o to the box surface (outside: to the box; inside: to the nearest face)
BT_DEV bool box_test(const float4* b, V3 o, V3 d, float tmin, float tmax, float& t_out, int& face_out, bool& front_out,
                     float* dist_out = nullptr) {
    const float4 b0 = b[0], b1 = b[1], b2 = b[2], b3 = b[3];
    const V3 oc = v3(b0) - o;
    const float inf = __int_as_float(0x7f800000);
    // per axis k: p = (C - o) . a_k, q = d . a_k; the ray meets the planes at (p -/+ h) / q
    const float p0 = sdot(oc, v3(b1)), q0 = sdot(d, v3(b1)), h0 = b0.w;
    const float p1 = sdot(oc, v3(b2)), q1 = sdot(d, v3(b2)), h1 = b1.w;
    const float p2 = sdot(oc, v3(b3)), q2 = sdot(d, v3(b3)), h2 = b2.w;
    // Rect::hit's parallel-ray cut-off (rect.rs:122-124): such a pair of faces cannot be hit, and the
    // ray must lie inside their slab to hit any of the other four
    const bool par0 = !(fabsf(q0) > 1e-5f), par1 = !(fabsf(q1) > 1e-5f), par2 = !(fabsf(q2) > 1e-5f);
    const float i0 = rcp_approx(par0 ? 1.0f : q0), i1 = rcp_approx(par1 ? 1.0f : q1), i2 = rcp_approx(par2 ? 1.0f : q2);
    const float s0 = copysignf(h0, q0), s1 = copysignf(h1, q1), s2 = copysignf(h2, q2);
    const float n0 = par0 ? -inf : (p0 - s0) * i0, f0 = par0 ? inf : (p0 + s0) * i0;
    const float n1 = par1 ? -inf : (p1 - s1) * i1, f1 = par1 ? inf : (p1 + s1) * i1;
    const float n2 = par2 ? -inf : (p2 - s2) * i2, f2 = par2 ? inf : (p2 + s2) * i2;
    const float tn = fmaxf(fmaxf(n0, n1), n2), tf = fminf(fminf(f0, f1), f2);
    bool ok = tn <= tf && !(par0 && fabsf(p0) > h0) && !(par1 && fabsf(p1) > h1) && !(par2 && fabsf(p2) > h2);
    const bool near = tn >= tmin;  // the entry face if it is in range, else the exit face
    const float t = near ? tn : tf;
    ok = ok && !(t < tmin) && t < tmax;
    const int k = near ? (tn == n0 ? 0 : (tn == n1 ? 1 : 2)) : (tf == f0 ? 0 : (tf == f1 ? 1 : 2));
    const float p = k == 0 ? p0 : (k == 1 ? p1 : p2), q = k == 0 ? q0 : (k == 1 ? q1 : q2), h = k == 0 ? h0 : (k == 1 ? h1 : h2);
    // entering through the face on the side the ray comes from, leaving through the opposite one
    const bool plus = near ? q < 0.0f : q > 0.0f;
    const int face = 2 * k + (plus ? 1 : 0);
    const bool flipped = (__float_as_uint(b3.w) >> face) & 1u;  // stored normal = -a_k
    const float pface = p + (plus ? h : -h);                     // (T_face - o) . a_k
    t_out = t;
    face_out = face;
    front_out = flipped ? pface > 0.0f : pface < 0.0f;
    if (dist_out) *dist_out = fabsf(fmaxf(fmaxf(fabsf(p0) - h0, fabsf(p1) - h1), fabsf(p2) - h2));
    return ok;
}

// ChunkState::try_hit / try_hit_volume (mod.rs:389-427): linear scan in canonical object order
// with a shrinking clip.max.  volume_obj >= 0 selects hit_volumetric for that object's sphere.
// DIST: the same pass also returns a conservative lower bound on the distance from `o` to the
// nearest primitive surface (spheres: ||o - c| - r|; rects: L-infinity distance to the world
// AABB), minus a margin that covers the rounding of the hit tests themselves -- a ray that starts
// at `o` cannot be reported as hitting anything within that distance (the stepper's chord skip).
// C: what the scene contains (CT_* bits, layout.h) -- a kernel compiled for a scene without rects carries no rect / box
// code, one without volumetric spheres no march code, one without Glass no Fresnel / refraction.
// The render loop's body has to stay near the 32 KB instruction cache; every shipped scene gets a
// variant without the code it cannot reach (variants.h).
// What a DIST scan learns about the surroundings of the ray's origin: the smallest per-primitive
// bound, the primitive it belongs to when that is a sphere (-1 otherwise) and the smallest bound among
// all the other primitives.  The stepper re-evaluates the nearest sphere's distance exactly at every
// step (sphere_free_bound) and lets only `rest` decay with the distance flown.
struct FreeInfo {
    float nearest, rest;
    int sphere;
};
BT_DEV void free_update(FreeInfo& fi, float b, int sphere) {
    if (b < fi.nearest) {
        fi.rest = fi.nearest;
        fi.nearest = b;
        fi.sphere = sphere;
    } else {
        fi.rest = fminf(fi.rest, b);
    }
}
// lower bound on the distance from o to the surface of the sphere record q, minus the margin that
// covers the rounding of Sphere::hit itself (see scan_prims_t<DIST>); l2 = |o - c|^2
BT_DEV float sphere_free_bound(float4 q0, float4 q1, float l2) {
    const float dc = sqrt_approx(l2);
    return fabsf(dc - q0.w) - (l2 * q1.z + 2e-5f * (dc + q0.w) + 1e-6f);
}
template <bool DIST, int C = CT_ALL, bool FLIGHT = false>
BT_DEV Hit scan_prims_t(const float4* prims, const float4* bounds, const float4* boxes, int n_prims, V3 o, V3 d, float tmin,
                        float tmax, int volume_obj, FreeInfo* free_out) {
    (void)bounds;
    (void)boxes;
    Hit h;
    h.t = tmax;
    h.prim = -1;
    h.face = 0;
    FreeInfo fi;
    fi.nearest = fi.rest = __int_as_float(0x7f800000);
    fi.sphere = -1;
    for (int i = 0; i < n_prims; ++i) {
        const float4* q = prims + i * PRIM_STRIDE;
        float4 meta = q[4];
        int type = __float_as_int(meta.x) & 3;
        if ((C & CT_SPHERES) && (!(C & CT_RECTS) || type == PRIM_SPHERE)) {
            float4 q0 = q[0];
            const float4 q1 = q[1];
            float r2 = q1.x;
            if ((C & CT_VOLUMES) && !DIST && volume_obj >= 0 && __float_as_int(meta.w) == volume_obj) {
                // Sphere::hit_volumetric, sphere.rs:150-166
                V3 e = xat(o, h.t, d) - v3(q0);
                if (xdot(e, e) <= r2) {
                    h.prim = i;
                    h.face = 2;  // Face::Volume at t = clip.max
                    continue;
                }
            }
            float t;
            const V3 oc = o - v3(q0);
            const float l2 = xdot(oc, oc);
            if (DIST) {
                // A reported root t puts the point o + t d within ~1e-6 |oc|^2 / r of the true surface
                // (the residual of the quadratic, however ill-conditioned t itself is for a grazing
                // ray), so dist(o, surface) <= t + that: the margin below is 20x it, plus the rounding
                // of this bound.  q1.z = 2e-5 / r.
                free_update(fi, sphere_free_bound(q0, q1, l2), i);
            }
            if (sphere_roots_oc<FLIGHT>(oc, l2, r2, d, tmin, h.t, t)) {
                h.t = t;
                h.prim = i;
                h.face = 8;  // resolved after the scan (needs the normal)
            }
        } else if (C & CT_RECTS) {
            float t;
            bool front;
            if (type == PRIM_CUBOID_FACE && __float_as_int(meta.z) > 0) {
                // the first face of a box-shaped cuboid: all six faces in one slab test
                int face;
                float bd;
                const bool hit = box_test(boxes + (__float_as_int(meta.z) - 1) * BOX_STRIDE, o, d, tmin, h.t, t, face, front, DIST ? &bd : nullptr);
                if (DIST) free_update(fi, bd - (1e-4f * (fabsf(o.x) + fabsf(o.y) + fabsf(o.z) + bd) + 1e-4f), -1);
                if (hit) {
                    h.t = t;
                    h.prim = i + face;
                    h.face = front ? 0 : 1;
                }
                i += 5;
                continue;
            }
            if (DIST) {
                const float4 lo = bounds[i * BOUND_STRIDE], hi = bounds[i * BOUND_STRIDE + 1];
                const float dx = fmaxf(lo.x - o.x, o.x - hi.x), dy = fmaxf(lo.y - o.y, o.y - hi.y), dz = fmaxf(lo.z - o.z, o.z - hi.z);
                const float m = 1e-4f * (fabsf(o.x) + fabsf(o.y) + fabsf(o.z) + fabsf(hi.x - lo.x) + fabsf(hi.y - lo.y) + fabsf(hi.z - lo.z)) + 1e-4f;
                free_update(fi, fmaxf(fmaxf(dx, dy), dz) - m, -1);
            }
            bool hit;
            if (type == PRIM_RECT_AA) {  // (uniform across the warp)
                const int k = (__float_as_int(meta.x) >> 2) & 3;
                hit = k == 0 ? rect_test_aa<0>(q, o, d, tmin, h.t, t, front)
                             : (k == 1 ? rect_test_aa<1>(q, o, d, tmin, h.t, t, front) : rect_test_aa<2>(q, o, d, tmin, h.t, t, front));
            } else {
                hit = rect_test(q, o, d, tmin, h.t, type == PRIM_CUBOID_FACE, t, front);
            }
            if (hit) {
                h.t = t;
                h.prim = i;
                h.face = front ? 0 : 1;
            }
        }
    }
    if (DIST) *free_out = fi;
    return h;
}
template <int C = CT_ALL>
BT_DEV Hit scan_prims(const float4* prims, const float4* boxes, int n_prims, V3 o, V3 d, float tmin, float tmax, int volume_obj) {
    return scan_prims_t<false, C>(prims, nullptr, boxes, n_prims, o, d, tmin, tmax, volume_obj, nullptr);
}

// Closest hit through the BVH (extension; scenes above the linear-scan budget).  Records and
// nodes are read from global memory (L1 / L2), the traversal stack lives in shared memory
// (stack[level * blockDim.x + tid]: conflict-free; levels >= BVH_STACK_SMEM, rarely reached, in local
// memory).  Same per-primitive tests as the scan; an exact-distance tie is decided by the canonical
// primitive index exactly as the reference's scan order would: the later record wins unless it is a
// cuboid face (strict '<', cuboid.rs:97).
// entry distance of the ray into one child box of a 4-wide node, +inf when it misses.  (nx, fx): the box's plane the
// ray meets first / last along x -- min.x and max.x, swapped for a ray that runs towards -x (bvh_node picks them by the
// sign of 1 / d while it fetches, which saves the six min / max that would sort the plane distances here).
BT_DEV float slab(float nx, float fx, float ny, float fy, float nz, float fz, V3 o, V3 inv, float tmin, float tmax) {
    const float tnear = fmaxf(fmaxf((nx - o.x) * inv.x, (ny - o.y) * inv.y), fmaxf((nz - o.z) * inv.z, tmin));
    const float tfar = fminf(fminf((fx - o.x) * inv.x, (fy - o.y) * inv.y), fminf((fz - o.z) * inv.z, tmax));
    // inclusive and slightly generous: never cull a scan hit
    return tnear <= tfar * 1.00001f + 1e-6f ? tnear : __int_as_float(0x7f800000);
}
// A closest-hit traversal in progress (resumable: the render kernel advances the lanes of a warp one
// unit at a time and leaves the loop when enough of them are done -- step compaction, as for the
// geodesic flights).
struct BvhTrav {
    uint32_t cur, sp;
    Hit h;
};
// Where one traversal keeps its stack: levels < k in shared memory (entry `level * stride + idx`, the entry
// distances k * stride words further), the rarely reached rest in `over` (local memory in the lane kernel, a
// global arena in the pooled one).
struct BvhStack {
    uint32_t* base;
    uint32_t stride, idx, k;
    uint2* over;
};
struct BvhSpill {  // the stack levels of one lane beyond those in shared memory (k >= 1: room for all of them)
    uint2 e[BVH_STACK];
};
BT_DEV BvhStack bvh_lane_stack(uint32_t* stack, BvhSpill& spill, uint32_t k = BVH_STACK_SMEM) {
    BvhStack s;
    s.base = stack;
    s.stride = blockDim.x;
    s.idx = threadIdx.x;
    s.k = min(k, (uint32_t)BVH_STACK_SMEM);
    s.over = spill.e;
    return s;
}
enum : uint32_t { BVH_DONE = 0xffffffffu };  // (leaf bit set: ends the descent loop)
BT_DEV void bvh_begin(BvhTrav& t, float tmax) {
    t.cur = 0;  // node 0 is always an inner node
    t.sp = 0;
    t.h.t = tmax;
    t.h.prim = -1;
    t.h.face = 0;
}
BT_DEV void bvh_push(BvhTrav& t, const BvhStack& st, uint32_t ref, float tn) {
    if (t.sp < st.k) {
        st.base[t.sp * st.stride + st.idx] = ref;
        st.base[(st.k + t.sp) * st.stride + st.idx] = __float_as_uint(tn);
    } else {
        st.over[t.sp - st.k] = make_uint2(ref, __float_as_uint(tn));
    }
    ++t.sp;
}
// pop, skipping subtrees that start beyond the hit found since they were pushed
BT_DEV uint32_t bvh_pop(BvhTrav& t, const BvhStack& st) {
    uint32_t sp = t.sp, cur = BVH_DONE;
    while (sp > st.k) {  // (the tail beyond the shared-memory levels: rarely entered)
        --sp;
        const uint2 e = st.over[sp - st.k];
        if (__uint_as_float(e.y) <= t.h.t) {
            t.sp = sp;
            return e.x;
        }
    }
    while (sp != 0) {
        --sp;
        const uint32_t ref = st.base[sp * st.stride + st.idx];
        if (__uint_as_float(st.base[(st.k + sp) * st.stride + st.idx]) <= t.h.t) {
            cur = ref;
            break;
        }
    }
    t.sp = sp;
    return cur;
}
// The traversal in two kinds of unit, so that a warp can run each kind with the lanes that want it
// (render_body picks the kind more lanes are waiting for; bvh_closest just alternates them):
// bvh_node visits ONE 4-wide inner node (four slab tests off one 128-byte fetch; descend into the
// nearest child hit, push the others far-to-near, or pop), bvh_leaf tests the records of the leaf held in
// t.cur and pops.  t.cur == BVH_DONE when the traversal is complete (t.h is the closest hit).
#define BT_BVH_CSWAP(ta, ra, tb, rb)            \
    {                                           \
        const bool sw = tb < ta;                \
        const float tlo = sw ? tb : ta;         \
        const uint32_t rlo = sw ? rb : ra;      \
        tb = sw ? ta : tb;                      \
        rb = sw ? ra : rb;                      \
        ta = tlo;                               \
        ra = rlo;                               \
    }
// the visit proper, on a fetched node: the near and far planes of the four child boxes per axis (slab), the references
BT_DEV void bvh_node_visit(BvhTrav& t, float4 nx, float4 fx, float4 ny, float4 fy, float4 nz, float4 fz, float4 rf, const BvhStack& st, V3 o,
                           V3 inv, float tmin) {
    const float inf = __int_as_float(0x7f800000);
    uint32_t r0 = __float_as_uint(rf.x), r1 = __float_as_uint(rf.y), r2 = __float_as_uint(rf.z), r3 = __float_as_uint(rf.w);
    float t0 = slab(nx.x, fx.x, ny.x, fy.x, nz.x, fz.x, o, inv, tmin, t.h.t);
    float t1 = slab(nx.y, fx.y, ny.y, fy.y, nz.y, fz.y, o, inv, tmin, t.h.t);
    float t2 = r2 != BVH_EMPTY ? slab(nx.z, fx.z, ny.z, fy.z, nz.z, fz.z, o, inv, tmin, t.h.t) : inf;
    float t3 = r3 != BVH_EMPTY ? slab(nx.w, fx.w, ny.w, fy.w, nz.w, fz.w, o, inv, tmin, t.h.t) : inf;
    if (r1 == BVH_EMPTY) t1 = inf;  // (a node has at least one child; empty slots come last)
    // nearest first (misses, at +inf, sort last)
    BT_BVH_CSWAP(t0, r0, t1, r1)
    BT_BVH_CSWAP(t2, r2, t3, r3)
    BT_BVH_CSWAP(t0, r0, t2, r2)
    BT_BVH_CSWAP(t1, r1, t3, r3)
    BT_BVH_CSWAP(t1, r1, t2, r2)
    if (t0 < inf) {
        if (t.sp + 3 <= st.k) {  // the usual case: straight-line, predicated stores
            uint32_t* e = st.base + t.sp * st.stride + st.idx;
            const uint32_t up = st.k * st.stride;
            if (t3 < inf) {
                e[0] = r3;
                e[up] = __float_as_uint(t3);
                e += st.stride;
            }
            if (t2 < inf) {
                e[0] = r2;
                e[up] = __float_as_uint(t2);
                e += st.stride;
            }
            if (t1 < inf) {
                e[0] = r1;
                e[up] = __float_as_uint(t1);
            }
            t.sp += (t1 < inf ? 1u : 0u) + (t2 < inf ? 1u : 0u) + (t3 < inf ? 1u : 0u);
        } else {
            if (t3 < inf) bvh_push(t, st, r3, t3);
            if (t2 < inf) bvh_push(t, st, r2, t2);
            if (t1 < inf) bvh_push(t, st, r1, t1);
        }
        t.cur = r0;
    } else {
        t.cur = bvh_pop(t, st);
    }
}
// sgn: bit k set when the ray runs towards -k (bvh_signs)
BT_DEV uint32_t bvh_signs(V3 inv) { return (inv.x < 0.0f ? 1u : 0u) | (inv.y < 0.0f ? 2u : 0u) | (inv.z < 0.0f ? 4u : 0u); }
BT_DEV void bvh_node(BvhTrav& t, const float4* __restrict__ nodes, const BvhStack& st, V3 o, V3 inv, uint32_t sgn, float tmin) {
    const float4* n = nodes + t.cur * BVH_STRIDE;
    const uint32_t sx = sgn & 1u, sy = (sgn >> 1) & 1u, sz = sgn >> 2;
    const float4 nx = __ldg(n + sx), fx = __ldg(n + (sx ^ 1u)), ny = __ldg(n + 2 + sy), fy = __ldg(n + 2 + (sy ^ 1u));
    const float4 nz = __ldg(n + 4 + sz), fz = __ldg(n + 4 + (sz ^ 1u));
    bvh_node_visit(t, nx, fx, ny, fy, nz, fz, __ldg(n + 6), st, o, inv, tmin);
}
#undef BT_BVH_CSWAP
// An exact-distance tie (tt == h.t, h.t possibly still the far clip with no hit behind it) is decided as the reference's scan
// order would decide it: the record that comes later in canonical order wins unless it is a cuboid face (strict '<',
// cuboid.rs:97).  Ties are rare (shared cuboid edges, coincident primitives), so the canonical index and the type of the
// two records are read only then -- the common path of a leaf test never touches q4.
BT_DEV bool bvh_tie_take(const float4* __restrict__ prims, int held, int cand) {
    int held_canon = -1;
    bool held_strict = false;
    if (held >= 0) {
        const int m = __float_as_int(__ldg(&prims[held * PRIM_STRIDE + 4].x));
        held_canon = m >> PRIM_CANON_SHIFT;
        held_strict = (m & 3) == PRIM_CUBOID_FACE;
    }
    const int m = __float_as_int(__ldg(&prims[cand * PRIM_STRIDE + 4].x));
    return (m >> PRIM_CANON_SHIFT) > held_canon ? (m & 3) != PRIM_CUBOID_FACE : held_strict;
}
// The records of the leaf held in t.cur, then pop.  The reference tells what the leaf holds (layout.h): all spheres (one
// float4 per test: r^2 is formed as the flattener forms it, one float product), no sphere (four float4), or a mix (the type
// word of every record is read first).  The builder makes leaves of ONE record, so the loops run once except for
// coincident primitives; the sphere loop keeps the next record in flight.
template <bool FLIGHT = false>
BT_DEV void bvh_leaf(BvhTrav& t, const float4* __restrict__ prims, const BvhStack& st, V3 o, V3 d, float tmin) {
    const uint32_t first = t.cur & 0x00ffffffu, count = (t.cur >> 24) & 0x1fu, kind = (t.cur >> 29) & 3u;
    const float4* q = prims + first * PRIM_STRIDE;
    if (kind == BVH_KIND_SPHERES) {
        float4 q0_n = __ldg(q);
        for (uint32_t i = 0; i < count; ++i, q += PRIM_STRIDE) {
            const float4 q0 = q0_n;
            if (i + 1 < count) q0_n = __ldg(q + PRIM_STRIDE);
            float tt;
            if (sphere_roots<FLIGHT>(q0, __fmul_rn(q0.w, q0.w), o, d, tmin, t.h.t, tt)) {
                if (tt < t.h.t || bvh_tie_take(prims, t.h.prim, (int)(first + i))) {  // (tt <= h.t here)
                    t.h.t = tt;
                    t.h.prim = (int)(first + i);
                    t.h.face = 8;
                }
            }
        }
    } else {
        for (uint32_t i = 0; i < count; ++i, q += PRIM_STRIDE) {
            const bool sphere = kind != BVH_KIND_RECTS && (__float_as_int(__ldg(&q[4].x)) & 3) == PRIM_SPHERE;
            const float4 q0 = __ldg(q);
            float tt;
            bool front = true, ok;
            if (sphere)
                ok = sphere_roots<FLIGHT>(q0, __fmul_rn(q0.w, q0.w), o, d, tmin, t.h.t, tt);
            else
                ok = rect_test_q(q0, __ldg(q + 1), __ldg(q + 2), __ldg(q + 3), o, d, tmin, t.h.t, false, tt, front);
            if (ok && (tt < t.h.t || bvh_tie_take(prims, t.h.prim, (int)(first + i)))) {
                t.h.t = tt;
                t.h.prim = (int)(first + i);
                t.h.face = sphere ? 8 : (front ? 0 : 1);
            }
        }
    }
    t.cur = bvh_pop(t, st);
}
template <bool FLIGHT = false>
BT_DEV Hit bvh_closest(const float4* __restrict__ prims, const float4* __restrict__ nodes, uint32_t* stack, V3 o, V3 d,
                       float tmin, float tmax) {
    BvhTrav t;
    BvhSpill spill;
    const BvhStack st = bvh_lane_stack(stack, spill);
    bvh_begin(t, tmax);
    const V3 inv = v3(m_rcp(d.x), m_rcp(d.y), m_rcp(d.z));
    const uint32_t sgn = bvh_signs(inv);
    while (t.cur != BVH_DONE) {  // "while-while": inside a warp the two phases never interleave
        while (!(t.cur & BVH_LEAF)) bvh_node(t, nodes, st, o, inv, sgn, tmin);
        if (t.cur != BVH_DONE) bvh_leaf<FLIGHT>(t, prims, st, o, d, tmin);
    }
    return t.h;
}

struct Surface {  // Manifold (ray.rs:36-47) reduced to what shading reads
    V3 position, normal;
    int face, mat, vol, obj;
    V3 center;   // sphere centre and radius (volume bbox = centre -/+ radius)
    float radius;
};
template <int C = CT_ALL>
BT_DEV Surface resolve_hit(const float4* prims, const Hit& h, V3 o, V3 d) {
    Surface s;
    const float4* q = prims + h.prim * PRIM_STRIDE;
    float4 meta = q[4];
    s.mat = __float_as_int(meta.y);
    s.obj = __float_as_int(meta.w);
    s.vol = -1;
    s.position = xat(o, h.t, d);
    s.center = v3(0.0f, 0.0f, 0.0f);
    s.radius = 0.0f;
    if ((C & CT_SPHERES) && (!(C & CT_RECTS) || (__float_as_int(meta.x) & 3) == PRIM_SPHERE)) {
        float4 q0 = q[0];
        s.vol = (C & CT_VOLUMES) ? __float_as_int(meta.z) : -1;
        s.center = v3(q0);
        s.radius = q0.w;
        if ((C & CT_VOLUMES) && h.face == 2) {  // generate_volume_manifold, sphere.rs:63-83
            s.normal = v3(0.0f, 0.0f, 0.0f);
            s.face = 2;
        } else {            // generate_surface_manifold, sphere.rs:85-119
            V3 normal = m_div(s.position - s.center, q0.w);
            bool front = dot(d, normal) < 0.0f;
            s.normal = front ? normal : -normal;
            s.face = (s.vol >= 0 ? 3 : 0) + (front ? 0 : 1);
        }
    } else if (C & CT_RECTS) {
        V3 n = v3(q[0]);
        s.normal = h.face == 0 ? n : -n;
        s.face = h.face;
    }
    return s;
}

// Object::pdf for the light's primitives (sphere.rs:44-61, rect.rs:92-108); 0 when missed.
// `lights`: the light table (a LIGHT_CUBOID record points at its six face sub-records in it).
template <int C = CT_ALL>
BT_DEV float light_pdf(const float4* prims, const float4* lights, const float4* light, V3 o, V3 d, float tmin, float tmax) {
    int type = __float_as_int(light[0].x);
    if (type == LIGHT_POINT) return 0.0f;
    if ((C & CT_CUBOID_LIGHT) && (C & CT_RECTS) && type == LIGHT_CUBOID) {
        // Cuboid::pdf, cuboid.rs:56-81: the face with the strictly smallest t below clip.max, then
        // Rect::pdf of that face (its re-hit returns the same t and +-n)
        const float4* face = lights + __float_as_int(light[2].z) * LIGHT_STRIDE;
        float best = tmax, shadow = 0.0f;
        bool any = false;
        for (int f = 0; f < 6; ++f, face += LIGHT_STRIDE) {
            const float4* q = prims + __float_as_int(face[0].y) * PRIM_STRIDE;
            float t;
            bool front;
            if (rect_test(q, o, d, tmin, best, true, t, front)) {
                const V3 n = v3(q[0]);
                best = t;
                shadow = face[5].w * fabsf(dot(d, front ? n : -n));
                any = true;
            }
        }
        return any ? (best * best) / shadow : 0.0f;
    }
    const float4* q = prims + __float_as_int(light[0].y) * PRIM_STRIDE;
    if ((C & CT_SPHERES) && (!(C & CT_RECTS) || type == LIGHT_SPHERE)) {
        float t;
        if (!sphere_roots(q[0], q[1].x, o, d, tmin, tmax, t)) return 0.0f;
        return (t * t) / q[1].y;
    }
    if (!(C & CT_RECTS)) return 0.0f;
    float t;
    bool front;
    if (!rect_test(q, o, d, tmin, tmax, false, t, front)) return 0.0f;
    V3 n = v3(q[0]);
    float shadow = q[4].z * fabsf(dot(d, front ? n : -n));
    return (t * t) / shadow;
}
// Object::random_point (object/mod.rs:145-152)
BT_DEV V3 light_point(Rng& rng, const Consts& k, const float4* light) {
    int type = __float_as_int(light[0].x);
    float4 l1 = light[1];
    if (type == LIGHT_SPHERE) return v3(l1) + unit_sphere(rng, k) * l1.w;  // sphere.rs:40-42
    if (type == LIGHT_POINT) return v3(l1);
    float4 l2 = light[2], l3 = light[3], l4 = light[4];
    float x = uniform_f32(rng, l1.w, l3.w);  // rect.rs:82-86
    float y = uniform_f32(rng, l2.w, l4.w);
    V3 local = v3(l1) * x + v3(l2) * y;
    return mat_vec(v3(l3), v3(l4), v3(light[5]), local) + v3(light[6]);
}

// DensityMap::sample(Trilinear), volume.rs:140-167
BT_DEV float density_at(const float* g, int w, int h, int x, int y, int z) { return __ldg(g + (z * h + y) * w + x); }
BT_DEV float density_trilinear(const float4* vol, const float* grids, V3 coord) {
    float4 v0 = vol[0], v1 = vol[1];
    int w = __float_as_int(v0.x), h = __float_as_int(v0.y), dd = __float_as_int(v0.z);
    if (w == 0 || h == 0 || dd == 0) return 0.0f;
    const float* g = grids + __float_as_int(v0.w);
    float cx = fminf(fmaxf(coord.x, 0.0f), 1.0f) * v1.x;
    float cy = fminf(fmaxf(coord.y, 0.0f), 1.0f) * v1.y;
    float cz = fminf(fmaxf(coord.z, 0.0f), 1.0f) * v1.z;
    // floor / ceil / fract of the reference (volume.rs:143-166) for c >= 0: one conversion each way per axis
    // (floor = trunc, ceil = floor + (c != floor), fract = c - trunc) instead of three roundings and two casts
    const int x0 = __float2int_rz(cx), y0 = __float2int_rz(cy), z0 = __float2int_rz(cz);
    const float fx = (float)x0, fy = (float)y0, fz = (float)z0;
    const int x1 = x0 + (cx > fx ? 1 : 0), y1 = y0 + (cy > fy ? 1 : 0), z1 = z0 + (cz > fz ? 1 : 0);
    const float tx = cx - fx, ty = cy - fy, tz = cz - fz;
    float a = density_at(g, w, h, x0, y0, z0), b = density_at(g, w, h, x1, y0, z0);
    float r0 = lerpf(a, b, tx);
    a = density_at(g, w, h, x0, y1, z0); b = density_at(g, w, h, x1, y1, z0);
    float r1 = lerpf(a, b, tx);
    float s0 = lerpf(r0, r1, ty);
    a = density_at(g, w, h, x0, y0, z1); b = density_at(g, w, h, x1, y0, z1);
    r0 = lerpf(a, b, tx);
    a = density_at(g, w, h, x0, y1, z1); b = density_at(g, w, h, x1, y1, z1);
    r1 = lerpf(a, b, tx);
    float s1 = lerpf(r0, r1, ty);
    return lerpf(s0, s1, tz);
}

// ------------------------------------------------------------------------------------------
// environment map (extension, DESIGN.md "Environment map"): the factor sample_root's colour is multiplied by
// ------------------------------------------------------------------------------------------
// Equirectangular texels (float4, .w unused: one LDG.128 per tap), row 0 = the +y pole, the centre column looks
// along -z, columns grow towards +x.  Bilinear; columns wrap, rows clamp.  The test oracle's lookup (tests/oracle_env.cpp) is the same
// operation sequence: every product and sum is rounded on its own (x*_rn intrinsics), so no FMA contraction -- which
// the fast flavour would decide per kernel -- can make the pooled and the lane kernel disagree; the flavours differ
// only in m_sqrt.  x and y are clamped to [-1, W] / [-1, H] before any index is formed (fmaxf returns the non-NaN
// operand, so a NaN lands on -1): no direction -- zero, non-unit, NaN or infinite components -- reads outside the map,
// and the weights are always finite, so a constant map returns its constant exactly (a + (b - a) t = a).
BT_DEV float xlerp(float a, float b, float t) { return __fadd_rn(a, __fmul_rn(__fsub_rn(b, a), t)); }
BT_DEV V3 env_lookup(const float4* env, uint32_t w, uint32_t h, V3 d) {
    const float phi = atan2f(d.x, -d.z), theta = atan2f(d.y, m_sqrt(__fadd_rn(__fmul_rn(d.x, d.x), __fmul_rn(d.z, d.z))));
    const float u = __fadd_rn(0.5f, __fmul_rn(phi, 0.159154943091895335769f)), v = __fsub_rn(0.5f, __fmul_rn(theta, 0.318309886183790671538f));
    const float x = fminf(fmaxf(__fsub_rn(__fmul_rn(u, (float)w), 0.5f), -1.0f), (float)w);
    const float y = fminf(fmaxf(__fsub_rn(__fmul_rn(v, (float)h), 0.5f), -1.0f), (float)h);
    const float fx = floorf(x), fy = floorf(y), tx = __fsub_rn(x, fx), ty = __fsub_rn(y, fy);
    const uint32_t c0 = fx < 0.0f ? w - 1 : min((uint32_t)fx, w - 1), c1 = c0 + 1 == w ? 0 : c0 + 1;
    const uint32_t r0 = fy < 0.0f ? 0 : min((uint32_t)fy, h - 1), r1 = fy < 0.0f ? 0 : min((uint32_t)fy + 1, h - 1);
    const float4 a = __ldg(env + r0 * w + c0), b = __ldg(env + r0 * w + c1), c = __ldg(env + r1 * w + c0), e = __ldg(env + r1 * w + c1);
    const V3 top = v3(xlerp(a.x, b.x, tx), xlerp(a.y, b.y, tx), xlerp(a.z, b.z, tx));
    const V3 bot = v3(xlerp(c.x, e.x, tx), xlerp(c.y, e.y, tx), xlerp(c.z, e.z, tx));
    return v3(xlerp(top.x, bot.x, ty), xlerp(top.y, bot.y, ty), xlerp(top.z, bot.z, ty));
}

// ------------------------------------------------------------------------------------------
// camera (mod.rs:272-302, ray.rs:103-137)
// ------------------------------------------------------------------------------------------
BT_DEV V3 with_frustum_dir(float yfov, float xfov, float u, float v) {
    float yrot = xfov * 0.5f * -u;
    float xrot = yfov * 0.5f * -v;
    float sy, cy, sx, cx;
    bt_sincos(yrot * 0.5f, &sy, &cy);
    bt_sincos(xrot * 0.5f, &sx, &cx);
    float qx = cy * sx, qy = sy * cx, qz = -(sy * sx), qw = cy * cx;
    V3 b = v3(qx, qy, qz);
    V3 vv = v3(0.0f, 0.0f, -1.0f);
    float b2 = dot(b, b);
    float s1 = qw * qw - b2;
    float s2 = dot(vv, b) * 2.0f;
    float s3 = qw * 2.0f;
    return (vv * s1 + b * s2) + cross(b, vv) * s3;
}
// (sub_i, sub_j): the sub-pixel of this path, i fastest (mod.rs:70-106)
BT_DEV void camera_ray(const CameraBlock& cam, const Consts& k, Rng& rng, uint32_t x, uint32_t y, uint32_t sub_i, uint32_t sub_j,
                       V3& origin, V3& direction) {
    float v = (float)y * cam.pixel_height - 1.0f;
    float u = (float)x * cam.pixel_width - 1.0f;
    float u_sub = 0.0f, v_sub = 0.0f;
    if (cam.sub_width != 0.0f) {
        u_sub = (float)sub_i * cam.sub_width;
        v_sub = (float)sub_j * cam.sub_width;
    }
    float u_offset = u_sub * cam.pixel_width + uniform_f32(rng, cam.su_low, cam.su_scale);
    float v_offset = v_sub * cam.pixel_height + uniform_f32(rng, cam.sv_low, cam.sv_scale);
    u = u + u_offset;
    v = v + v_offset;
    V3 dir_cam = with_frustum_dir(cam.yfov, cam.xfov, u, v);
    V3 c0 = v3(cam.m[0], cam.m[1], cam.m[2]), c1 = v3(cam.m[3], cam.m[4], cam.m[5]), c2 = v3(cam.m[6], cam.m[7], cam.m[8]);
    V3 t = v3(cam.t[0], cam.t[1], cam.t[2]);
    V3 o = t + v3(0.0f, 0.0f, 0.0f);
    V3 d = normalize_a(normalize_or_zero_s(mat_vec(c0, c1, c2, dir_cam)));
    if (cam.has_focus) {
        float angle = uniform_f32(rng, 0.0f, k.tau_scale);  // UnitDisk, distr.rs:105-138
        float r = uniform_f32(rng, 0.0f, k.one_scale);
        float s, c;
        bt_sincos(angle, &s, &c);
        V3 dx = v3(cam.disk_x[0], cam.disk_x[1], cam.disk_x[2]), dy = v3(cam.disk_y[0], cam.disk_y[1], cam.disk_y[2]);
        V3 defocus = (dx * c + dy * s) * r;
        V3 defocus_offset = mat_vec(c0, c1, c2, defocus * cam.aperture);
        float frac_f_z = cam.focus / fabsf(dir_cam.z);
        o = o + defocus_offset;
        d = normalize_a(d * frac_f_z - defocus_offset);
    }
    origin = o;
    direction = d;
}

// ------------------------------------------------------------------------------------------
// geodesic stepper (extension; DESIGN.md "Geodesic model").  FMAs are explicit.
// ------------------------------------------------------------------------------------------
// The lens table is read through a provider: LensShared walks the shared-memory records,
// LensRegs<N> holds N masses in registers with the loop fully unrolled (no LDS, no loop
// overhead in the stepper's inner loop).
struct LensShared {
    const float4* p;
    int count;
    enum { UNROLL = 4 };
    BT_DEV int n() const { return count; }
    BT_DEV float4 e0(int m) const { return p[m * LENS_STRIDE]; }
    BT_DEV float4 e1(int m) const { return p[m * LENS_STRIDE + 1]; }
};
template <int N>
struct LensRegs {
    float4 a[N], b[N];
    enum { UNROLL = N };
    BT_DEV explicit LensRegs(const float4* p) {
#pragma unroll
        for (int m = 0; m < N; ++m) {
            a[m] = p[m * LENS_STRIDE];
            b[m] = p[m * LENS_STRIDE + 1];
        }
    }
    BT_DEV int n() const { return N; }
    BT_DEV float4 e0(int m) const { return a[m]; }
    BT_DEV float4 e1(int m) const { return b[m]; }
};
// MUFU.RSQ without the denormal-input fix-up of rsqrtf() (|d|^2 is never denormal here)
BT_DEV float rsqrt_approx(float x) {
    float r;
    asm("rsqrt.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
    return r;
}
// The stepper's vectors as one register pair (x, y) and a single z: the x and y components of every vector operation
// go through one paired FP32 instruction (FFMA2 / FADD2 / FMUL2, sm_100), z through a scalar one.  Each component is
// the operation the scalar code would perform, correctly rounded on its own (the paired intrinsics round per component
// like __fmaf_rn / __fadd_rn / __fmul_rn), so the pairing changes no bit.  The pairs cost no MOV as long as the
// pair of a value stays the same pair: the stepper, the chord and the pooled STEP loop all keep this one layout.
struct P3 {
    float2 xy;
    float z;
};
BT_DEV P3 p3(float2 xy, float z) { P3 r = {xy, z}; return r; }
BT_DEV P3 p3(V3 a) { return p3(make_float2(a.x, a.y), a.z); }
BT_DEV P3 p3(float4 q) { return p3(make_float2(q.x, q.y), q.z); }
BT_DEV V3 v3(P3 a) { return v3(a.xy.x, a.xy.y, a.z); }
BT_DEV float2 f2(float a) { return make_float2(a, a); }
BT_DEV P3 operator+(P3 a, P3 b) { return p3(__fadd2_rn(a.xy, b.xy), __fadd_rn(a.z, b.z)); }
// a - b as a + (-b): the same IEEE operation (a FADD2 with a negated operand)
BT_DEV P3 operator-(P3 a, P3 b) { return p3(__fadd2_rn(a.xy, make_float2(-b.xy.x, -b.xy.y)), __fsub_rn(a.z, b.z)); }
BT_DEV P3 axpy(float a, P3 x, P3 y) { return p3(__ffma2_rn(f2(a), x.xy, y.xy), __fmaf_rn(a, x.z, y.z)); }
// Per-step cache of d0_m = x - c_m, filled by the k1 evaluation and reused by the three stage
// evaluations (register-resident tables only; the shared-memory walk recomputes it).
template <class L>
struct D0Cache {
    enum { CACHED = 0 };
    BT_DEV P3 get(int, P3 x, float4 e0) const { return x - p3(e0); }
    BT_DEV void put(int, P3) {}
};
template <int N>
struct D0Cache<LensRegs<N> > {
    enum { CACHED = 1 };
    P3 d[N];
    BT_DEV P3 get(int m, P3, float4) const { return d[m]; }
    BT_DEV void put(int m, P3 v) { d[m] = v; }
};
// a = sum_m -(3/2) r_s |d x v|^2 d / |d|^5 evaluated at x + a*w, written as d = fma(a, w, x - c)
// (STAGE 0: a = 0, d = x - c).  INFO 1 also returns min |d|; INFO 2 adds the capture / far flags.
// d, w, v and the sum are paired (P3); |d|^2, the cross product and what follows from it stay scalar: each is a chain
// whose x and y terms feed one another, or needs pairs such as (y, z) that the layout does not hold.
template <int INFO, bool EXACT, int STAGE, class L>
BT_DEV P3 lens_accel(const L& lens, D0Cache<L>& cache, P3 x, float a, P3 w, P3 v, float& rmin, bool& captured, bool& far) {
    P3 acc = p3(make_float2(0.0f, 0.0f), 0.0f);
    if (INFO >= 1) rmin = __int_as_float(0x7f800000);
    if (INFO >= 2) {
        captured = false;
        far = true;
    }
    const int n_lens = lens.n();
#pragma unroll(L::UNROLL)
    for (int m = 0; m < n_lens; ++m) {
        const float4 e0 = lens.e0(m);  // (c.xyz, -1.5 r_s)
        P3 d;
        if (STAGE == 0) {
            d = x - p3(e0);
            cache.put(m, d);
        } else {
            d = axpy(a, w, cache.get(m, x, e0));
        }
        const float dx = d.xy.x, dy = d.xy.y, dz = d.z, vx = v.xy.x, vy = v.xy.y, vz = v.z;
        float r2 = fmaf(dz, dz, fmaf(dy, dy, dx * dx));
        float lx = fmaf(dy, vz, -(dz * vy));
        float ly = fmaf(dz, vx, -(dx * vz));
        float lz = fmaf(dx, vy, -(dy * vx));
        float h2 = fmaf(lz, lz, fmaf(ly, ly, lx * lx));
        // fast: MUFU.RSQ (<= 2 ulp); exact: correctly rounded, bit-identical to the CPU oracle
        float inv = EXACT ? __frsqrt_rn(r2) : rsqrt_approx(r2);
        float inv2 = inv * inv;
        float inv5 = (inv2 * inv2) * inv;
        float s = (e0.w * h2) * inv5;
        acc = axpy(s, d, acc);
        if (INFO >= 1) {
            float r = r2 * inv;
            rmin = fminf(rmin, r);
            if (INFO >= 2) {
                const float4 e1 = lens.e1(m);  // (r_s, r_far * r_s, -, -)
                if (r < e1.x) captured = true;
                if (r > e1.y) {  // beyond r_far of this mass (rare): receding?
                    const float dv = fmaf(dz, vz, fmaf(dy, vy, dx * vx));
                    if (!(dv > 0.0f)) far = false;
                } else {
                    far = false;
                }
            }
        }
    }
    return acc;
}
// classic RK4 given k1 = accel(x, v) (whose evaluation filled `cache`)
template <bool EXACT, class L>
BT_DEV void rk4_from_k1(const L& lens, D0Cache<L>& cache, P3& x, P3& v, P3 k1, float h) {
    float hh = 0.5f * h, h6 = h * (float)(1.0 / 6.0);
    float ru;
    bool bu;
    P3 v2 = axpy(hh, k1, v);
    P3 k2 = lens_accel<0, EXACT, 1>(lens, cache, x, hh, v, v2, ru, bu, bu);
    P3 v3_ = axpy(hh, k2, v);
    P3 k3 = lens_accel<0, EXACT, 1>(lens, cache, x, hh, v2, v3_, ru, bu, bu);
    P3 v4 = axpy(h, k3, v);
    P3 k4 = lens_accel<0, EXACT, 1>(lens, cache, x, h, v3_, v4, ru, bu, bu);
    P3 sv = axpy(2.0f, v2 + v3_, v + v4);
    P3 sk = axpy(2.0f, k2 + k3, k1 + k4);
    x = axpy(h6, sv, x);
    v = axpy(h6, sk, v);
}
BT_DEV float step_size(float kappa, float h_min, float h_max, float rmin) { return fminf(fmaxf(kappa * rmin, h_min), h_max); }
// chord direction and length.  EXACT: IEEE square root and reciprocal (the oracle's values);
// otherwise one MUFU.RSQ (<= 2 ulp), like the stepper's own 1/|d|.
template <bool EXACT>
BT_DEV V3 normalize_fma(P3 a, float* len_out) {
    const float ax = a.xy.x, ay = a.xy.y;
    float l2 = fmaf(a.z, a.z, fmaf(ay, ay, ax * ax));
    float inv = EXACT ? 1.0f / sqrtf(l2) : rsqrt_approx(l2);
    if (len_out) *len_out = l2 * inv;
    return v3(ax * inv, ay * inv, a.z * inv);
}

}  // namespace bt
