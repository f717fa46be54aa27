// scene.cpp -- Scene wire format (serde_json-compatible), scene-graph update, and the flattener.
//
// Wire format: reference src/scene/mod.rs:16-20,84-90 (Scene, Collection), src/scene/object/mod.rs
// :23-41,247-256 (Object, ObjectFlags, ObjectKind), src/scene/object/transform.rs:10-15,
// src/scene/object/{sphere.rs:11-16,rect.rs:11-19,cuboid.rs:12-15,camera.rs:3-10},
// src/scene/data/mod.rs:9-15,46-51, src/scene/data/material.rs:22-44, volume.rs:21-24,75-82.
// serde's externally-tagged enums: unit variants are strings ("Empty"), others {"Variant": {...}};
// newtype structs (ObjectRef, DataRef) are bare integers; HashMap<u64-newtype, V> keys are strings.
#include "scene.hpp"

#include <zlib.h>

#include <algorithm>
#include <charconv>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <limits>
#include <memory>

namespace bt {

// ------------------------------------------------------------------------------------------
// minimal JSON
// ------------------------------------------------------------------------------------------
namespace {

struct JValue;
typedef std::shared_ptr<JValue> JPtr;
struct JValue {
    enum Type { Null, Bool, Number, String, Array, Object } type;
    bool b;
    std::string text;  // number token or string contents
    std::vector<JPtr> arr;
    std::vector<std::pair<std::string, JPtr> > obj;
    JValue() : type(Null), b(false) {}
    const JValue* get(const char* key) const {
        for (size_t i = 0; i < obj.size(); ++i)
            if (obj[i].first == key) return obj[i].second.get();
        return 0;
    }
};

struct Parser {
    const char* p;
    const char* end;
    [[noreturn]] void fail(const char* what) const {
        char buf[160];
        std::snprintf(buf, sizeof buf, "%s at byte %ld", what, (long)(p - start));
        throw ParseError(buf);
    }
    const char* start;
    int depth = 0;  // serde_json's recursion limit: 128 nested arrays / objects, then an error (never a stack overflow)
    struct Nest {
        Parser& ps;
        explicit Nest(Parser& p_) : ps(p_) {
            if (++ps.depth > 128) ps.fail("recursion limit exceeded");
        }
        ~Nest() { --ps.depth; }
    };
    void ws() {
        while (p < end && (*p == ' ' || *p == '\n' || *p == '\t' || *p == '\r')) ++p;
    }
    JPtr value() {
        ws();
        if (p >= end) fail("EOF while parsing a value");
        JPtr v(new JValue());
        char c = *p;
        if (c == '{') {
            Nest nest(*this);
            v->type = JValue::Object;
            ++p;
            ws();
            if (p < end && *p == '}') {
                ++p;
                return v;
            }
            for (;;) {
                ws();
                if (p >= end || *p != '"') fail("key must be a string");
                std::string k = string();
                ws();
                if (p >= end || *p != ':') fail("expected `:`");
                ++p;
                v->obj.push_back(std::make_pair(k, value()));
                ws();
                if (p < end && *p == ',') {
                    ++p;
                    continue;
                }
                if (p < end && *p == '}') {
                    ++p;
                    return v;
                }
                fail("expected `,` or `}`");
            }
        }
        if (c == '[') {
            Nest nest(*this);
            v->type = JValue::Array;
            ++p;
            ws();
            if (p < end && *p == ']') {
                ++p;
                return v;
            }
            for (;;) {
                v->arr.push_back(value());
                ws();
                if (p < end && *p == ',') {
                    ++p;
                    continue;
                }
                if (p < end && *p == ']') {
                    ++p;
                    return v;
                }
                fail("expected `,` or `]`");
            }
        }
        if (c == '"') {
            v->type = JValue::String;
            v->text = string();
            return v;
        }
        if (c == 't' && end - p >= 4 && !std::memcmp(p, "true", 4)) {
            v->type = JValue::Bool;
            v->b = true;
            p += 4;
            return v;
        }
        if (c == 'f' && end - p >= 5 && !std::memcmp(p, "false", 5)) {
            v->type = JValue::Bool;
            p += 5;
            return v;
        }
        if (c == 'n' && end - p >= 4 && !std::memcmp(p, "null", 4)) {
            p += 4;
            return v;
        }
        if (c == '-' || (c >= '0' && c <= '9')) {
            const char* s = p;
            if (*p == '-') ++p;
            while (p < end && ((*p >= '0' && *p <= '9') || *p == '.' || *p == 'e' || *p == 'E' || *p == '+' || *p == '-')) ++p;
            v->type = JValue::Number;
            v->text.assign(s, p);
            return v;
        }
        fail("expected value");
    }
    std::string string() {
        ++p;  // opening quote
        std::string out;
        while (p < end && *p != '"') {
            if (*p == '\\') {
                ++p;
                if (p >= end) fail("EOF while parsing a string");
                switch (*p) {
                    case 'n': out += '\n'; break;
                    case 't': out += '\t'; break;
                    case 'r': out += '\r'; break;
                    case 'b': out += '\b'; break;
                    case 'f': out += '\f'; break;
                    case 'u': {
                        if (end - p < 5) fail("invalid escape");
                        unsigned cp = (unsigned)std::strtoul(std::string(p + 1, p + 5).c_str(), 0, 16);
                        p += 4;
                        if (cp < 0x80) out += (char)cp;
                        else if (cp < 0x800) { out += (char)(0xC0 | (cp >> 6)); out += (char)(0x80 | (cp & 0x3F)); }
                        else { out += (char)(0xE0 | (cp >> 12)); out += (char)(0x80 | ((cp >> 6) & 0x3F)); out += (char)(0x80 | (cp & 0x3F)); }
                        break;
                    }
                    default: out += *p; break;
                }
                ++p;
            } else {
                out += *p++;
            }
        }
        if (p >= end) fail("EOF while parsing a string");
        ++p;
        return out;
    }
};

const JValue& need(const JValue& v, const char* key) {
    if (v.type != JValue::Object) throw ParseError(std::string("expected a map with field `") + key + "`");
    const JValue* r = v.get(key);
    if (!r) throw ParseError(std::string("missing field `") + key + "`");
    return *r;
}
float as_f32(const JValue& v) {  // serde_json: parsed as f64, cast to f32
    if (v.type != JValue::Number) throw ParseError("invalid type: expected f32");
    return (float)std::strtod(v.text.c_str(), 0);
}
uint64_t as_u64(const JValue& v) {
    if (v.type != JValue::Number || v.text.empty() || v.text[0] == '-' || v.text.find_first_of(".eE") != std::string::npos)
        throw ParseError("invalid type: expected u64");
    return std::strtoull(v.text.c_str(), 0, 10);
}
void as_vec3(const JValue& v, float out[3]) {
    if (v.type != JValue::Array || v.arr.size() != 3) throw ParseError("invalid length, expected 3 floats");
    for (int i = 0; i < 3; ++i) out[i] = as_f32(*v.arr[i]);
}
Affine as_affine(const JValue& v) {
    if (v.type != JValue::Array || v.arr.size() != 12) throw ParseError("invalid length, expected 12 floats");
    Affine a;
    for (int i = 0; i < 12; ++i) a.f[i] = as_f32(*v.arr[i]);
    return a;
}
Rect as_rect(const JValue& v) {
    Rect r;
    r.material = as_u64(need(v, "material"));
    r.half_width = as_f32(need(v, "half_width"));
    r.half_height = as_f32(need(v, "half_height"));
    as_vec3(need(v, "x"), r.x);
    as_vec3(need(v, "y"), r.y);
    as_vec3(need(v, "z"), r.z);
    return r;
}
const JValue* opt(const JValue& v, const char* key) {
    const JValue* r = v.type == JValue::Object ? v.get(key) : 0;
    return (r && r->type != JValue::Null) ? r : 0;
}

Object parse_object(const JValue& v) {
    Object o = Object();
    if (const JValue* r = opt(v, "object_ref")) {
        o.has_object_ref = true;
        o.object_ref = as_u64(*r);
    }
    if (const JValue* t = opt(v, "tag")) {
        if (t->type != JValue::String) throw ParseError("invalid type: tag must be a string");
        o.has_tag = true;
        o.tag = t->text;
    }
    o.flags = (uint32_t)as_u64(need(need(v, "flags"), "bits"));
    const JValue& tf = need(v, "transform");
    o.transform_world = as_affine(need(tf, "transform_world"));
    o.transform_local = as_affine(need(tf, "transform_local"));
    if (const JValue* p = opt(tf, "transform_parent")) {
        o.has_parent = true;
        o.transform_parent = as_affine(*p);
    }
    if (const JValue* c = opt(v, "children")) {
        o.has_children = true;
        for (size_t i = 0; i < c->arr.size(); ++i) o.children.push_back(as_u64(*c->arr[i]));
    }
    const JValue& inner = need(v, "inner");
    if (inner.type == JValue::String) {
        if (inner.text != "Empty") throw ParseError("unknown variant `" + inner.text + "`");
        o.kind = OBJ_EMPTY;
    } else if (inner.type == JValue::Object && inner.obj.size() == 1) {
        const std::string& k = inner.obj[0].first;
        const JValue& b = *inner.obj[0].second;
        if (k == "Empty") {
            o.kind = OBJ_EMPTY;
        } else if (k == "Camera") {
            o.kind = OBJ_CAMERA;
            o.camera.sensor_size = as_f32(need(b, "sensor_size"));
            o.camera.focal_length = as_f32(need(b, "focal_length"));
            o.camera.aspect_ratio = as_f32(need(b, "aspect_ratio"));
            o.camera.fstop = as_f32(need(b, "fstop"));
            if (const JValue* f = opt(b, "focus")) {
                o.camera.has_focus = true;
                o.camera.focus = as_f32(*f);
            }
        } else if (k == "Sphere") {
            o.kind = OBJ_SPHERE;
            o.material = as_u64(need(b, "material"));
            if (const JValue* vol = opt(b, "volume")) {
                o.has_volume = true;
                o.volume = as_u64(*vol);
            }
            o.radius = as_f32(need(b, "radius"));
        } else if (k == "Rect") {
            o.kind = OBJ_RECT;
            o.rect = as_rect(b);
        } else if (k == "Cuboid") {
            o.kind = OBJ_CUBOID;
            const JValue& faces = need(b, "faces");
            if (faces.type != JValue::Array || faces.arr.size() != 6) throw ParseError("invalid length, expected an array of length 6");
            for (int i = 0; i < 6; ++i) {
                const JValue& pair = *faces.arr[i];
                if (pair.type != JValue::Array || pair.arr.size() != 2) throw ParseError("invalid length, expected a tuple of size 2");
                as_vec3(*pair.arr[0], o.face_offset[i]);
                o.faces[i] = as_rect(*pair.arr[1]);
            }
        } else {
            throw ParseError("unknown variant `" + k + "`, expected one of `Empty`, `Camera`, `Sphere`, `Rect`, `Cuboid`");
        }
    } else {
        throw ParseError("invalid type for ObjectKind");
    }
    return o;
}

Data parse_data(const JValue& v) {
    Data d = Data();
    const JValue& inner = need(v, "inner");
    if (inner.type != JValue::Object || inner.obj.size() != 1) throw ParseError("invalid type for DataKind");
    const std::string& k = inner.obj[0].first;
    const JValue& b = *inner.obj[0].second;
    if (k == "Material") {
        d.kind = DATA_MATERIAL;
        if (b.type != JValue::Object || b.obj.size() != 1) throw ParseError("invalid type for Material");
        const std::string& mk = b.obj[0].first;
        const JValue& m = *b.obj[0].second;
        static const char* names[5] = {"Flat", "Diffuse", "Metallic", "Glass", "Emissive"};
        d.mat_kind = -1;
        for (int i = 0; i < 5; ++i)
            if (mk == names[i]) d.mat_kind = i;
        if (d.mat_kind < 0) throw ParseError("unknown variant `" + mk + "`");
        const JValue& a = need(m, "albedo");
        d.albedo[0] = as_f32(need(a, "r"));
        d.albedo[1] = as_f32(need(a, "g"));
        d.albedo[2] = as_f32(need(a, "b"));
        if (d.mat_kind == MAT_DIFFUSE || d.mat_kind == MAT_METALLIC || d.mat_kind == MAT_GLASS) d.roughness = as_f32(need(m, "roughness"));
        if (d.mat_kind == MAT_GLASS) d.ior = as_f32(need(m, "ior"));
        if (d.mat_kind == MAT_EMISSIVE) d.intensity = as_f32(need(m, "intensity"));
    } else if (k == "Volume") {
        d.kind = DATA_VOLUME;
        if (b.type != JValue::Object || b.obj.size() != 1 || b.obj[0].first != "DensityMap") throw ParseError("unknown Volume variant");
        const JValue& m = *b.obj[0].second;
        d.width = as_u64(need(m, "width"));
        d.height = as_u64(need(m, "height"));
        d.depth = as_u64(need(m, "depth"));
        as_vec3(need(m, "size"), d.size);
        const JValue& buf = need(m, "buffer");
        if (buf.type != JValue::Array) throw ParseError("invalid type: buffer must be a sequence");
        d.buffer.reserve(buf.arr.size());
        for (size_t i = 0; i < buf.arr.size(); ++i) d.buffer.push_back(as_f32(*buf.arr[i]));
    } else {
        throw ParseError("unknown variant `" + k + "`, expected `Material` or `Volume`");
    }
    return d;
}

std::string gunzip(const void* bytes, size_t n) {
    z_stream zs;
    std::memset(&zs, 0, sizeof zs);
    if (inflateInit2(&zs, 16 + MAX_WBITS) != Z_OK) throw ParseError("zlib init failed");
    zs.next_in = (Bytef*)bytes;
    zs.avail_in = (uInt)n;
    std::string out;
    char buf[1 << 15];
    int rc;
    do {
        zs.next_out = (Bytef*)buf;
        zs.avail_out = sizeof buf;
        rc = inflate(&zs, Z_NO_FLUSH);
        if (rc != Z_OK && rc != Z_STREAM_END) {
            inflateEnd(&zs);
            throw ParseError("corrupt deflate stream");
        }
        out.append(buf, sizeof buf - zs.avail_out);
    } while (rc != Z_STREAM_END);
    inflateEnd(&zs);
    return out;
}

// ---- writer ----
void put_f32(std::string& s, float v) {
    if (!std::isfinite(v)) {  // serde_json writes non-finite floats as null
        s += "null";
        return;
    }
    char buf[48];
    std::to_chars_result r = std::to_chars(buf, buf + sizeof buf, v);
    std::string t(buf, r.ptr);
    if (t.find_first_of(".eEn") == std::string::npos) t += ".0";
    s += t;
}
void put_u64(std::string& s, uint64_t v) { s += std::to_string(v); }
void put_vec3(std::string& s, const float v[3]) {
    s += '[';
    for (int i = 0; i < 3; ++i) {
        if (i) s += ',';
        put_f32(s, v[i]);
    }
    s += ']';
}
void put_affine(std::string& s, const Affine& a) {
    s += '[';
    for (int i = 0; i < 12; ++i) {
        if (i) s += ',';
        put_f32(s, a.f[i]);
    }
    s += ']';
}
void put_string(std::string& s, const std::string& v) {
    s += '"';
    for (size_t i = 0; i < v.size(); ++i) {
        unsigned char c = (unsigned char)v[i];
        if (c == '"' || c == '\\') { s += '\\'; s += (char)c; }
        else if (c == '\n') s += "\\n";
        else if (c == '\t') s += "\\t";
        else if (c == '\r') s += "\\r";
        else if (c < 0x20) { char b[8]; std::snprintf(b, sizeof b, "\\u%04x", c); s += b; }
        else s += (char)c;
    }
    s += '"';
}
void put_rect(std::string& s, const Rect& r) {
    s += "{\"material\":";
    put_u64(s, r.material);
    s += ",\"half_width\":";
    put_f32(s, r.half_width);
    s += ",\"half_height\":";
    put_f32(s, r.half_height);
    s += ",\"x\":";
    put_vec3(s, r.x);
    s += ",\"y\":";
    put_vec3(s, r.y);
    s += ",\"z\":";
    put_vec3(s, r.z);
    s += '}';
}

// ---- f32 helpers in glam's operation order (host code is built with -ffp-contract=off) ----
inline void mat_vec(const Affine& a, const float v[3], float out[3]) {  // Mat3A * Vec3A
    for (int i = 0; i < 3; ++i) {
        float r = a.f[i] * v[0];
        r = r + a.f[3 + i] * v[1];
        r = r + a.f[6 + i] * v[2];
        out[i] = r;
    }
}
inline float f32_dec(float x) {
    uint32_t b;
    std::memcpy(&b, &x, 4);
    b -= 1;
    std::memcpy(&x, &b, 4);
    return x;
}
inline float4 f4(float x, float y, float z, float w) {
    float4 r;
    r.x = x; r.y = y; r.z = z; r.w = w;
    return r;
}
inline float as_f(uint32_t u) {
    float f;
    std::memcpy(&f, &u, 4);
    return f;
}
inline uint32_t as_u(float f) {
    uint32_t u;
    std::memcpy(&u, &f, 4);
    return u;
}

}  // namespace

float uniform_scale(float low, float high) {  // rand 0.8.5 UniformFloat::new
    const float max_rand = 1.0f - 1.1920929e-07f;
    float scale = high - low;
    while (scale * max_rand + low >= high) scale = f32_dec(scale);
    return scale;
}
float uniform_scale_inclusive(float low, float high) {  // UniformFloat::new_inclusive
    const float max_rand = 1.0f - 1.1920929e-07f;
    float scale = (high - low) / max_rand;
    while (scale * max_rand + low > high) scale = f32_dec(scale);
    return scale;
}

Affine affine_mul(const Affine& a, const Affine& b) {  // glam Affine3A * Affine3A
    Affine r;
    mat_vec(a, &b.f[0], &r.f[0]);
    mat_vec(a, &b.f[3], &r.f[3]);
    mat_vec(a, &b.f[6], &r.f[6]);
    float t[3];
    mat_vec(a, &b.f[9], t);
    for (int i = 0; i < 3; ++i) r.f[9 + i] = t[i] + a.f[9 + i];
    return r;
}
Affine affine_inverse(const Affine& a) {  // glam Mat3A::inverse (cross / det, transposed)
    const float* x = &a.f[0];
    const float* y = &a.f[3];
    const float* z = &a.f[6];
    float t0[3] = {y[1] * z[2] - z[1] * y[2], y[2] * z[0] - z[2] * y[0], y[0] * z[1] - z[0] * y[1]};
    float t1[3] = {z[1] * x[2] - x[1] * z[2], z[2] * x[0] - x[2] * z[0], z[0] * x[1] - x[0] * z[1]};
    float t2[3] = {x[1] * y[2] - y[1] * x[2], x[2] * y[0] - y[2] * x[0], x[0] * y[1] - y[0] * x[1]};
    float det = (z[0] * t2[0] + z[1] * t2[1]) + z[2] * t2[2];
    float inv_det = 1.0f / det;
    Affine r;
    for (int i = 0; i < 3; ++i) {
        r.f[0 + i] = (i == 0 ? t0[0] : i == 1 ? t1[0] : t2[0]) * inv_det;
        r.f[3 + i] = (i == 0 ? t0[1] : i == 1 ? t1[1] : t2[1]) * inv_det;
        r.f[6 + i] = (i == 0 ? t0[2] : i == 1 ? t1[2] : t2[2]) * inv_det;
    }
    float t[3];
    mat_vec(r, &a.f[9], t);
    for (int i = 0; i < 3; ++i) r.f[9 + i] = -t[i];
    return r;
}

// ------------------------------------------------------------------------------------------
// Scene
// ------------------------------------------------------------------------------------------
Scene Scene::from_json(const void* bytes, size_t n) {
    std::string text;
    const unsigned char* b = (const unsigned char*)bytes;
    if (n >= 2 && b[0] == 0x1f && b[1] == 0x8b)
        text = gunzip(bytes, n);
    else
        text.assign((const char*)bytes, n);
    Parser ps;
    ps.p = ps.start = text.data();
    ps.end = text.data() + text.size();
    JPtr root = ps.value();
    ps.ws();
    if (ps.p != ps.end) ps.fail("trailing characters");

    Scene s = Scene();
    const JValue& r = *root;
    if (const JValue* roots = opt(r, "roots"))
        for (size_t i = 0; i < roots->arr.size(); ++i) s.roots.push_back(as_u64(*roots->arr[i]));
    s.root_material = as_u64(need(r, "root_material"));
    const JValue& objs = need(r, "objects");
    const JValue& ocoll = need(objs, "collection");
    if (ocoll.type != JValue::Object) throw ParseError("invalid type: objects.collection must be a map");
    for (size_t i = 0; i < ocoll.obj.size(); ++i) {
        char* endp = 0;
        uint64_t key = std::strtoull(ocoll.obj[i].first.c_str(), &endp, 10);
        if (ocoll.obj[i].first.empty() || *endp) throw ParseError("invalid ObjectRef key `" + ocoll.obj[i].first + "`");
        s.objects[key] = parse_object(*ocoll.obj[i].second);
    }
    s.objects_next_key = as_u64(need(objs, "next_key"));
    const JValue& datas = need(r, "data");
    const JValue& dcoll = need(datas, "collection");
    if (dcoll.type != JValue::Object) throw ParseError("invalid type: data.collection must be a map");
    for (size_t i = 0; i < dcoll.obj.size(); ++i) {
        char* endp = 0;
        uint64_t key = std::strtoull(dcoll.obj[i].first.c_str(), &endp, 10);
        if (dcoll.obj[i].first.empty() || *endp) throw ParseError("invalid DataRef key `" + dcoll.obj[i].first + "`");
        s.data[key] = parse_data(*dcoll.obj[i].second);
    }
    s.data_next_key = as_u64(need(datas, "next_key"));
    s.lens_config.kappa = 0.05f;
    s.lens_config.h_min = 0.02f;
    s.lens_config.h_max = 5.0f;
    s.lens_config.r_far = 500.0f;
    s.lens_config.max_steps = 4096;
    s.lens_config.flags = 0;
    if (const JValue* lenses = opt(r, "lenses")) {  // extension; serde ignores unknown keys
        if (lenses->type != JValue::Array) throw ParseError("invalid type: lenses must be a sequence");
        for (size_t i = 0; i < lenses->arr.size(); ++i) {
            const JValue& l = *lenses->arr[i];
            if (l.type != JValue::Array || l.arr.size() != 4) throw ParseError("invalid length, expected [x, y, z, r_s]");
            Lens ln;
            for (int k = 0; k < 3; ++k) ln.c[k] = as_f32(*l.arr[k]);
            ln.rs = as_f32(*l.arr[3]);
            s.lenses.push_back(ln);
        }
    }
    return s;
}

std::string Scene::to_json() const {
    std::string s;
    s += "{\"roots\":[";
    for (size_t i = 0; i < roots.size(); ++i) {
        if (i) s += ',';
        put_u64(s, roots[i]);
    }
    s += "],\"root_material\":";
    put_u64(s, root_material);
    s += ",\"objects\":{\"collection\":{";
    bool first = true;
    for (std::map<uint64_t, Object>::const_iterator it = objects.begin(); it != objects.end(); ++it) {
        const Object& o = it->second;
        if (!first) s += ',';
        first = false;
        s += '"';
        put_u64(s, it->first);
        s += "\":{\"object_ref\":";
        if (o.has_object_ref) put_u64(s, o.object_ref); else s += "null";
        s += ",\"tag\":";
        if (o.has_tag) put_string(s, o.tag); else s += "null";
        s += ",\"flags\":{\"bits\":";
        put_u64(s, o.flags);
        s += "},\"transform\":{\"transform_world\":";
        put_affine(s, o.transform_world);
        s += ",\"transform_local\":";
        put_affine(s, o.transform_local);
        s += ",\"transform_parent\":";
        if (o.has_parent) put_affine(s, o.transform_parent); else s += "null";
        s += "},\"inner\":";
        switch (o.kind) {
            case OBJ_EMPTY: s += "\"Empty\""; break;
            case OBJ_CAMERA:
                s += "{\"Camera\":{\"sensor_size\":";
                put_f32(s, o.camera.sensor_size);
                s += ",\"focal_length\":";
                put_f32(s, o.camera.focal_length);
                s += ",\"aspect_ratio\":";
                put_f32(s, o.camera.aspect_ratio);
                s += ",\"fstop\":";
                put_f32(s, o.camera.fstop);
                s += ",\"focus\":";
                if (o.camera.has_focus) put_f32(s, o.camera.focus); else s += "null";
                s += "}}";
                break;
            case OBJ_SPHERE:
                s += "{\"Sphere\":{\"material\":";
                put_u64(s, o.material);
                s += ",\"volume\":";
                if (o.has_volume) put_u64(s, o.volume); else s += "null";
                s += ",\"radius\":";
                put_f32(s, o.radius);
                s += "}}";
                break;
            case OBJ_RECT:
                s += "{\"Rect\":";
                put_rect(s, o.rect);
                s += '}';
                break;
            case OBJ_CUBOID:
                s += "{\"Cuboid\":{\"faces\":[";
                for (int i = 0; i < 6; ++i) {
                    if (i) s += ',';
                    s += '[';
                    put_vec3(s, o.face_offset[i]);
                    s += ',';
                    put_rect(s, o.faces[i]);
                    s += ']';
                }
                s += "]}}";
                break;
        }
        s += ",\"children\":";
        if (o.has_children) {
            s += '[';
            for (size_t i = 0; i < o.children.size(); ++i) {
                if (i) s += ',';
                put_u64(s, o.children[i]);
            }
            s += ']';
        } else {
            s += "null";
        }
        s += '}';
    }
    s += "},\"next_key\":";
    put_u64(s, objects_next_key);
    s += "},\"data\":{\"collection\":{";
    first = true;
    for (std::map<uint64_t, Data>::const_iterator it = data.begin(); it != data.end(); ++it) {
        const Data& d = it->second;
        if (!first) s += ',';
        first = false;
        s += '"';
        put_u64(s, it->first);
        s += "\":{\"inner\":";
        if (d.kind == DATA_MATERIAL) {
            static const char* names[5] = {"Flat", "Diffuse", "Metallic", "Glass", "Emissive"};
            s += "{\"Material\":{\"";
            s += names[d.mat_kind];
            s += "\":{\"albedo\":{\"r\":";
            put_f32(s, d.albedo[0]);
            s += ",\"g\":";
            put_f32(s, d.albedo[1]);
            s += ",\"b\":";
            put_f32(s, d.albedo[2]);
            s += '}';
            if (d.mat_kind == MAT_DIFFUSE || d.mat_kind == MAT_METALLIC || d.mat_kind == MAT_GLASS) {
                s += ",\"roughness\":";
                put_f32(s, d.roughness);
            }
            if (d.mat_kind == MAT_GLASS) {
                s += ",\"ior\":";
                put_f32(s, d.ior);
            }
            if (d.mat_kind == MAT_EMISSIVE) {
                s += ",\"intensity\":";
                put_f32(s, d.intensity);
            }
            s += "}}}";
        } else {
            s += "{\"Volume\":{\"DensityMap\":{\"width\":";
            put_u64(s, d.width);
            s += ",\"height\":";
            put_u64(s, d.height);
            s += ",\"depth\":";
            put_u64(s, d.depth);
            s += ",\"size\":";
            put_vec3(s, d.size);
            s += ",\"buffer\":[";
            for (size_t i = 0; i < d.buffer.size(); ++i) {
                if (i) s += ',';
                put_f32(s, d.buffer[i]);
            }
            s += "]}}}";
        }
        s += '}';
    }
    s += "},\"next_key\":";
    put_u64(s, data_next_key);
    s += '}';
    if (!lenses.empty()) {
        s += ",\"lenses\":[";
        for (size_t i = 0; i < lenses.size(); ++i) {
            if (i) s += ',';
            s += '[';
            for (int k = 0; k < 3; ++k) {
                put_f32(s, lenses[i].c[k]);
                s += ',';
            }
            put_f32(s, lenses[i].rs);
            s += ']';
        }
        s += ']';
    }
    s += '}';
    return s;
}

bool Scene::find_by_tag(const char* tag, uint64_t* out) const {
    for (std::map<uint64_t, Object>::const_iterator it = objects.begin(); it != objects.end(); ++it)
        if (it->second.has_tag && it->second.tag == tag) {
            *out = it->first;
            return true;
        }
    return false;
}
Object& Scene::get_object(uint64_t r) {
    std::map<uint64_t, Object>::iterator it = objects.find(r);
    if (it == objects.end()) throw SceneError("invalid object ref");
    return it->second;
}
const Object& Scene::get_object(uint64_t r) const {
    std::map<uint64_t, Object>::const_iterator it = objects.find(r);
    if (it == objects.end()) throw SceneError("invalid object ref");
    return it->second;
}
const Data& Scene::get_data(uint64_t r) const {
    std::map<uint64_t, Data>::const_iterator it = data.find(r);
    if (it == data.end()) throw SceneError("invalid data ref");
    return it->second;
}

namespace {
// Object::apply_parent_transform, object/mod.rs:200-210 (the queue is replaced by recursion: the
// reference's breadth-first UpdateQueue::commit reaches the same fixed point)
void apply_parent(Scene& s, uint64_t ref, const Affine& parent, int depth) {
    if (depth > 256) throw SceneError("scene graph cycle");
    Object& o = s.get_object(ref);
    o.has_parent = true;
    o.transform_parent = parent;
    o.transform_world = affine_mul(parent, o.transform_local);  // transform.rs:45-48
    Affine world = o.transform_world;
    std::vector<uint64_t> children = o.children;
    for (size_t i = 0; i < children.size(); ++i) apply_parent(s, children[i], world, depth + 1);
}
}  // namespace

void Scene::apply_transform(uint64_t object_ref, const Affine& affine) {  // object/mod.rs:212-223
    Object& o = get_object(object_ref);
    o.transform_local = affine_mul(o.transform_local, affine);  // transform.rs:34-42
    o.transform_world = o.has_parent ? affine_mul(o.transform_parent, o.transform_local) : o.transform_local;
    Affine world = o.transform_world;
    std::vector<uint64_t> children = o.children;
    for (size_t i = 0; i < children.size(); ++i) apply_parent(*this, children[i], world, 0);
}

// ------------------------------------------------------------------------------------------
// flattening
// ------------------------------------------------------------------------------------------
namespace {

typedef AABB Bounds;
// LIGHT_RECT fields l1..l6 of a light record (layout.h): Rect::random_point, rect.rs:82-86
void fill_rect_light(float4* l, const Rect& r, const Affine& tf) {
    l[1] = f4(r.x[0], r.x[1], r.x[2], -r.half_width);
    l[2] = f4(r.y[0], r.y[1], r.y[2], -r.half_height);
    l[3] = f4(tf.f[0], tf.f[1], tf.f[2], uniform_scale_inclusive(-r.half_width, r.half_width));
    l[4] = f4(tf.f[3], tf.f[4], tf.f[5], uniform_scale_inclusive(-r.half_height, r.half_height));
    l[5] = f4(tf.f[6], tf.f[7], tf.f[8], 0.0f);
    l[6] = f4(tf.f[9], tf.f[10], tf.f[11], 0.0f);
}
// 0 / 1 / 2 when v is exactly +-1 on that axis and (+-)0 on the others, else -1
int unit_axis(const float v[3]) {
    int k = -1;
    for (int i = 0; i < 3; ++i) {
        if (v[i] == 0.0f) continue;
        if (std::fabs(v[i]) != 1.0f || k >= 0) return -1;
        k = i;
    }
    return k;
}
void push_rect(std::vector<float4>& blob, std::vector<Bounds>& bounds, const Rect& r, const Affine& tf, int type, uint32_t mat, uint32_t obj,
               bool allow_aa = false) {
    {   // world-space AABB of the four corners (rect.rs:38-56)
        Bounds b;
        for (int k = 0; k < 3; ++k) { b.lo[k] = 3.0e38f; b.hi[k] = -3.0e38f; }
        for (int c = 0; c < 4; ++c) {
            float sx = (c & 1) ? -r.half_width : r.half_width, sy = (c & 2) ? -r.half_height : r.half_height;
            float local[3] = {r.x[0] * sx + r.y[0] * sy, r.x[1] * sx + r.y[1] * sy, r.x[2] * sx + r.y[2] * sy}, w[3];
            mat_vec(tf, local, w);
            for (int k = 0; k < 3; ++k) {
                float v = w[k] + tf.f[9 + k];
                b.lo[k] = std::min(b.lo[k], v);
                b.hi[k] = std::max(b.hi[k], v);
            }
        }
        bounds.push_back(b);
    }
    float n[3];
    mat_vec(tf, r.z, n);  // rect.rs:119: transform.transform_vector3a(self.z)
    // local = M^-1 (pos - T);  local.x = dot(pos, ax) + cx with ax = M^-T x, cx = -dot(ax, T)
    double m[9], inv[9];
    for (int i = 0; i < 9; ++i) m[i] = tf.f[i];
    // column-major: element (row r, col c) = m[3*c + r]
    double det = m[0] * (m[4] * m[8] - m[7] * m[5]) - m[3] * (m[1] * m[8] - m[7] * m[2]) + m[6] * (m[1] * m[5] - m[4] * m[2]);
    double id = 1.0 / det;
    // inverse, row-major rows R0,R1,R2 (so that local = R * (pos - T))
    inv[0] = (m[4] * m[8] - m[7] * m[5]) * id;
    inv[1] = (m[6] * m[5] - m[3] * m[8]) * id;
    inv[2] = (m[3] * m[7] - m[6] * m[4]) * id;
    inv[3] = (m[7] * m[2] - m[1] * m[8]) * id;
    inv[4] = (m[0] * m[8] - m[6] * m[2]) * id;
    inv[5] = (m[6] * m[1] - m[0] * m[7]) * id;
    inv[6] = (m[1] * m[5] - m[4] * m[2]) * id;
    inv[7] = (m[3] * m[2] - m[0] * m[5]) * id;
    inv[8] = (m[0] * m[4] - m[3] * m[1]) * id;
    double ax[3], ay[3];
    for (int k = 0; k < 3; ++k) {
        ax[k] = r.x[0] * inv[0 + k] + r.x[1] * inv[3 + k] + r.x[2] * inv[6 + k];
        ay[k] = r.y[0] * inv[0 + k] + r.y[1] * inv[3 + k] + r.y[2] * inv[6 + k];
    }
    double cx = -(ax[0] * tf.f[9] + ax[1] * tf.f[10] + ax[2] * tf.f[11]);
    double cy = -(ay[0] * tf.f[9] + ay[1] * tf.f[10] + ay[2] * tf.f[11]);
    double x2 = (double)r.x[0] * r.x[0] + (double)r.x[1] * r.x[1] + (double)r.x[2] * r.x[2];
    double y2 = (double)r.y[0] * r.y[0] + (double)r.y[1] * r.y[1] + (double)r.y[2] * r.y[2];
    float hw2 = (float)((double)(r.half_width * r.half_width) / x2);
    float hh2 = (float)((double)(r.half_height * r.half_height) / y2);
    float area = 4.0f * r.half_width * r.half_height;  // rect.rs:88-90
    float4 q2 = f4((float)ax[0], (float)ax[1], (float)ax[2], (float)cx), q3 = f4((float)ay[0], (float)ay[1], (float)ay[2], (float)cy);
    // axis-aligned? (normal and both plane axes exact +-unit coordinate axes, on three different axes)
    uint32_t aa_axis = 0;
    if (type == PRIM_RECT && allow_aa) {
        const float fn[3] = {n[0], n[1], n[2]}, fx[3] = {q2.x, q2.y, q2.z}, fy[3] = {q3.x, q3.y, q3.z};
        int kn = unit_axis(fn), kx = unit_axis(fx), ky = unit_axis(fy);
        if (kn >= 0 && kx >= 0 && ky >= 0 && kn != kx && kn != ky && kx != ky) {
            if (kx != (kn + 1) % 3) {  // the inside test is symmetric in (q2, hw2) and (q3, hh2)
                std::swap(q2, q3);
                std::swap(hw2, hh2);
            }
            type = PRIM_RECT_AA;
            aa_axis = (uint32_t)kn;
        }
    }
    blob.push_back(f4(n[0], n[1], n[2], hw2));
    blob.push_back(f4(tf.f[9], tf.f[10], tf.f[11], hh2));
    blob.push_back(q2);
    blob.push_back(q3);
    blob.push_back(f4(as_f((uint32_t)type | (aa_axis << 2) | ((uint32_t)(blob.size() / PRIM_STRIDE) << PRIM_CANON_SHIFT)), as_f(mat),
                      type != PRIM_CUBOID_FACE ? area : as_f(0u), as_f(obj)));
}

// A Cuboid whose six faces really are the faces of one rectangular box (Cuboid::new, cuboid.rs:19-30,
// under a rigid transform) gets a BOX record: the scan then finds the closest face with one slab
// test instead of six rect tests.  Anything else (hand-edited faces, sheared transforms) keeps the
// six rect tests.  Faces come in opposite pairs (0,1) (2,3) (4,5).
bool make_box(const Object& o, const Affine& tf, float4 out[BOX_STRIDE]) {
    double c[6][3], n[6][3], ex[6][3], ey[6][3], C[3] = {0, 0, 0};
    for (int i = 0; i < 6; ++i) {
        float t[3], v[3];
        mat_vec(tf, o.face_offset[i], t);
        for (int k = 0; k < 3; ++k) { c[i][k] = (double)t[k] + tf.f[9 + k]; C[k] += c[i][k] / 6.0; }
        mat_vec(tf, o.faces[i].z, v);
        for (int k = 0; k < 3; ++k) n[i][k] = v[k];
        mat_vec(tf, o.faces[i].x, v);
        for (int k = 0; k < 3; ++k) ex[i][k] = (double)v[k] * o.faces[i].half_width;
        mat_vec(tf, o.faces[i].y, v);
        for (int k = 0; k < 3; ++k) ey[i][k] = (double)v[k] * o.faces[i].half_height;
    }
    auto dot = [](const double* a, const double* b) { return a[0] * b[0] + a[1] * b[1] + a[2] * b[2]; };
    auto len = [&](const double* a) { return std::sqrt(dot(a, a)); };
    double a[3][3], h[3];
    for (int k = 0; k < 3; ++k) {
        double d[3], m[3];
        for (int j = 0; j < 3; ++j) { d[j] = c[2 * k + 1][j] - c[2 * k][j]; m[j] = c[2 * k + 1][j] + c[2 * k][j] - 2.0 * C[j]; }
        h[k] = 0.5 * len(d);
        if (!(h[k] > 1e-12)) return false;
        for (int j = 0; j < 3; ++j) a[k][j] = d[j] / (2.0 * h[k]);
        if (len(m) > 1e-4 * (h[0] + h[k] + 1e-12)) return false;
    }
    const double scale = h[0] + h[1] + h[2];
    const double tol = 1e-4;
    for (int k = 0; k < 3; ++k)
        if (std::fabs(dot(a[k], a[(k + 1) % 3])) > tol) return false;
    uint32_t bits = 0;
    for (int i = 0; i < 6; ++i) {
        const int k = i / 2, k1 = (k + 1) % 3, k2 = (k + 2) % 3;
        const double nl = len(n[i]);
        if (!(nl > 1e-12)) return false;
        const double na = dot(n[i], a[k]) / nl;
        if (std::fabs(std::fabs(na) - 1.0) > tol) return false;          // the face normal is the pair's axis
        if (na < 0) bits |= 1u << i;
        // the rect's extents are the other two axes' half-extents (either assignment)
        const double x1 = std::fabs(dot(ex[i], a[k1])), x2 = std::fabs(dot(ex[i], a[k2]));
        const double y1 = std::fabs(dot(ey[i], a[k1])), y2 = std::fabs(dot(ey[i], a[k2]));
        const bool direct = std::fabs(x1 - h[k1]) <= tol * scale && x2 <= tol * scale && std::fabs(y2 - h[k2]) <= tol * scale && y1 <= tol * scale;
        const bool swapped = std::fabs(x2 - h[k2]) <= tol * scale && x1 <= tol * scale && std::fabs(y1 - h[k1]) <= tol * scale && y2 <= tol * scale;
        if (!direct && !swapped) return false;
        if (std::fabs(dot(ex[i], a[k])) > tol * scale || std::fabs(dot(ey[i], a[k])) > tol * scale) return false;
    }
    out[0] = f4((float)C[0], (float)C[1], (float)C[2], (float)h[0]);
    out[1] = f4((float)a[0][0], (float)a[0][1], (float)a[0][2], (float)h[1]);
    out[2] = f4((float)a[1][0], (float)a[1][1], (float)a[1][2], (float)h[2]);
    out[3] = f4((float)a[2][0], (float)a[2][1], (float)a[2][2], as_f(bits));
    return true;
}

// ---- binned-SAH build of a binary tree (one primitive per leaf), collapsed to the 4-wide nodes the device reads -----
struct BvhBuild {
    const std::vector<Bounds>& b;
    std::vector<uint32_t> order;   // record position -> canonical primitive index
    enum { STRIDE2 = 4 };          // binary node: (L box, R box, left, right), the builder's own format
    std::vector<float4> nodes;     // STRIDE2 float4 per binary inner node
    std::vector<float4> wide;      // BVH_STRIDE float4 per 4-wide node (collapse())
    explicit BvhBuild(const std::vector<Bounds>& bounds) : b(bounds) {
        for (uint32_t i = 0; i < b.size(); ++i) order.push_back(i);
    }
    static void grow(Bounds& box, const Bounds& p) {
        for (int k = 0; k < 3; ++k) {
            box.lo[k] = std::min(box.lo[k], p.lo[k]);
            box.hi[k] = std::max(box.hi[k], p.hi[k]);
        }
    }
    static Bounds empty() {
        Bounds e;
        for (int k = 0; k < 3; ++k) { e.lo[k] = 3.0e38f; e.hi[k] = -3.0e38f; }
        return e;
    }
    static float area(const Bounds& x) {
        float d[3] = {x.hi[0] - x.lo[0], x.hi[1] - x.lo[1], x.hi[2] - x.lo[2]};
        if (d[0] < 0) return 0.0f;
        return d[0] * d[1] + d[1] * d[2] + d[2] * d[0];
    }
    static Bounds padded(Bounds box) {  // conservative: the tree must never cull what the scan would hit
        for (int k = 0; k < 3; ++k) {
            float pad = 1e-4f * std::max(1.0f, std::max(std::fabs(box.lo[k]), std::fabs(box.hi[k])));
            box.lo[k] -= pad;
            box.hi[k] += pad;
        }
        return box;
    }
    std::vector<uint8_t> sphere;   // per canonical primitive: is it a sphere record (leaf kinds)
    uint32_t leaf_ref(uint32_t first, uint32_t count) const {
        uint32_t n_sph = 0;
        for (uint32_t i = first; i < first + count; ++i) n_sph += order[i] < sphere.size() && sphere[order[i]];
        const uint32_t kind = count == 0 ? 0u : (n_sph == count ? (uint32_t)BVH_KIND_SPHERES : (n_sph == 0 ? (uint32_t)BVH_KIND_RECTS : 0u));
        return BVH_LEAF | (kind << 29) | (count << 24) | first;
    }
    void set_inner(uint32_t self, uint32_t left, const Bounds& l, uint32_t right, const Bounds& r) {  // (unpadded boxes)
        nodes[self * STRIDE2] = f4(l.lo[0], l.lo[1], l.lo[2], l.hi[0]);
        nodes[self * STRIDE2 + 1] = f4(l.hi[1], l.hi[2], r.lo[0], r.lo[1]);
        nodes[self * STRIDE2 + 2] = f4(r.lo[2], r.hi[0], r.hi[1], r.hi[2]);
        nodes[self * STRIDE2 + 3] = f4(as_f(left), as_f(right), 0.0f, 0.0f);
    }
    uint32_t make_inner(uint32_t left, const Bounds& lb, uint32_t right, const Bounds& rb) {
        uint32_t self = (uint32_t)(nodes.size() / STRIDE2);
        nodes.resize(nodes.size() + STRIDE2);
        set_inner(self, left, lb, right, rb);
        return self;
    }
    struct Child { uint32_t ref; Bounds box; };
    void children_of(uint32_t node, Child* l, Child* r) const {
        const float4* q = &nodes[(size_t)node * STRIDE2];
        l->ref = as_u(q[3].x);
        r->ref = as_u(q[3].y);
        l->box.lo[0] = q[0].x; l->box.lo[1] = q[0].y; l->box.lo[2] = q[0].z; l->box.hi[0] = q[0].w; l->box.hi[1] = q[1].x; l->box.hi[2] = q[1].y;
        r->box.lo[0] = q[1].z; r->box.lo[1] = q[1].w; r->box.lo[2] = q[2].x; r->box.hi[0] = q[2].y; r->box.hi[1] = q[2].z; r->box.hi[2] = q[2].w;
    }
    static bool is_inner(uint32_t ref) { return !(ref & BVH_LEAF); }
    static bool is_empty_leaf(uint32_t ref) { return (ref & BVH_LEAF) && ((ref >> 24) & 0x1fu) == 0; }
    static void write_wide(float4* q, const Child* c, int n) {  // (pads the boxes)
        float v[6][4];
        uint32_t ref[4];
        for (int i = 0; i < (int)BVH_WIDTH; ++i) {
            Bounds b = i < n ? padded(c[i].box) : empty();
            for (int k = 0; k < 3; ++k) { v[2 * k][i] = b.lo[k]; v[2 * k + 1][i] = b.hi[k]; }
            ref[i] = i < n ? c[i].ref : (uint32_t)BVH_EMPTY;
        }
        for (int k = 0; k < 6; ++k) q[k] = f4(v[k][0], v[k][1], v[k][2], v[k][3]);
        q[6] = f4(as_f(ref[0]), as_f(ref[1]), as_f(ref[2]), as_f(ref[3]));
        q[7] = f4(0.0f, 0.0f, 0.0f, 0.0f);
    }
    // Binary node -> 4-wide node: both children are opened when they are inner nodes (so a wide level spans two
    // binary levels and the wide tree is at most half as deep), then the largest remaining inner child while a slot
    // is free.  A wide node is stored before its children (refit_bvh sweeps backwards).
    uint32_t collapse(uint32_t node) {
        Child c[BVH_WIDTH + 1];
        int n = 2;
        children_of(node, &c[0], &c[1]);
        auto open = [&](int i) {
            Child l, r;
            children_of(c[i].ref, &l, &r);
            c[i] = l;
            c[n++] = r;
        };
        const bool open0 = is_inner(c[0].ref), open1 = is_inner(c[1].ref);
        if (open0) open(0);
        if (open1) open(1);
        while (n < (int)BVH_WIDTH) {
            int best = -1;
            for (int i = 0; i < n; ++i)
                if (is_inner(c[i].ref) && (best < 0 || area(c[i].box) > area(c[best].box))) best = i;
            if (best < 0) break;
            open(best);
        }
        int m = 0;
        for (int i = 0; i < n; ++i)
            if (!is_empty_leaf(c[i].ref)) c[m++] = c[i];
        n = m;
        const uint32_t self = (uint32_t)(wide.size() / BVH_STRIDE);
        wide.resize(wide.size() + BVH_STRIDE);
        for (int i = 0; i < n; ++i)
            if (is_inner(c[i].ref)) c[i].ref = collapse(c[i].ref);
        write_wide(&wide[(size_t)self * BVH_STRIDE], c, n);
        return self;
    }
    // returns a child reference (inner node index, or BVH_LEAF | count << 24 | first) and its box
    uint32_t build(uint32_t first, uint32_t count, int depth, Bounds* box_out) {
        Bounds box = empty(), cb = empty();
        for (uint32_t i = first; i < first + count; ++i) {
            const Bounds& p = b[order[i]];
            grow(box, p);
            Bounds c;
            for (int k = 0; k < 3; ++k) c.lo[k] = c.hi[k] = 0.5f * (p.lo[k] + p.hi[k]);
            grow(cb, c);
        }
        *box_out = box;
        int axis = 0;
        for (int k = 1; k < 3; ++k)
            if (cb.hi[k] - cb.lo[k] > cb.hi[axis] - cb.lo[axis]) axis = k;
        // The traversal stack bounds the depth (layout.h: 3 pushes per wide level = per two levels here).  A skewed SAH split is only taken while median splits could
        // still bring what remains down to leaf size; coincident centroids (no axis to split on) are halved by
        // index -- a leaf holds at most BVH_LEAF_MAX records.
        const int remaining = (int)BVH_MAX_DEPTH2 - 2 - depth;
        const bool degenerate = !(cb.hi[axis] > cb.lo[axis]);
        // one primitive per leaf: measured 1 / 2 / 3 / 4 / 6 / 8 -> 270 / 252 / 255 / 244 / 232 / 222 Msamples/s on the 32 k-primitive scene (a
        // leaf test is a divergent loop over records of mixed type; a node visit is four uniform slab tests).  BT_BVH_LEAF: experiments.
        static const uint32_t leaf_max = std::getenv("BT_BVH_LEAF") ? (uint32_t)std::max(1, std::atoi(std::getenv("BT_BVH_LEAF"))) : 1u;
        if (count <= leaf_max || remaining <= 0 || (degenerate && count <= (uint32_t)BVH_LEAF_MAX)) {
            if (count > (uint32_t)BVH_LEAF_MAX) throw SceneError("BVH: the scene is too large for the traversal stack");
            return leaf_ref(first, count);
        }
        const bool force_median = degenerate || (uint64_t)count > ((uint64_t)64 << std::max(0, remaining - 2));
        // binned SAH: the cheapest of the candidate planes of all three axes (env BT_BVH_SAH_AXES=1: the widest centroid axis only)
        const int NB = 16;
        static const bool all_axes = !(std::getenv("BT_BVH_SAH_AXES") && std::atoi(std::getenv("BT_BVH_SAH_AXES")) == 1);
        const int widest = axis;
        int best = -1, best_axis = widest;
        float best_cost = 3.0e38f;
        auto bin_on = [&](uint32_t prim, int ax) {
            const float ext = cb.hi[ax] - cb.lo[ax];
            int k = (int)((0.5f * (b[prim].lo[ax] + b[prim].hi[ax]) - cb.lo[ax]) * (ext > 0.0f ? (float)NB / ext : 0.0f));
            return std::min(std::max(k, 0), NB - 1);
        };
        for (int ax = 0; ax < 3 && !degenerate; ++ax) {
            if (!(all_axes || ax == widest) || !(cb.hi[ax] > cb.lo[ax])) continue;
            Bounds bin_box[NB];
            uint32_t bin_n[NB];
            for (int i = 0; i < NB; ++i) { bin_box[i] = empty(); bin_n[i] = 0; }
            for (uint32_t i = first; i < first + count; ++i) {
                int k = bin_on(order[i], ax);
                grow(bin_box[k], b[order[i]]);
                bin_n[k]++;
            }
            float right_area[NB];
            Bounds acc = empty();
            for (int i = NB - 1; i > 0; --i) {
                grow(acc, bin_box[i]);
                right_area[i] = area(acc);
            }
            acc = empty();
            uint32_t nl = 0;
            for (int i = 0; i < NB - 1; ++i) {
                grow(acc, bin_box[i]);
                nl += bin_n[i];
                if (nl == 0 || nl == count) continue;
                float cost = area(acc) * (float)nl + right_area[i + 1] * (float)(count - nl);
                if (cost < best_cost) { best_cost = cost; best = i; best_axis = ax; }
            }
        }
        if (best >= 0 && !force_median) axis = best_axis;
        auto bin_of = [&](uint32_t prim) { return bin_on(prim, axis); };
        uint32_t mid;
        if (best >= 0 && !force_median) {
            mid = (uint32_t)(std::partition(order.begin() + first, order.begin() + first + count,
                                            [&](uint32_t prim) { return bin_of(prim) <= best; }) - order.begin());
        } else {
            mid = first + count / 2;
            std::nth_element(order.begin() + first, order.begin() + mid, order.begin() + first + count,
                             [&](uint32_t x, uint32_t y) { return b[x].lo[axis] + b[x].hi[axis] < b[y].lo[axis] + b[y].hi[axis]; });
        }
        Bounds lb, rb;
        uint32_t self = make_inner(0, box, 0, box);  // reserve the slot before the children (root = node 0)
        uint32_t left = build(first, mid - first, depth + 1, &lb);
        uint32_t right = build(mid, first + count - mid, depth + 1, &rb);
        set_inner(self, left, lb, right, rb);
        return self;
    }
};

// ---- the records of ONE object (flatten() appends them; update_flat() overwrites them in place after a transform edit) ----
struct EmitCtx {
    const Scene& scene;
    const std::map<uint64_t, uint32_t>& mat_index;
    const std::map<uint64_t, uint32_t>& vol_index;
    bool aa_rects;
    uint32_t material(uint64_t r) const {
        const Data& d = scene.get_data(r);
        if (d.kind != DATA_MATERIAL) throw SceneError("expected material data");
        return mat_index.find(r)->second;
    }
};
struct ObjRecords {
    std::vector<float4> prims;        // PRIM_STRIDE per primitive, canonical indices first_prim ..
    std::vector<Bounds> bounds;
    bool any_diffuse = false, has_volume = false;
    bool has_box = false;             // a Cuboid whose faces form one rectangular box
    float4 box[BOX_STRIDE];
    bool is_light = false, zero_area = false;
    std::vector<float4> light;        // LIGHT_STRIDE (l0.y = first_prim, canonical)
    std::vector<float4> face_lights;  // 6 x LIGHT_STRIDE for a LIGHT Cuboid
};
ObjRecords emit_object(const EmitCtx& ctx, const Object& o, uint32_t obj, uint32_t first_prim) {
    ObjRecords rec;
    const Scene& scene = ctx.scene;
    std::vector<float4>& prims = rec.prims;
    uint32_t n_prims = 0;
    const Affine& tf = o.transform_world;
    if (o.kind == OBJ_SPHERE) {
        uint32_t mat = ctx.material(o.material);
        uint32_t vol = 0xffffffffu;
        if (o.has_volume) {
            const Data& d = scene.get_data(o.volume);
            if (d.kind != DATA_VOLUME) throw SceneError("expected volume data");
            vol = ctx.vol_index.find(o.volume)->second;
            rec.has_volume = true;
        }
        float r = o.radius;
        prims.push_back(f4(tf.f[9], tf.f[10], tf.f[11], r));
        prims.push_back(f4(r * r, 3.14159265358979323846f * r * r, r > 0.0f ? 2e-5f / r : 3.0e38f, 0.0f));
        prims.push_back(f4(0, 0, 0, 0));
        prims.push_back(f4(0, 0, 0, 0));
        prims.push_back(f4(as_f((uint32_t)PRIM_SPHERE), as_f(mat), as_f(vol), as_f(obj)));
        {
            Bounds b;
            for (int k = 0; k < 3; ++k) { b.lo[k] = tf.f[9 + k] - r; b.hi[k] = tf.f[9 + k] + r; }
            rec.bounds.push_back(b);
        }
        n_prims = 1;
        rec.any_diffuse |= scene.get_data(o.material).mat_kind == MAT_DIFFUSE;
    } else if (o.kind == OBJ_RECT) {
        push_rect(prims, rec.bounds, o.rect, tf, PRIM_RECT, ctx.material(o.rect.material), obj, ctx.aa_rects);
        n_prims = 1;
        rec.any_diffuse |= scene.get_data(o.rect.material).mat_kind == MAT_DIFFUSE;
    } else if (o.kind == OBJ_CUBOID) {
        for (int i = 0; i < 6; ++i) {
            // transform * Affine3A::from_translation(offset), cuboid.rs:95
            Affine ftf = tf;
            float t[3];
            mat_vec(tf, o.face_offset[i], t);
            for (int k = 0; k < 3; ++k) ftf.f[9 + k] = t[k] + tf.f[9 + k];
            push_rect(prims, rec.bounds, o.faces[i], ftf, PRIM_CUBOID_FACE, ctx.material(o.faces[i].material), obj);
            rec.any_diffuse |= scene.get_data(o.faces[i].material).mat_kind == MAT_DIFFUSE;
        }
        rec.has_box = make_box(o, tf, rec.box);
        n_prims = 6;
    }
    // the canonical primitive index lives in the high bits of q4.x (layout.h: PRIM_CANON_SHIFT)
    for (uint32_t i = 0; i < n_prims; ++i) {
        float4& meta = prims[(size_t)i * PRIM_STRIDE + 4];
        meta.x = as_f((as_u(meta.x) & ((1u << PRIM_CANON_SHIFT) - 1u)) | ((first_prim + i) << PRIM_CANON_SHIFT));
    }
    if (o.flags & 1u) {  // ObjectFlags::LIGHT
        rec.is_light = true;
        std::vector<float4>& lights = rec.light;
        lights.assign(LIGHT_STRIDE, f4(0, 0, 0, 0));
        if (o.kind == OBJ_SPHERE) {
            lights[0] = f4(as_f(LIGHT_SPHERE), as_f(first_prim), as_f(n_prims), as_f(obj));
            lights[1] = f4(tf.f[9], tf.f[10], tf.f[11], o.radius);
        } else if (o.kind == OBJ_RECT) {
            lights[0] = f4(as_f(LIGHT_RECT), as_f(first_prim), as_f(n_prims), as_f(obj));
            fill_rect_light(&lights[0], o.rect, tf);
        } else if (o.kind == OBJ_CUBOID) {
            // Cuboid::random_point, cuboid.rs:48-54: WeightedIndex over the face areas (rand 0.8.5:
            // cumulative sums without the last weight, Uniform::new(0, total)), then the face's
            // Rect::random_point.  The six faces become LIGHT_RECT sub-records behind the object
            // lights (appended by flatten); l2.z holds the first one's index.
            float cumulative[5];
            float total = 4.0f * o.faces[0].half_width * o.faces[0].half_height;
            for (int i = 1; i < 6; ++i) {
                cumulative[i - 1] = total;
                total += 4.0f * o.faces[i].half_width * o.faces[i].half_height;
            }
            if (!(total > 0.0f)) rec.zero_area = true;
            lights[0] = f4(as_f(LIGHT_CUBOID), as_f(first_prim), as_f(n_prims), as_f(obj));
            lights[1] = f4(cumulative[0], cumulative[1], cumulative[2], cumulative[3]);
            lights[2] = f4(cumulative[4], total > 0.0f ? uniform_scale(0.0f, total) : 0.0f, as_f(0u), 0.0f);
            for (int i = 0; i < 6; ++i) {
                Affine ftf = tf;
                float t[3];
                mat_vec(tf, o.face_offset[i], t);
                for (int k = 0; k < 3; ++k) ftf.f[9 + k] = t[k] + tf.f[9 + k];
                size_t fb = rec.face_lights.size();
                rec.face_lights.resize(fb + LIGHT_STRIDE, f4(0, 0, 0, 0));
                rec.face_lights[fb] = f4(as_f(LIGHT_RECT), as_f(first_prim + (uint32_t)i), as_f(1u), as_f(obj));
                fill_rect_light(&rec.face_lights[fb], o.faces[i], ftf);
                rec.face_lights[fb + 5].w = 4.0f * o.faces[i].half_width * o.faces[i].half_height;  // Rect::area (rect.rs:98)
            }
        } else {
            lights[0] = f4(as_f(LIGHT_POINT), as_f(0), as_f(0), as_f(obj));
            lights[1] = f4(tf.f[9], tf.f[10], tf.f[11], 0.0f);
        }
    }
    return rec;
}

// The free-distance grid of a lensed linear-scan scene (SceneHeader::dist_*).  A geodesic chord shorter than the distance
// from its start to the nearest primitive surface cannot hit anything and is not intersected (DESIGN.md, "Geodesic
// flights"); the grid makes that distance one byte load per RK4 step instead of per-flight bookkeeping that decays and is
// refreshed by intersection passes.  Every cell stores a LOWER bound valid for all of its points: the distance from the
// cell centre to the nearest primitive (spheres exactly, everything else through its world AABB), minus the cell's half
// diagonal, minus the rounding margins of the hit tests (those of scan_prims_t<DIST>), rounded down to the quantum.
// Spheres that span the scene (the r = 100 ground of the shipped scenes) would blow the box up: up to two of them are
// left out of the BOX (the cells inside it account for them like for every other primitive) and evaluated exactly for
// points outside it.  Returns false (the per-flight scheme stays) when there are
// more, or nothing to put in a grid.
bool build_dist_grid(const std::vector<float4>& prims, const std::vector<Bounds>& bounds, SceneHeader& h, std::vector<uint8_t>* out, bool fill) {
    const uint32_t n = h.n_prims;
    if (n == 0 || bounds.size() < n) return false;
    std::vector<float> size(n);
    for (uint32_t i = 0; i < n; ++i) {
        float e = 0.0f;
        for (int k = 0; k < 3; ++k) e = std::max(e, bounds[i].hi[k] - bounds[i].lo[k]);
        size[i] = e;
    }
    std::vector<float> sorted(size);
    std::sort(sorted.begin(), sorted.end());
    const float median = sorted[n / 2];
    std::vector<char> far(n, 0);
    h.n_far = 0;
    h.far_prim[0] = h.far_prim[1] = -1;
    for (uint32_t i = 0; i < n; ++i) {
        const uint32_t type = as_u(prims[i * PRIM_STRIDE + 4].x) & 3u;
        if (type == PRIM_SPHERE && n > 1 && size[i] > 16.0f * median) {
            if (h.n_far == 2) return false;
            far[i] = 1;
            h.far_prim[h.n_far++] = (int32_t)i;
        }
    }
    Bounds box = BvhBuild::empty();
    uint32_t n_in = 0;
    for (uint32_t i = 0; i < n; ++i)
        if (!far[i]) {
            BvhBuild::grow(box, bounds[i]);
            ++n_in;
        }
    if (n_in == 0) return false;
    float extent = 0.0f;
    for (int k = 0; k < 3; ++k) extent = std::max(extent, box.hi[k] - box.lo[k]);
    if (!(extent > 0.0f) || !std::isfinite(extent)) return false;
    const float pad = std::max(0.1f * extent, 0.25f);
    double volume = 1.0;
    for (int k = 0; k < 3; ++k) {
        box.lo[k] -= pad;
        box.hi[k] += pad;
        volume *= (double)(box.hi[k] - box.lo[k]);
    }
    // 2^21 cells at most, and at most 2^24 cell x primitive distance evaluations on the host
    const double max_cells = std::min(2097152.0, 16777216.0 / (double)n);
    const float cell = (float)std::cbrt(volume / max_cells) * 1.0001f;
    uint32_t dims[3];
    for (int k = 0; k < 3; ++k) dims[k] = std::max(1u, (uint32_t)std::ceil((box.hi[k] - box.lo[k]) / cell));
    const float q = 0.5f * cell;
    // a point is binned with float arithmetic and may land one ulp into the neighbouring cell: the half diagonal is padded
    const double half_diag = 0.5 * std::sqrt(3.0) * (double)cell * 1.01 + 1e-5;
    // The stepper bins with fma(x, 1 / cell, -lo / cell): rounded 1 / cell, rounded offset and the rounded sum put a point of
    // the box at most (|x| / cell + |lo| / cell + index) * 2^-23 cells off its true cell coordinate along each axis.  The
    // padding above covers a point 0.005 cells outside its cell (sqrt(3) * 0.005 < 0.01 * 0.5 * sqrt(3)); a box that far
    // from the origin, measured in cells, keeps the per-flight scheme.
    const float inv_cell = 1.0f / cell;
    float off[3];
    for (int k = 0; k < 3; ++k) {
        off[k] = -box.lo[k] * inv_cell;
        const double reach = std::max(std::fabs((double)box.lo[k]), std::fabs((double)box.lo[k] + (double)dims[k] * cell)) / cell;
        if ((2.0 * reach + dims[k] + 2.0) * std::ldexp(1.0, -23) > 0.005) return false;
    }
    for (uint32_t i = 0; i < h.n_far; ++i) {  // the far spheres' records, as the stepper reads them (sphere_free_bound)
        const float4* rec = &prims[(size_t)h.far_prim[i] * PRIM_STRIDE];
        h.far_c[i][0] = rec[0].x;
        h.far_c[i][1] = rec[0].y;
        h.far_c[i][2] = rec[0].z;
        h.far_c[i][3] = rec[0].w;
        h.far_k[i] = rec[1].z;
    }
    // The cells are normally filled ON THE DEVICE (engine.cu: dist_grid_kernel, the same arithmetic in the same order, one thread
    // per cell: a 2M-cell grid takes 65 - 140 ms here and well under a millisecond there); BT_DIST_GRID_HOST=1 fills them here.
    out->clear();
    if (fill) out->assign((size_t)dims[0] * dims[1] * dims[2], 0);
    for (uint32_t z = 0; fill && z < dims[2]; ++z)
        for (uint32_t y = 0; y < dims[1]; ++y)
            for (uint32_t x = 0; x < dims[0]; ++x) {
                const double c[3] = {box.lo[0] + (x + 0.5) * (double)cell, box.lo[1] + (y + 0.5) * (double)cell, box.lo[2] + (z + 0.5) * (double)cell};
                const double l1 = std::fabs(c[0]) + std::fabs(c[1]) + std::fabs(c[2]) + 3.0 * half_diag;
                double best = 1e30;
                for (uint32_t i = 0; i < n; ++i) {  // (the scene-spanning spheres too: they are only left out of the BOX)
                    const float4* rec = &prims[i * PRIM_STRIDE];
                    double b;
                    if ((as_u(rec[4].x) & 3u) == PRIM_SPHERE) {
                        const double dx = c[0] - rec[0].x, dy = c[1] - rec[0].y, dz = c[2] - rec[0].z, r = rec[0].w;
                        const double dc = std::sqrt(dx * dx + dy * dy + dz * dz), dmax = dc + half_diag;
                        // sphere_free_bound's margin at the farthest point of the cell (rec[1].z = 2e-5 / r)
                        b = std::fabs(dc - r) - (dmax * dmax * (double)rec[1].z + 2e-5 * (dmax + r) + 1e-6);
                    } else {
                        double d2 = 0.0, ext = 0.0;
                        for (int k = 0; k < 3; ++k) {
                            const double d = std::max(std::max((double)bounds[i].lo[k] - c[k], c[k] - (double)bounds[i].hi[k]), 0.0);
                            d2 += d * d;
                            ext += std::fabs((double)bounds[i].hi[k] - (double)bounds[i].lo[k]);
                        }
                        // the margin of the rect / box bounds of scan_prims_t<DIST>
                        b = std::sqrt(d2) - (1e-4 * (l1 + ext + std::sqrt(d2)) + 1e-4);
                    }
                    best = std::min(best, b);
                }
                const double v = std::floor((best - half_diag) / (double)q);
                (*out)[((size_t)z * dims[1] + y) * dims[0] + x] = (uint8_t)std::min(std::max(v, 0.0), 255.0);
            }
    for (int k = 0; k < 3; ++k) {
        h.dist_lo[k] = box.lo[k];
        h.dist_hi[k] = box.lo[k] + (float)dims[k] * cell;
        h.dist_off[k] = off[k];
    }
    h.dist_cell = cell;
    h.dist_inv_cell = inv_cell;
    h.dist_q = q;
    h.dist_pad = pad;
    h.dist_nx = dims[0];
    h.dist_ny = dims[1];
    h.dist_nz = dims[2];
    return true;
}

}  // namespace

FlatScene flatten(const Scene& scene, int accel) {
    FlatScene fs;
    std::memset(&fs.header, 0, sizeof fs.header);
    fs.diffuse_without_light = false;
    fs.cuboid_light_without_area = false;

    // data tables
    std::map<uint64_t, uint32_t> mat_index, vol_index;
    std::vector<float4> mats, vols;
    for (std::map<uint64_t, Data>::const_iterator it = scene.data.begin(); it != scene.data.end(); ++it) {
        const Data& d = it->second;
        if (d.kind == DATA_MATERIAL) {
            mat_index[it->first] = (uint32_t)(mats.size() / MAT_STRIDE);
            mats.push_back(f4(d.albedo[0], d.albedo[1], d.albedo[2], as_f((uint32_t)d.mat_kind)));
            mats.push_back(f4(d.roughness, d.ior, d.intensity, 0.0f));
        } else {
            if (d.buffer.size() != d.width * d.height * d.depth && d.width && d.height && d.depth)
                throw SceneError("index out of bounds: density buffer length does not match width*height*depth");
            for (int k = 0; k < 3; ++k) {
                uint64_t dim = k == 0 ? d.width : k == 1 ? d.height : d.depth;
                if (dim && !(d.size[k] >= 0.0f && std::ceil(d.size[k]) <= (float)(dim - 1))) throw SceneError("volume index out of bounds");
            }
            for (size_t i = 0; i < d.buffer.size(); ++i)
                if (!(d.buffer[i] >= 0.0f)) throw SceneError("p is outside range [0.0, 1.0] (negative or NaN density)");
            vol_index[it->first] = (uint32_t)(vols.size() / VOL_STRIDE);
            vols.push_back(f4(as_f((uint32_t)d.width), as_f((uint32_t)d.height), as_f((uint32_t)d.depth), as_f((uint32_t)fs.grids.size())));
            vols.push_back(f4(d.size[0], d.size[1], d.size[2], 0.0f));
            fs.grids.insert(fs.grids.end(), d.buffer.begin(), d.buffer.end());
        }
    }
    // root material folded to the ColorData sample_root returns (src/tracer/mod.rs:429-452)
    {
        const Data& d = scene.get_data(scene.root_material);
        if (d.kind != DATA_MATERIAL) throw SceneError("expected root material to be a material");
        SceneHeader& h = fs.header;
        for (int k = 0; k < 3; ++k) {
            switch (d.mat_kind) {
                case MAT_FLAT: h.root_color[k] = 0.0f + d.albedo[k]; h.root_albedo[k] = 0.0f; break;
                case MAT_EMISSIVE: h.root_color[k] = 0.0f + d.albedo[k] * d.intensity; h.root_albedo[k] = 0.0f; break;
                default: h.root_color[k] = d.albedo[k] + 0.0f; h.root_albedo[k] = d.albedo[k]; break;
            }
        }
        h.root_keeps_normal = d.mat_kind == MAT_EMISSIVE ? 0u : 1u;
    }

    // BT_ACCEL_LINEAR_FACES keeps the literal tests: six Rect::hit per cuboid, the general rect test everywhere
    const bool aa_rects = accel != ACCEL_LINEAR_FACES && !std::getenv("BT_NO_AA_RECTS");
    const EmitCtx ctx = {scene, mat_index, vol_index, aa_rects};
    std::vector<float4> prims, lights, face_lights, boxes;
    std::vector<size_t> cuboid_lights;  // offsets of the LIGHT_CUBOID records in `lights`
    std::vector<std::pair<uint32_t, uint32_t> > box_of_prim;  // (first face record, box index)
    std::vector<Bounds> bounds;
    bool any_diffuse = false;
    for (std::map<uint64_t, Object>::const_iterator it = scene.objects.begin(); it != scene.objects.end(); ++it) {
        const uint32_t obj = (uint32_t)fs.object_refs.size(), first_prim = (uint32_t)(prims.size() / PRIM_STRIDE);
        fs.object_refs.push_back(it->first);
        const ObjRecords rec = emit_object(ctx, it->second, obj, first_prim);
        ObjSpan span = {first_prim, (uint32_t)(rec.prims.size() / PRIM_STRIDE), -1, -1, false};
        prims.insert(prims.end(), rec.prims.begin(), rec.prims.end());
        bounds.insert(bounds.end(), rec.bounds.begin(), rec.bounds.end());
        any_diffuse |= rec.any_diffuse;
        if (rec.has_volume) fs.header.has_volume_prims = 1;
        if (rec.has_box) {  // q4.z of the first face: 1 + box index (cuboid faces carry no area)
            span.box = (int32_t)(boxes.size() / BOX_STRIDE);
            box_of_prim.push_back(std::make_pair(first_prim, (uint32_t)span.box));
            boxes.insert(boxes.end(), rec.box, rec.box + BOX_STRIDE);
        }
        if (rec.is_light) {
            const size_t base = lights.size();
            span.light = (int32_t)(base / LIGHT_STRIDE);
            lights.insert(lights.end(), rec.light.begin(), rec.light.end());
            if (!rec.face_lights.empty()) {  // a LIGHT Cuboid: l2.z = index of its first face sub-record (made absolute below)
                span.cuboid_light = true;
                lights[base + 2].z = as_f((uint32_t)(face_lights.size() / LIGHT_STRIDE));
                cuboid_lights.push_back(base);
                face_lights.insert(face_lights.end(), rec.face_lights.begin(), rec.face_lights.end());
                fs.header.content |= CT_CUBOID_LIGHT;
                if (rec.zero_area) fs.cuboid_light_without_area = true;  // WeightedIndex::new(..).unwrap() panics
            }
        }
        fs.spans.push_back(span);
    }
    // object lights first (Uniform::new(0, count) indexes them), the cuboid face sub-records behind
    const uint32_t n_object_lights = (uint32_t)(lights.size() / LIGHT_STRIDE);
    for (size_t i = 0; i < cuboid_lights.size(); ++i) {
        uint32_t rel;
        std::memcpy(&rel, &lights[cuboid_lights[i] + 2].z, 4);
        lights[cuboid_lights[i] + 2].z = as_f(n_object_lights + rel);
    }
    lights.insert(lights.end(), face_lights.begin(), face_lights.end());

    std::vector<float4> lens;
    for (size_t i = 0; i < scene.lenses.size(); ++i) {
        const Lens& l = scene.lenses[i];
        if (!(l.rs > 0.0f)) continue;  // r_s <= 0: no mass -> exact flat limit
        lens.push_back(f4(l.c[0], l.c[1], l.c[2], -1.5f * l.rs));
        lens.push_back(f4(l.rs, scene.lens_config.r_far * l.rs, 0.0f, 0.0f));
    }

    SceneHeader& h = fs.header;
    h.n_prims = (uint32_t)(prims.size() / PRIM_STRIDE);
    h.n_mats = (uint32_t)(mats.size() / MAT_STRIDE);
    h.n_lights = n_object_lights;
    h.n_vols = (uint32_t)(vols.size() / VOL_STRIDE);
    h.n_lens = (uint32_t)(lens.size() / LENS_STRIDE);
    h.prim_off = 0;
    h.content &= CT_CUBOID_LIGHT;  // (set while flattening the lights)
    for (uint32_t i = 0; i < h.n_prims; ++i) {
        uint32_t type;
        std::memcpy(&type, &prims[(size_t)i * PRIM_STRIDE + 4].x, 4);
        h.content |= (type & 3u) == PRIM_SPHERE ? CT_SPHERES : CT_RECTS;
    }
    if (h.has_volume_prims) h.content |= CT_VOLUMES;
    for (std::map<uint64_t, Data>::const_iterator it = scene.data.begin(); it != scene.data.end(); ++it) {
        if (it->second.kind != DATA_MATERIAL) continue;
        if (it->second.mat_kind == MAT_METALLIC) h.content |= CT_METAL;
        if (it->second.mat_kind == MAT_GLASS) h.content |= CT_GLASS;
    }
    // acceleration structure: the linear scan of the reference for small scenes, a BVH beyond
    bool use_bvh = accel == ACCEL_BVH || (accel == ACCEL_AUTO && h.n_prims > (uint32_t)BVH_AUTO_PRIMS);
    if (h.has_volume_prims) use_bvh = false;  // hit_volumetric is scan-order dependent (mod.rs:414-424)
    std::vector<float4> nodes;
    for (uint32_t i = 0; i < h.n_prims; ++i) fs.prim_order.push_back(i);
    if (use_bvh && h.n_prims > 0) {
        BvhBuild bvh(bounds);
        for (uint32_t i = 0; i < h.n_prims; ++i) bvh.sphere.push_back((as_u(prims[(size_t)i * PRIM_STRIDE + 4].x) & 3u) == (uint32_t)PRIM_SPHERE);
        // primitives that span a large part of the scene (a ground sphere of radius 100 ...) would
        // bloat every node they fall into: they go to one leaf beside the tree of the rest
        std::vector<float> diag(h.n_prims);
        for (uint32_t i = 0; i < h.n_prims; ++i) {
            float d2 = 0.0f;
            for (int k = 0; k < 3; ++k) d2 += (bounds[i].hi[k] - bounds[i].lo[k]) * (bounds[i].hi[k] - bounds[i].lo[k]);
            diag[i] = std::sqrt(d2);
        }
        std::vector<float> sorted_diag(diag);
        std::nth_element(sorted_diag.begin(), sorted_diag.begin() + sorted_diag.size() / 2, sorted_diag.end());
        const float big_cut = 16.0f * std::max(sorted_diag[sorted_diag.size() / 2], 1e-6f);
        uint32_t n_big = (uint32_t)(std::stable_partition(bvh.order.begin(), bvh.order.end(),
                                                          [&](uint32_t i) { return diag[i] > big_cut; }) - bvh.order.begin());
        Bounds all = BvhBuild::empty();
        for (uint32_t i = 0; i < h.n_prims; ++i) BvhBuild::grow(all, bounds[i]);
        if (n_big == h.n_prims || n_big > (uint32_t)BVH_LEAF_MAX) n_big = 0;  // (too many to sit in one leaf: no special case)
        // node 0 is always an inner node: (left = big-primitive leaf or empty leaf, right = the tree)
        bvh.make_inner(0, all, 0, all);
        Bounds rest_box;
        uint32_t rest = bvh.build(n_big, h.n_prims - n_big, 1, &rest_box);
        uint32_t big = bvh.leaf_ref(0, n_big);
        if (h.n_prims >= 0x00fffff0u) throw SceneError("BVH: too many primitives for a leaf reference");
        bvh.set_inner(0, big, n_big ? all : BvhBuild::empty(), rest, rest_box);
        bvh.collapse(0);  // wide node 0 = the root
        std::vector<float4> sorted(prims.size());
        std::vector<uint32_t> where(h.n_prims);
        for (uint32_t pos = 0; pos < h.n_prims; ++pos) {
            where[bvh.order[pos]] = pos;
            for (int k = 0; k < PRIM_STRIDE; ++k) sorted[pos * PRIM_STRIDE + k] = prims[bvh.order[pos] * PRIM_STRIDE + k];
        }
        prims.swap(sorted);
        fs.prim_order = bvh.order;
        nodes.swap(bvh.wide);
        for (size_t l = 0; l < lights.size(); l += LIGHT_STRIDE) {  // lights point at their primitive record
            uint32_t first;
            std::memcpy(&first, &lights[l].y, 4);
            uint32_t count;
            std::memcpy(&count, &lights[l].z, 4);
            if (count) lights[l].y = as_f(where[first]);
        }
    }
    fs.blob = prims;
    h.mat_off = (uint32_t)fs.blob.size();
    fs.blob.insert(fs.blob.end(), mats.begin(), mats.end());
    h.light_off = (uint32_t)fs.blob.size();
    fs.blob.insert(fs.blob.end(), lights.begin(), lights.end());
    h.vol_off = (uint32_t)fs.blob.size();
    fs.blob.insert(fs.blob.end(), vols.begin(), vols.end());
    h.lens_off = (uint32_t)fs.blob.size();
    fs.blob.insert(fs.blob.end(), lens.begin(), lens.end());
    // BOX records (linear-scan scenes): the first face of each box-shaped cuboid points at its record
    h.box_off = (uint32_t)fs.blob.size();
    h.n_boxes = 0;
    if (nodes.empty() && accel != ACCEL_LINEAR_FACES) {
        h.n_boxes = (uint32_t)(boxes.size() / BOX_STRIDE);
        fs.blob.insert(fs.blob.end(), boxes.begin(), boxes.end());
        for (size_t i = 0; i < box_of_prim.size(); ++i)
            fs.blob[(size_t)box_of_prim[i].first * PRIM_STRIDE + 4].z = as_f(box_of_prim[i].second + 1u);
    }
    // world AABBs for the stepper's free-distance query (scan scenes under a lens field only)
    h.bound_off = (uint32_t)fs.blob.size();
    h.lens_skip = 0;
    if (h.n_lens > 0 && nodes.empty() && !(scene.lens_config.flags & 2u)) {
        h.lens_skip = 1;
        for (uint32_t i = 0; i < h.n_prims; ++i) {
            fs.blob.push_back(f4(bounds[i].lo[0], bounds[i].lo[1], bounds[i].lo[2], 0.0f));
            fs.blob.push_back(f4(bounds[i].hi[0], bounds[i].hi[1], bounds[i].hi[2], 0.0f));
        }
        if (!std::getenv("BT_NO_DIST_GRID") && build_dist_grid(prims, bounds, h, &fs.dist, std::getenv("BT_DIST_GRID_HOST") != 0)) h.lens_skip = 3;
    }
    if (!nodes.empty())
        while (fs.blob.size() % BVH_STRIDE) fs.blob.push_back(f4(0, 0, 0, 0));  // a node = one 128-byte line
    h.bvh_off = (uint32_t)fs.blob.size();
    h.n_bvh = (uint32_t)(nodes.size() / BVH_STRIDE);
    fs.blob.insert(fs.blob.end(), nodes.begin(), nodes.end());
    h.blob_f4 = (uint32_t)fs.blob.size();
    // shared-memory staging: everything for the linear scan; under a BVH the primitives and nodes
    // stay in global memory (L2 / HBM) and only the small tables are staged
    h.stage_off = h.n_bvh ? h.mat_off : 0;
    h.stage_f4 = h.bvh_off - h.stage_off;
    h.kappa = scene.lens_config.kappa;
    h.h_min = scene.lens_config.h_min;
    h.h_max = scene.lens_config.h_max;
    h.max_steps = scene.lens_config.max_steps;
    h.lens_exact = scene.lens_config.flags & 1u;
    fs.diffuse_without_light = any_diffuse && h.n_lights == 0;
    fs.where.assign(h.n_prims, 0);
    for (uint32_t pos = 0; pos < h.n_prims; ++pos) fs.where[fs.prim_order[pos]] = pos;
    fs.prim_bounds = bounds;
    fs.accel = accel;
    if (fs.blob.empty()) fs.blob.push_back(f4(0, 0, 0, 0));
    if (fs.grids.empty()) fs.grids.push_back(0.0f);
    return fs;
}

namespace {
// Recompute every node box of the BVH from the primitives' current bounds: same topology, same leaves.  Children are
// stored behind their parent (BvhBuild::collapse reserves the parent's slot first), so one backward sweep sees every
// child before its parent.
void refit_bvh(FlatScene& fs) {
    const SceneHeader& h = fs.header;
    float4* nodes = &fs.blob[h.bvh_off];
    std::vector<Bounds> own(h.n_bvh, BvhBuild::empty());  // unpadded box of each inner node
    auto child_box = [&](uint32_t ref) {
        if (!(ref & BVH_LEAF)) return own[ref];
        Bounds b = BvhBuild::empty();
        const uint32_t first = ref & 0x00ffffffu, count = (ref >> 24) & 0x1fu;
        for (uint32_t pos = first; pos < first + count; ++pos) BvhBuild::grow(b, fs.prim_bounds[fs.prim_order[pos]]);
        return b;
    };
    for (uint32_t n = h.n_bvh; n-- > 0;) {
        float4* q = nodes + (size_t)n * BVH_STRIDE;
        const uint32_t ref[BVH_WIDTH] = {as_u(q[6].x), as_u(q[6].y), as_u(q[6].z), as_u(q[6].w)};
        BvhBuild::Child c[BVH_WIDTH];
        int m = 0;
        for (; m < (int)BVH_WIDTH && ref[m] != (uint32_t)BVH_EMPTY; ++m) {
            c[m].ref = ref[m];
            c[m].box = child_box(ref[m]);
            BvhBuild::grow(own[n], c[m].box);
        }
        BvhBuild::write_wide(q, c, m);
    }
}
}  // namespace

bool update_flat(FlatScene& fs, const Scene& scene, const std::vector<uint64_t>& refs, std::vector<std::pair<uint32_t, uint32_t> >* dirty,
                 bool* dist_changed) {
    *dist_changed = false;
    SceneHeader& h = fs.header;
    // the data tables in the order flatten() numbers them
    std::map<uint64_t, uint32_t> mat_index, vol_index;
    {
        uint32_t nm = 0, nv = 0;
        for (std::map<uint64_t, Data>::const_iterator it = scene.data.begin(); it != scene.data.end(); ++it)
            if (it->second.kind == DATA_MATERIAL) mat_index[it->first] = nm++; else vol_index[it->first] = nv++;
    }
    const EmitCtx ctx = {scene, mat_index, vol_index, fs.accel != ACCEL_LINEAR_FACES && !std::getenv("BT_NO_AA_RECTS")};
    std::map<uint64_t, uint32_t> index_of;
    for (uint32_t i = 0; i < fs.object_refs.size(); ++i) index_of[fs.object_refs[i]] = i;
    if (index_of.size() != scene.objects.size()) return false;
    // first pass: everything must keep its shape
    std::vector<std::pair<uint32_t, ObjRecords> > recs;
    for (size_t k = 0; k < refs.size(); ++k) {
        std::map<uint64_t, uint32_t>::const_iterator it = index_of.find(refs[k]);
        if (it == index_of.end()) return false;
        const uint32_t obj = it->second;
        const ObjSpan& sp = fs.spans[obj];
        ObjRecords rec = emit_object(ctx, scene.get_object(refs[k]), obj, sp.first_prim);
        const bool boxes_used = h.n_bvh == 0 && fs.accel != ACCEL_LINEAR_FACES;
        if (rec.prims.size() / PRIM_STRIDE != sp.n_prims || rec.is_light != (sp.light >= 0) || sp.cuboid_light || !rec.face_lights.empty() ||
            (boxes_used && rec.has_box != (sp.box >= 0)))
            return false;
        for (uint32_t i = 0; i < sp.n_prims; ++i) {  // a rect that stops (or starts) being axis-aligned changes its record type only
            const uint32_t pos = fs.where[sp.first_prim + i];
            const uint32_t was = as_u(fs.blob[h.prim_off + (size_t)pos * PRIM_STRIDE + 4].x) & 3u, is = as_u(rec.prims[(size_t)i * PRIM_STRIDE + 4].x) & 3u;
            if ((was == PRIM_SPHERE) != (is == PRIM_SPHERE)) return false;
        }
        recs.push_back(std::make_pair(obj, rec));
    }
    // second pass: overwrite in place
    for (size_t k = 0; k < recs.size(); ++k) {
        const uint32_t obj = recs[k].first;
        const ObjRecords& rec = recs[k].second;
        const ObjSpan& sp = fs.spans[obj];
        for (uint32_t i = 0; i < sp.n_prims; ++i) {
            const uint32_t canon = sp.first_prim + i, pos = fs.where[canon];
            const size_t at = h.prim_off + (size_t)pos * PRIM_STRIDE;
            for (int j = 0; j < PRIM_STRIDE; ++j) fs.blob[at + j] = rec.prims[(size_t)i * PRIM_STRIDE + j];
            if (i == 0 && sp.box >= 0 && h.n_boxes) fs.blob[at + 4].z = as_f((uint32_t)sp.box + 1u);
            dirty->push_back(std::make_pair((uint32_t)at, (uint32_t)PRIM_STRIDE));
            fs.prim_bounds[canon] = rec.bounds[i];
            if (h.lens_skip) {
                const size_t b = h.bound_off + (size_t)canon * BOUND_STRIDE;
                fs.blob[b] = f4(rec.bounds[i].lo[0], rec.bounds[i].lo[1], rec.bounds[i].lo[2], 0.0f);
                fs.blob[b + 1] = f4(rec.bounds[i].hi[0], rec.bounds[i].hi[1], rec.bounds[i].hi[2], 0.0f);
                dirty->push_back(std::make_pair((uint32_t)b, (uint32_t)BOUND_STRIDE));
            }
        }
        if (sp.box >= 0 && h.n_boxes) {
            const size_t b = h.box_off + (size_t)sp.box * BOX_STRIDE;
            for (int j = 0; j < BOX_STRIDE; ++j) fs.blob[b + j] = rec.box[j];
            dirty->push_back(std::make_pair((uint32_t)b, (uint32_t)BOX_STRIDE));
        }
        if (sp.light >= 0) {
            const size_t l = h.light_off + (size_t)sp.light * LIGHT_STRIDE;
            for (int j = 0; j < LIGHT_STRIDE; ++j) fs.blob[l + j] = rec.light[j];
            if (as_u(rec.light[0].z)) fs.blob[l].y = as_f(fs.where[sp.first_prim]);  // lights point at their primitive RECORD
            dirty->push_back(std::make_pair((uint32_t)l, (uint32_t)LIGHT_STRIDE));
        }
    }
    if (h.n_bvh) {
        refit_bvh(fs);
        dirty->push_back(std::make_pair(h.bvh_off, h.n_bvh * (uint32_t)BVH_STRIDE));
    }
    if (h.lens_skip == 3) {  // the free-distance grid describes the old geometry: rebuilt (host, tens of ms -- see DESIGN.md)
        std::vector<float4> canon_prims((size_t)h.n_prims * PRIM_STRIDE);
        for (uint32_t c = 0; c < h.n_prims; ++c)
            for (int j = 0; j < PRIM_STRIDE; ++j) canon_prims[(size_t)c * PRIM_STRIDE + j] = fs.blob[h.prim_off + (size_t)fs.where[c] * PRIM_STRIDE + j];
        if (!build_dist_grid(canon_prims, fs.prim_bounds, h, &fs.dist, std::getenv("BT_DIST_GRID_HOST") != 0)) h.lens_skip = 1;
        *dist_changed = true;
    }
    return true;
}

CameraBlock make_camera_block(const Scene& scene, uint64_t camera_ref, uint32_t width, uint32_t height, uint32_t subsample) {
    const Object& o = scene.get_object(camera_ref);
    if (o.kind != OBJ_CAMERA) throw SceneError("expected a camera object");
    CameraBlock c;
    std::memset(&c, 0, sizeof c);
    for (int i = 0; i < 9; ++i) c.m[i] = o.transform_world.f[i];
    for (int i = 0; i < 3; ++i) c.t[i] = o.transform_world.f[9 + i];
    const Camera& cam = o.camera;
    c.yfov = 2.0f * std::atan2(cam.sensor_size, 2.0f * cam.focal_length);  // mod.rs:248
    c.xfov = c.yfov * cam.aspect_ratio;                                     // mod.rs:249
    c.pixel_width = 2.0f * (1.0f / (float)width);                           // buffer.rs:68-76
    c.pixel_height = 2.0f * (1.0f / (float)height);
    float subpixel_scale = subsample == 0 ? 1.0f : 1.0f / (float)subsample;  // mod.rs:55-60
    c.su_low = -0.5f * c.pixel_width * subpixel_scale;                      // mod.rs:255-265
    c.su_scale = uniform_scale(c.su_low, 0.5f * c.pixel_width * subpixel_scale);
    c.sv_low = -0.5f * c.pixel_height * subpixel_scale;
    c.sv_scale = uniform_scale(c.sv_low, 0.5f * c.pixel_height * subpixel_scale);
    c.sub_width = subsample == 0 ? 0.0f : 1.0f / (float)subsample;
    c.sub_n = subsample == 0 ? 1u : subsample;
    c.projection = cam.projection;
    c.has_focus = cam.has_focus && cam.projection == PROJ_PERSPECTIVE ? 1u : 0u;  // a panorama is a pinhole
    c.focus = cam.focus;
    c.aperture = 0.5f * cam.focal_length / cam.fstop;  // mod.rs:289
    // UnitDisk::new(Vec3::NEG_Z): any_orthonormal_pair((0,0,-1)) = ((1,-0,0),(0,-1,-0))
    c.disk_x[0] = 1.0f; c.disk_x[1] = -0.0f; c.disk_x[2] = 0.0f;
    c.disk_y[0] = 0.0f; c.disk_y[1] = -1.0f; c.disk_y[2] = -0.0f;
    return c;
}

}  // namespace bt
