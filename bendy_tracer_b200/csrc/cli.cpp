// cli.cpp -- headless stand-in for the reference's window loop (src/main.rs:49-72, 74-254, 275-298),
// written against the C ABI only (include/bendy_b200.h).
//
//   bendy_b200_cli --output full|albedo|normal [--width 768] [--height 512] [--samples 64]
//                  [--subsample 2] [--screenshot screenshots/render.png] [--scene scene.json]
//                  [--lens x,y,z,r_s] [--environment sky.pfm] [--projection perspective|equirectangular]
//                  [--seed 0] [--save-scene out.json(.gz)]
//
// Same flags, defaults and semantics as the reference's clap CLI: `--output` is required; the scene
// file is read when it exists (gzip when the extension is .gz), otherwise the built-in Cornell box
// is used (main.rs:108-213); the camera tagged "camera" gets aspect_ratio = width / height
// (main.rs:216-223); the tracer runs ONE pass per iteration (`samples = 1`) until
// buffer.samples() >= --samples (main.rs:248-254; buffer.samples() counts sub-samples); the preview
// is written as PNG (what Ctrl+P does, main.rs:275-298).  Instead of the title bar the per-pass
// time, average and total are printed to stderr (main.rs:352-388).  --environment (an extension, like --lens) sets an
// equirectangular environment map from a PFM file (bt_scene_set_environment); a malformed file is an error even in the
// GPU-less --samples 0 dry run.  --projection equirectangular (an extension too) renders the whole sphere around the
// camera (bt_scene_set_camera_projection; --width = 2 --height gives square pixels); an unknown value is an error before
// any GPU work.
#include <zlib.h>

#include <cctype>
#include <chrono>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <filesystem>
#include <fstream>
#include <sstream>
#include <string>
#include <vector>

#include "../../include/bendy_b200.h"

namespace {

[[noreturn]] void die(const std::string& msg) {
    std::fprintf(stderr, "error: %s\n", msg.c_str());
    std::exit(2);
}
void ck(int code, const char* what) {
    if (code != BT_OK) die(std::string(what) + ": " + bt_last_error());
}

// ---- the built-in scene of main.rs:108-213, emitted in the scene wire format -----------------
std::string fnum(double v) {
    char b[40];
    std::snprintf(b, sizeof b, "%.9g", (double)(float)v);
    std::string s(b);
    if (s.find_first_of(".e") == std::string::npos) s += ".0";
    return s;
}
std::string vec3(double x, double y, double z) { return "[" + fnum(x) + "," + fnum(y) + "," + fnum(z) + "]"; }
struct V {
    double x, y, z;
};
V cross(V a, V b) { return {a.y * b.z - a.z * b.y, a.z * b.x - a.x * b.z, a.x * b.y - a.y * b.x}; }
double len(V a) { return std::sqrt(a.x * a.x + a.y * a.y + a.z * a.z); }
// Rect::new(material, x, y): half extents are the lengths, axes are normalised, z = x cross y
std::string rect(int mat, V x, V y) {
    double hw = len(x), hh = len(y);
    V xn = {x.x / hw, x.y / hw, x.z / hw}, yn = {y.x / hh, y.y / hh, y.z / hh}, z = cross(xn, yn);
    return "{\"material\":" + std::to_string(mat) + ",\"half_width\":" + fnum(hw) + ",\"half_height\":" + fnum(hh) +
           ",\"x\":" + vec3(xn.x, xn.y, xn.z) + ",\"y\":" + vec3(yn.x, yn.y, yn.z) + ",\"z\":" + vec3(z.x, z.y, z.z) + "}";
}
V neg(V a) { return {-a.x, -a.y, -a.z}; }
// Cuboid::new(material, x, y, z): the six (offset, Rect) pairs of cuboid.rs:19-30
std::string cuboid(int mat, V x, V y, V z) {
    struct F {
        V off, a, b;
    } f[6] = {{neg(z), x, y}, {z, neg(x), y}, {neg(x), z, y}, {x, neg(z), y}, {neg(y), x, z}, {y, x, neg(z)}};
    std::string s = "{\"Cuboid\":{\"faces\":[";
    for (int i = 0; i < 6; ++i)
        s += std::string(i ? "," : "") + "[" + vec3(f[i].off.x, f[i].off.y, f[i].off.z) + "," + rect(mat, f[i].a, f[i].b) + "]";
    return s + "]}}";
}
std::string object(int key, const std::string& inner, const double m[9], V t, int flags, const char* tag) {
    std::string tf = "[";
    for (int i = 0; i < 9; ++i) tf += fnum(m[i]) + ",";
    tf += fnum(t.x) + "," + fnum(t.y) + "," + fnum(t.z) + "]";
    return "\"" + std::to_string(key) + "\":{\"object_ref\":" + std::to_string(key) + ",\"tag\":" +
           (tag ? "\"" + std::string(tag) + "\"" : std::string("null")) + ",\"flags\":{\"bits\":" + std::to_string(flags) +
           "},\"transform\":{\"transform_world\":" + tf + ",\"transform_local\":" + tf + ",\"transform_parent\":null},\"inner\":" +
           inner + ",\"children\":null}";
}
std::string material(int key, const char* kind, double r, double g, double b, const char* extra) {
    return "\"" + std::to_string(key) + "\":{\"inner\":{\"Material\":{\"" + kind + "\":{\"albedo\":{\"r\":" + fnum(r) + ",\"g\":" +
           fnum(g) + ",\"b\":" + fnum(b) + "}" + extra + "}}}}";
}
std::string builtin_cornell() {
    const double I[9] = {1, 0, 0, 0, 1, 0, 0, 0, 1};
    // Affine3A::from_rotation_translation(Quat::from_euler(YXZ, 20 deg, 0, 0), ..) = Ry(20 deg); the
    // two f32 values are the ones the reference's own build serialised (cornell2.json.gz, object 7)
    const double c20 = 0.9396926, s20 = 0.34202018;
    const double R[9] = {c20, 0, -s20, 0, 1, 0, s20, 0, c20};
    // data keys: 0 root (Scene::new), 1 light, 2 white, 3 metal, 4 red, 5 green
    std::string data = material(0, "Flat", 0, 0, 0, "") + "," + material(1, "Emissive", 1, 1, 1, ",\"intensity\":20.0") + "," +
                       material(2, "Diffuse", 0.73, 0.73, 0.73, ",\"roughness\":1.0") + "," +
                       material(3, "Metallic", 0.55, 0.55, 0.55, ",\"roughness\":0.01") + "," +
                       material(4, "Diffuse", 0.7, 0.1, 0.1, ",\"roughness\":0.5") + "," +
                       material(5, "Diffuse", 0.2, 0.7, 0.4, ",\"roughness\":0.8");
    std::string cam = "{\"Camera\":{\"sensor_size\":0.024,\"focal_length\":0.05,\"aspect_ratio\":1.5,\"fstop\":1.4,\"focus\":12.5}}";
    auto R_ = [](int m, V x, V y) { return "{\"Rect\":" + rect(m, x, y) + "}"; };
    std::string objs = object(0, cam, I, {0, 2.5, 10}, 0, "camera") + "," +
                       object(1, R_(5, {0, 0, -2.5}, {0, 2.5, 0}), I, {-2.5, 2.5, -2.5}, 0, nullptr) + "," +   // left
                       object(2, R_(4, {0, 0, 2.5}, {0, 2.5, 0}), I, {2.5, 2.5, -2.5}, 0, nullptr) + "," +     // right
                       object(3, R_(2, {2.5, 0, 0}, {0, 2.5, 0}), I, {0, 2.5, -5}, 0, nullptr) + "," +         // back
                       object(4, R_(2, {2.5, 0, 0}, {0, 0, -2.5}), I, {0, 0, -2.5}, 0, nullptr) + "," +        // floor
                       object(5, R_(2, {2.5, 0, 0}, {0, 0, 2.5}), I, {0, 5, -2.5}, 0, nullptr) + "," +         // ceiling
                       object(6, R_(1, {0.5, 0, 0}, {0, 0, 0.5}), I, {0, 4.999, -2.5}, 1, nullptr) + "," +     // light
                       object(7, cuboid(3, {0.5, 0, 0}, {0, 1, 0}, {0, 0, 0.4}), R, {-1.2, 1, -3.2}, 0, nullptr) + "," +
                       object(8, cuboid(2, {0.5, 0, 0}, {0, 0.6, 0}, {0, 0, 0.5}), I, {1, 0.6, -1.4}, 0, nullptr);
    return "{\"roots\":[],\"root_material\":0,\"objects\":{\"collection\":{" + objs + "},\"next_key\":9},\"data\":{\"collection\":{" +
           data + "},\"next_key\":6}}";
}

// ---- PNG (RGBA8, zlib deflate) -----------------------------------------------------------
void put32(std::vector<unsigned char>& v, uint32_t x) {
    for (int s = 24; s >= 0; s -= 8) v.push_back((unsigned char)(x >> s));
}
void chunk(std::vector<unsigned char>& png, const char* type, const std::vector<unsigned char>& body) {
    put32(png, (uint32_t)body.size());
    size_t at = png.size();
    png.insert(png.end(), type, type + 4);
    png.insert(png.end(), body.begin(), body.end());
    put32(png, (uint32_t)crc32(0, png.data() + at, (uInt)(png.size() - at)));
}
bool write_png(const std::string& path, const std::vector<uint8_t>& rgba, uint32_t w, uint32_t h) {
    std::vector<unsigned char> raw;
    raw.reserve((size_t)h * (w * 4 + 1));
    for (uint32_t y = 0; y < h; ++y) {
        raw.push_back(0);
        raw.insert(raw.end(), rgba.begin() + (size_t)y * w * 4, rgba.begin() + (size_t)(y + 1) * w * 4);
    }
    uLongf cap = compressBound((uLong)raw.size());
    std::vector<unsigned char> z(cap);
    if (compress2(z.data(), &cap, raw.data(), (uLong)raw.size(), 6) != Z_OK) return false;
    z.resize(cap);
    std::vector<unsigned char> png = {0x89, 'P', 'N', 'G', 0x0d, 0x0a, 0x1a, 0x0a}, ihdr;
    put32(ihdr, w);
    put32(ihdr, h);
    const unsigned char tail[5] = {8, 6, 0, 0, 0};  // 8 bit, RGBA
    ihdr.insert(ihdr.end(), tail, tail + 5);
    chunk(png, "IHDR", ihdr);
    chunk(png, "IDAT", z);
    chunk(png, "IEND", std::vector<unsigned char>());
    std::ofstream f(path, std::ios::binary);
    f.write((const char*)png.data(), (std::streamsize)png.size());
    return (bool)f;
}

// ---- PFM (the float image format: "PF" RGB / "Pf" grey, then "W H", then scale -- negative: little-endian --, one
// whitespace byte and W * H pixels of 32-bit floats, bottom row first) -> top-row-first RGB -------------------
std::vector<float> read_pfm(const std::string& path, uint32_t* w_out, uint32_t* h_out) {
    std::ifstream in(path, std::ios::binary);
    if (!in) die("cannot open environment map " + path);
    std::string bytes((std::istreambuf_iterator<char>(in)), std::istreambuf_iterator<char>());
    size_t at = 0;
    auto token = [&]() -> std::string {
        while (at < bytes.size() && std::isspace((unsigned char)bytes[at])) ++at;
        const size_t start = at;
        while (at < bytes.size() && !std::isspace((unsigned char)bytes[at])) ++at;
        return bytes.substr(start, at - start);
    };
    const std::string magic = token(), ws = token(), hs = token(), ss = token();
    if (magic != "PF" && magic != "Pf") die(path + ": not a PFM file (header must start with PF or Pf)");
    char* end = nullptr;
    const unsigned long long w = std::strtoull(ws.c_str(), &end, 10);
    if (ws.empty() || *end || ws[0] == '-' || w == 0) die(path + ": bad PFM width '" + ws + "'");
    const unsigned long long h = std::strtoull(hs.c_str(), &end, 10);
    if (hs.empty() || *end || hs[0] == '-' || h == 0) die(path + ": bad PFM height '" + hs + "'");
    const double scale = std::strtod(ss.c_str(), &end);
    if (ss.empty() || *end || !(scale != 0.0) || !std::isfinite(scale)) die(path + ": bad PFM scale '" + ss + "'");
    if (at >= bytes.size() || !std::isspace((unsigned char)bytes[at])) die(path + ": truncated PFM header");
    ++at;  // the single whitespace byte that ends the header
    if (w >= (1ull << 31) || h >= (1ull << 31) || w * h >= (1ull << 31)) die(path + ": PFM image too large");
    const size_t ch = magic == "PF" ? 3 : 1, n = (size_t)(w * h) * ch;
    if (bytes.size() - at < n * 4)
        die(path + ": truncated PFM data (" + std::to_string(bytes.size() - at) + " bytes, " + std::to_string(n * 4) + " expected)");
    const bool little = scale < 0.0;
    const uint16_t probe = 1;
    const bool host_little = *(const unsigned char*)&probe == 1;
    std::vector<float> rgb((size_t)(w * h) * 3);
    for (size_t y = 0; y < h; ++y)
        for (size_t x = 0; x < w; ++x)
            for (size_t c = 0; c < 3; ++c) {
                unsigned char b[4];
                std::memcpy(b, bytes.data() + at + (((h - 1 - y) * w + x) * ch + (ch == 3 ? c : 0)) * 4, 4);
                if (little != host_little) {
                    std::swap(b[0], b[3]);
                    std::swap(b[1], b[2]);
                }
                std::memcpy(&rgb[(y * w + x) * 3 + c], b, 4);
            }
    *w_out = (uint32_t)w;
    *h_out = (uint32_t)h;
    return rgb;
}

}  // namespace

int main(int argc, char** argv) {
    uint32_t width = 768, height = 512, subsample = 2;
    uint64_t samples = 64, seed = 0;
    int output = -1, projection = BT_PROJECTION_PERSPECTIVE;
    std::string screenshot = "screenshots/render.png", scene_path = "scene.json", save_scene, environment;
    std::vector<float> lens;
    for (int i = 1; i < argc; ++i) {
        std::string a = argv[i];
        auto val = [&]() -> std::string {
            if (i + 1 >= argc) die("missing value for " + a);
            return argv[++i];
        };
        if (a == "--width") width = (uint32_t)std::stoul(val());
        else if (a == "--height") height = (uint32_t)std::stoul(val());
        else if (a == "--samples") samples = std::stoull(val());
        else if (a == "--subsample") subsample = (uint32_t)std::stoul(val());
        else if (a == "--seed") seed = std::stoull(val());
        else if (a == "--screenshot") screenshot = val();
        else if (a == "--scene") scene_path = val();
        else if (a == "--save-scene") save_scene = val();
        else if (a == "--environment") environment = val();
        else if (a == "--projection") {
            std::string v = val();
            projection = v == "perspective" ? BT_PROJECTION_PERSPECTIVE : v == "equirectangular" ? BT_PROJECTION_EQUIRECTANGULAR : -1;
            if (projection < 0) die("invalid value '" + v + "' for '--projection <PROJECTION>' [possible values: perspective, equirectangular]");
        }
        else if (a == "--lens") {
            std::stringstream ss(val());
            std::string tok;
            while (std::getline(ss, tok, ',')) lens.push_back(std::stof(tok));
            if (lens.size() % 4) die("--lens takes x,y,z,r_s[,x,y,z,r_s...]");
        } else if (a == "--output") {
            std::string v = val();
            output = v == "full" ? BT_OUTPUT_FULL : v == "albedo" ? BT_OUTPUT_ALBEDO : v == "normal" ? BT_OUTPUT_NORMAL : -1;
            if (output < 0) die("invalid value '" + v + "' for '--output <OUTPUT>' [possible values: full, albedo, normal]");
        } else {
            die("unexpected argument '" + a + "'");
        }
    }
    if (output < 0) die("the following required arguments were not provided: --output <OUTPUT>");
    if (width == 0 || height == 0) die("empty image");

    bt_scene* scene = nullptr;
    bt_engine* engine = nullptr;  // created after the scene work: --samples 0 is a GPU-less dry run
    std::ifstream in(scene_path, std::ios::binary);
    if (in) {  // main.rs:93-106
        std::string bytes((std::istreambuf_iterator<char>(in)), std::istreambuf_iterator<char>());
        ck(bt_scene_create_json(engine, bytes.data(), bytes.size(), &scene), "scene");
        std::fprintf(stderr, "loaded scene from %s\n", scene_path.c_str());
    } else {   // main.rs:107-213
        std::string text = builtin_cornell();
        ck(bt_scene_create_json(engine, text.data(), text.size(), &scene), "built-in scene");
    }
    if (!lens.empty()) ck(bt_scene_set_lenses(scene, lens.data(), (uint32_t)(lens.size() / 4), nullptr), "lenses");
    if (!environment.empty()) {
        uint32_t ew = 0, eh = 0;
        const std::vector<float> rgb = read_pfm(environment, &ew, &eh);
        ck(bt_scene_set_environment(scene, rgb.data(), ew, eh), ("environment map " + environment).c_str());
        std::fprintf(stderr, "environment map %s: %u x %u\n", environment.c_str(), ew, eh);
    }
    uint64_t camera = 0;
    ck(bt_scene_find_by_tag(scene, "camera", &camera), "find_by_tag(\"camera\")");
    ck(bt_scene_set_camera_aspect(scene, camera, (float)width / (float)height), "camera aspect");  // main.rs:218-223
    if (projection != BT_PROJECTION_PERSPECTIVE) {
        ck(bt_scene_set_camera_projection(scene, camera, projection), "camera projection");
        std::fprintf(stderr, "projection equirectangular: %u x %u\n", width, height);
    }
    if (!save_scene.empty()) {  // what Ctrl+K does, main.rs:299-313 (plain JSON here)
        char* text = nullptr;
        size_t n = 0;
        ck(bt_scene_to_json(scene, &text, &n), "to_json");
        std::ofstream(save_scene, std::ios::binary).write(text, (std::streamsize)n);
        bt_free(text);
        std::fprintf(stderr, "saved scene to %s\n", save_scene.c_str());
    }

    if (samples == 0) {  // Status::Done: nothing to render
        bt_scene_destroy(scene);
        return 0;
    }
    ck(bt_engine_create(0, &engine), "engine");

    bt_config cfg;
    bt_config_default(&cfg);
    cfg.output = output;
    cfg.chunks_x = 8;  // main.rs:225-230
    cfg.chunks_y = 4;
    bt_render_config rc;
    bt_render_config_default(&rc);
    rc.samples = 1;    // one pass per iteration, main.rs:248
    rc.subsample = subsample <= 1 ? 0 : subsample;
    const uint64_t sub = rc.subsample ? (uint64_t)rc.subsample * rc.subsample : 1;

    std::vector<float> buffer((size_t)width * height * 4, 0.0f);  // Buffer::new: BLACK_ALPHA_ONE
    for (size_t i = 3; i < buffer.size(); i += 4) buffer[i] = 1.0f;
    uint64_t have = 0, passes = 0;
    double total = 0.0;
    while (have < samples) {  // main.rs:245-254
        auto t0 = std::chrono::steady_clock::now();
        int32_t status = 0;
        ck(bt_render(engine, scene, camera, &cfg, &rc, seed, have / sub, buffer.data(), BT_MEM_HOST, width, height, &have, &status),
           "render");
        double dt = std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
        total += dt;
        ++passes;
        std::fprintf(stderr, "\rbendy tracer | %llu/%llu samples | %.1f ms/pass | avg %.1f ms | total %.2f s",
                     (unsigned long long)have, (unsigned long long)samples, dt * 1e3, total / passes * 1e3, total);
    }
    std::fprintf(stderr, "\n%.1f Msamples/s\n", (double)width * height * have / total / 1e6);

    std::vector<uint8_t> rgba((size_t)width * height * 4);
    int cs = output == BT_OUTPUT_NORMAL ? BT_CS_NORMAL : BT_CS_SRGB;  // Output::color_space, main.rs:40-46
    ck(bt_resolve_u8(engine, buffer.data(), BT_MEM_HOST, width, height, have, cs, rgba.data()), "resolve");
    if (screenshot.find('.') == std::string::npos) screenshot += "/render.png";  // DEFAULT_SCREENSHOT, main.rs:21,277-281
    size_t slash = screenshot.find_last_of('/');
    if (slash != std::string::npos && slash > 0) {  // fs::create_dir_all(parent), main.rs:283-285
        std::error_code ec;
        std::filesystem::create_directories(screenshot.substr(0, slash), ec);
        if (ec) die("cannot create " + screenshot.substr(0, slash) + ": " + ec.message());
    }
    if (!write_png(screenshot, rgba, width, height)) die("cannot write " + screenshot);
    std::fprintf(stderr, "saved screenshot to %s\n", screenshot.c_str());
    bt_scene_destroy(scene);
    bt_engine_destroy(engine);
    return 0;
}
