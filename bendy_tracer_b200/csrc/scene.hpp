// scene.hpp -- host-side Scene model (serde-compatible with reference src/scene/mod.rs:84-90),
// JSON(.gz) reader / writer and the flattener that produces the device blob of layout.h.
#pragma once
#include <cstdint>
#include <map>
#include <stdexcept>
#include <string>
#include <vector>

#include <vector_types.h>

#include "layout.h"

namespace bt {

struct ParseError : std::runtime_error {
    explicit ParseError(const std::string& m) : std::runtime_error(m) {}
};
struct SceneError : std::runtime_error {  // a condition on which the reference panics
    explicit SceneError(const std::string& m) : std::runtime_error(m) {}
};

struct Affine {  // glam Affine3A: matrix3 columns then translation, 12 floats on the wire
    float f[12];
    static Affine identity() {
        Affine a = {{1, 0, 0, 0, 1, 0, 0, 0, 1, 0, 0, 0}};
        return a;
    }
};
Affine affine_mul(const Affine& a, const Affine& b);
Affine affine_inverse(const Affine& a);

struct Rect {  // reference src/scene/object/rect.rs:11-19
    uint64_t material;
    float half_width, half_height;
    float x[3], y[3], z[3];
};
struct Camera {  // reference src/scene/object/camera.rs:3-10
    float sensor_size, focal_length, aspect_ratio, fstop;
    bool has_focus;
    float focus;
    uint32_t projection;  // PROJ_* (bt_scene_set_camera_projection): host-only, not part of the wire format
};
enum ObjectKind { OBJ_EMPTY, OBJ_CAMERA, OBJ_SPHERE, OBJ_RECT, OBJ_CUBOID };

struct Object {  // reference src/scene/object/mod.rs:33-41
    bool has_object_ref;
    uint64_t object_ref;
    bool has_tag;
    std::string tag;
    uint32_t flags;  // ObjectFlags bits (LIGHT = 1)
    Affine transform_world, transform_local;
    bool has_parent;
    Affine transform_parent;
    ObjectKind kind;
    Camera camera;
    // Sphere (sphere.rs:11-16)
    uint64_t material;
    bool has_volume;
    uint64_t volume;
    float radius;
    Rect rect;
    float face_offset[6][3];  // Cuboid (cuboid.rs:12-15)
    Rect faces[6];
    bool has_children;
    std::vector<uint64_t> children;
};

enum DataKind { DATA_MATERIAL, DATA_VOLUME };
struct Data {  // reference src/scene/data/mod.rs:9-51
    DataKind kind;
    int mat_kind;  // MAT_*
    float albedo[3];
    float roughness, ior, intensity;
    uint64_t width, height, depth;  // DensityMap (volume.rs:75-82)
    float size[3];
    std::vector<float> buffer;
};

struct Lens {
    float c[3];
    float rs;
};

struct LensConfig {
    float kappa, h_min, h_max, r_far;
    uint32_t max_steps;
    uint32_t flags;
};

struct Scene {  // reference src/scene/mod.rs:84-90
    std::vector<uint64_t> roots;
    uint64_t root_material;
    std::map<uint64_t, Object> objects;  // ascending ObjectRef = the canonical iteration order
    uint64_t objects_next_key;
    std::map<uint64_t, Data> data;
    uint64_t data_next_key;
    std::vector<Lens> lenses;  // extension: top-level "lenses" key
    LensConfig lens_config;

    static Scene from_json(const void* bytes, size_t n);  // gzip auto-detected
    std::string to_json() const;

    bool find_by_tag(const char* tag, uint64_t* out) const;  // mod.rs:124-129
    Object& get_object(uint64_t r);                           // mod.rs:131-133 (throws SceneError)
    const Object& get_object(uint64_t r) const;
    const Data& get_data(uint64_t r) const;                   // mod.rs:135-137
    // Object::apply_transform + UpdateQueue::commit (object/mod.rs:200-223, scene/mod.rs:204-213)
    void apply_transform(uint64_t object_ref, const Affine& affine);
};

// where the records of one object live in the flattened scene (update_flat rewrites them in place)
struct ObjSpan {
    uint32_t first_prim, n_prims;   // canonical primitive indices
    int32_t light;                  // index of its record in the light table (-1: not a LIGHT object)
    int32_t box;                    // index of its BOX record (-1: none)
    bool cuboid_light;              // a LIGHT Cuboid (face sub-records: not updated in place)
};
struct AABB {
    float lo[3], hi[3];
};

// The flattened scene: the blob of layout.h + the tables the host keeps.
struct FlatScene {
    SceneHeader header;
    std::vector<float4> blob;
    std::vector<float> grids;
    std::vector<uint8_t> dist;          // free-distance grid (SceneHeader::dist_*); empty unless header.lens_skip == 3
    std::vector<uint64_t> object_refs;  // object index -> ObjectRef
    std::vector<uint32_t> prim_order;   // record position -> canonical primitive index (identity without a BVH)
    std::vector<uint32_t> where;        // canonical primitive index -> record position
    std::vector<ObjSpan> spans;         // per object index
    std::vector<AABB> prim_bounds;      // world AABB per canonical primitive (BVH refit, free-distance grid)
    int accel;                          // the mode it was flattened with
    bool diffuse_without_light;         // a Diffuse material is reachable but no LIGHT exists
    bool cuboid_light_without_area;     // a LIGHT Cuboid whose face areas sum to 0: WeightedIndex::new(..).unwrap() panics (cuboid.rs:49)
};
// accel: 0 = automatic (BVH above BVH_AUTO_PRIMS primitives), 1 = linear scan, 2 = BVH
enum { ACCEL_AUTO = 0, ACCEL_LINEAR = 1, ACCEL_BVH = 2, ACCEL_LINEAR_FACES = 3, BVH_AUTO_PRIMS = 64 };
FlatScene flatten(const Scene& scene, int accel = ACCEL_AUTO);
// Transform-only edits (Object::apply_transform, UpdateQueue::commit -- reference src/scene/mod.rs:154-239): rewrite the records
// of the objects `refs` in place, REFIT the BVH (same topology, new boxes) and list the blob ranges that changed
// (float4 offset, count).  Returns false -- and leaves `fs` untouched -- when the edit changes the layout (a cuboid that stops
// being a box, a LIGHT Cuboid, ...): the caller flattens from scratch.  `dist_changed`: the free-distance grid was rebuilt.
bool update_flat(FlatScene& fs, const Scene& scene, const std::vector<uint64_t>& refs, std::vector<std::pair<uint32_t, uint32_t> >* dirty,
                 bool* dist_changed);

// Uniform<f32>::new / new_inclusive scale (rand 0.8.5 UniformFloat) -- host-side constants
float uniform_scale(float low, float high);
float uniform_scale_inclusive(float low, float high);

// per-call camera block (reference src/tracer/mod.rs:244-267)
CameraBlock make_camera_block(const Scene& scene, uint64_t camera_ref, uint32_t width, uint32_t height,
                              uint32_t subsample);

}  // namespace bt
