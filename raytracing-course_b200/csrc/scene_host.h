// scene_host.h -- host side of the hw5 path: scene description, the reference-order SAH BVH,
// the index BVH built on top of it, and the flattened arrays that are uploaded to HBM.
#pragma once
#include <cstdint>
#include <string>
#include <vector>

#include "vecmath.h"

// Index-BVH child boxes as fp16 (centre, half-extent) instead of (min, max): the slab test then
// runs on the FMA pipe (3 FFMA per child and axis) instead of 2 FFMA + 2 FMNMX; k_traverse is bound
// by the ALU pipe (profiles/r01_experiments.md).  0 selects the min/max layout for A/B runs.
// Index nodes carry a direction cone per child (DESIGN.md "Feasibility cones"): 6 float4 = 96 bytes per node
// instead of 4 float4 = 64 bytes.  RTC_NODE_CONES=0 builds the plain 64-byte nodes.
#ifndef RTC_NODE_CONES
#define RTC_NODE_CONES 1
#endif
#ifndef RTC_NODE_CENTRE_HALF
#define RTC_NODE_CENTRE_HALF 1
#endif

namespace rtc {

// The course's five homework snapshots of the renderer read five dialects of the scene format and
// render with five variants of Scene::RayTrace; hw5 is the hot path, hw1-hw4 are its callers' formats
// (DESIGN.md section 8, row f).  /root/reference/hwN/src/scene.cpp for each.
enum Dialect : int {
    DIALECT_HW1 = 1,  // ray casting: colour of the closest primitive, no tone mapping
    DIALECT_HW2 = 2,  // Whitted: ambient + point/directional lights with shadows, metallic, dielectric (Schlick blend)
    DIALECT_HW3 = 3,  // path tracing, uniform-hemisphere sampling (2 C L cos), EMISSION / SAMPLES
    DIALECT_HW4 = 4,  // path tracing with the cosine + light mix distribution (hw5 without triangles and BVH)
    DIALECT_HW5 = 5   // + TRIANGLE, SAH BVH
};

// hw2 light (src/lights.cpp): directional (dir) or point (pos, attenuation c0 + c1 d + c2 d^2)
struct PointLight {
    vec3 intensity{0, 0, 0}, pos{0, 0, 0}, att{0, 0, 0}, dir{0, 0, 0};
    int directed = 0;
};

// PRIMITIVE_TYPE / MATERIAL values follow include/primitives.h:13-18 and include/materials.h
enum PrimType : int { PT_PLANE = 1, PT_BOX = 2, PT_ELLIPSOID = 4, PT_TRIANGLE = 8 };
enum Material : int { MAT_DIFFUSE = 0, MAT_METALLIC = 1, MAT_DIELECTRIC = 2 };

// per-primitive flag bits stored next to the type on the device
enum PrimFlags : int {
    PF_TYPE_MASK = 0xF,
    PF_IDENT = 1 << 4,     // pos == 0 and rot == identity: world space == local space (dragon triangles)
    PF_ROT_IDENT = 1 << 5  // rot == identity (pos may be non-zero)
};

// what a scene contains, as far as the shading kernel's code size is concerned (rt_device.cuh prim_flags_for)
enum SceneFeature : unsigned {
    FE_ROTATION = 1,   // some primitive has a rotation other than identity
    FE_ELLIPSOID = 2,  // some primitive (light or not) is an ellipsoid
    FE_SPECULAR = 4,   // some primitive is METALLIC or DIELECTRIC
    FE_ALL = 7
};

struct Primitive {
    int type = 0;
    int material = MAT_DIFFUSE;
    int orig = -1;  // index in file order
    vec3 col{0, 0, 0}, emission{0, 0, 0}, pos{0, 0, 0};
    quat rot{0, 0, 0, 1};
    float ior = 0.f;
    vec3 d0{0, 0, 0}, d1{0, 0, 0}, d2{0, 0, 0};  // plane n | box s | ellipsoid r | triangle a,b,c
};

struct Aabb {
    vec3 mn, mx;
};

// BVH_t::nodes entry (include/bvh.h:30-36)
struct RefNode {
    Aabb box;
    uint32_t left, right, first, count;
};

struct Camera {
    vec3 pos{0, 0, 0}, right{0, 0, 0}, up{0, 0, 0}, forward{0, 0, 0};
    float fov_x = 0.f;
    unsigned width = 0, height = 0;
};

struct f4 {
    float x, y, z, w;
};
struct u4 {
    uint32_t x, y, z, w;
};

// Everything the device needs, as flat arrays (see DESIGN.md "Data layout in HBM").
struct FlatScene {
    // per primitive, final order
    std::vector<f4> geo0, geo1, geo2;  // triangle: (a,n.x) (b,n.y) (c,n.z); others: (d0,0) 0 0
    std::vector<f4> xf_pos;            // (pos.xyz, bits(type|flags))
    std::vector<f4> xf_rot;            // quaternion xyzw
    std::vector<f4> mat0, mat1;        // (col.rgb, bits(material)) (emission.rgb, ior)
    // index BVH, 4-wide, kIndexNodeF4 x f4 per node (96 bytes): child boxes as fp16 rounded OUTWARD, refs, child cones
    // (min.x[4] min.y[4] min.z[4] max.x[4] | max.y[4] max.z[4] refs[4]); exact leaf boxes: ubox
    std::vector<f4> inodes;
    uint32_t iroot = 0;  // child reference of the root (may be a leaf reference)
    // reference BVH: 2 x f4 per node (centre.xyz, bits(left)) (half.xyz, bits(right)) + meta
    std::vector<f4> rnodes;
    std::vector<u4> rmeta;  // (first, leaf ? count : cut, depth, 0)
    // LCA range-min table over cut positions: levels x nbvh entries of node ids
    std::vector<uint32_t> lca;
    uint32_t lca_levels = 0;
    std::vector<f4> ubox;              // 2 x f4 per primitive slot: (min,0) (max,0) of the reference leaf starting there
    std::vector<f4> planes;            // 2 x f4 per plane: (n, bits(prim id)) (pos, bits(no rotation))
    std::vector<int32_t> lights;
    std::vector<f4> plights;           // hw2: 4 x f4 per light: (intensity, bits(directed)) (pos,0) (attenuation,0) (normalised dir,0)
    uint32_t index_depth = 0, ref_depth = 0, units = 0;
    uint32_t features = 0;             // SceneFeature bits present in this scene
    // the extent the index BVH was built for: max(|camera position|inf, |unit box coordinates|inf); its child boxes are
    // widened by 2^-20 of it (bvh_build.cpp IndexBuilder::slack), so a camera farther out needs a rebuild
    double index_extent = 0;
};

struct HostScene {
    int dialect = DIALECT_HW5;
    Camera cam;
    vec3 background{0, 0, 0};
    vec3 ambient{0, 0, 0};                 // hw2 AMBIENT_LIGHT
    std::vector<PointLight> point_lights;  // hw2 NEW_LIGHT blocks
    unsigned ray_depth = 0, samples = 0;
    std::vector<Primitive> prims;  // final order after init()
    uint32_t nbvh = 0;             // non-plane primitives, stored first
    std::vector<RefNode> nodes;    // reference BVH, in creation (pre-)order
    uint32_t root = 0;
    std::vector<int32_t> lights;   // emissive boxes / ellipsoids
    FlatScene flat;
    // thin lens of the camera (rtc_scene_set_lens): aperture radius (0 = pinhole) and focus distance
    float lens_r = 0.f, lens_f = 1.f;

    // Scene::Load (hw5 src/sceneload.cpp:112-176; hwN src/scene.cpp Scene::Load for the other dialects):
    // only the words of `dialect` are commands, the rest is reported as unexpected and skipped
    void parse(const std::string& text);
    // Scene::InitScene (src/scene.cpp:7-40) + our index structures + flattening
    void init();
    // the units (reference leaves), their exact boxes and the index BVH over them, for cameras up to `cam_extent` (the
    // largest |position|inf): the stage of init() after the reference tree, and the whole rebuild when a camera is set
    // beyond flat.index_extent.  Reads prims and nodes in their final order; changes only units, ubox, inodes, iroot,
    // index_depth and index_extent.
    void build_index(double cam_extent);
};

// child reference encoding of the index BVH
constexpr uint32_t IREF_LEAF = 0x80000000u;
constexpr uint32_t IREF_NONE = 0xFFFFFFFFu;
// in a reference to an INNER node (bit 31 clear): none of the node's children has a direction cone, the visit skips
// the third 32-byte load (the upper levels of the tree: cones only bite in the lowest five)
constexpr uint32_t IREF_NOCONE = 0x40000000u;
constexpr uint32_t IREF_NODE_MASK = 0x00FFFFFFu;   // index of an inner node inside its reference
constexpr uint32_t IREF_FAST = 0x40000000u;     // leaf = one triangle with pos 0 and identity rotation
constexpr uint32_t IREF_MAX_LEAF_PRIMS = 64;   // 6 bits (24..29)
constexpr uint32_t IREF_MAX_PRIMS = 1u << 24;
// Children per index node: 4, or 8 = two 4-child blocks of the same layout fetched by ONE visit (the collapse
// predicts 35 % fewer entered nodes at 8: profiles/r01_experiments.md; prepared for an A/B run, 4 is the measured
// default).
#ifndef RTC_NODE_WIDTH
#define RTC_NODE_WIDTH 4
#endif
static_assert(RTC_NODE_WIDTH == 4 || RTC_NODE_WIDTH == 8, "index nodes hold 4 or 8 children");
constexpr uint32_t kNodeWidth = RTC_NODE_WIDTH;
constexpr uint32_t kIndexBlockF4 = RTC_NODE_CONES ? 6 : 4;                  // float4 per block of 4 children
constexpr uint32_t kIndexNodeF4 = kIndexBlockF4 * (kNodeWidth / 4);          // float4 per index node

Aabb aabb_of_primitive(const Primitive& p);  // AABB_t::AABB_t(const Primitive&) src/bvh.cpp:41-87

}  // namespace rtc
