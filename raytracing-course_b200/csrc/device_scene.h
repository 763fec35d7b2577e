// device_scene.h -- what a kernel sees of a scene: pointers into HBM plus a few scalars, passed
// BY VALUE as a kernel parameter (lives in the constant bank, no extra load to reach a pointer).
#pragma once
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>
#include <string.h>

#include "scene_host.h"

namespace rtc {

// Camera::GetToRay's inputs as the kernels read them (src/scene.cpp:180-187): position, axes, tan(fov_x / 2) and the
// tangent of the vertical half-angle, tan(fov_x / 2) * height / width
struct DevCamera {
    float3 pos, right, up, forward;
    float tan_fov_x, tan_fov_y;
};
// the one place a host camera becomes a DevCamera: the scene's own (fill_dev_scalars) and every view of a batched render
inline DevCamera dev_camera(const Camera& cam) {
    DevCamera C;
    C.pos = make_float3(cam.pos.x, cam.pos.y, cam.pos.z);
    C.right = make_float3(cam.right.x, cam.right.y, cam.right.z);
    C.up = make_float3(cam.up.x, cam.up.y, cam.up.z);
    C.forward = make_float3(cam.forward.x, cam.forward.y, cam.forward.z);
    // Camera::GetToRay, src/scene.cpp:181-182 (tan evaluated in double, as the reference's
    // unqualified tan() does; checked bit-exact against it in tests/)
    float tx = (float)tan((double)(cam.fov_x / 2));
    C.tan_fov_x = tx;
    C.tan_fov_y = tx * (float)cam.height / (float)cam.width;
    return C;
}

// The thin lens as the camera kernels read it (DESIGN.md "Thin lens"): aperture radius r and r / f.  It travels as a
// trailing kernel parameter of the kernels that make camera rays, not in DevScene: DevScene is the first parameter of
// every kernel, and a larger DevScene would move every parameter after it, in every kernel.
struct DevLens {
    float r, r_over_f;
};
inline DevLens dev_lens(const HostScene& host) { return DevLens{host.lens_r, host.lens_r / host.lens_f}; }

struct DevScene {
    // per primitive (final order), 16-byte aligned float4 arrays
    const float4* geo0;    // triangle (a, n.x) | other (d0, 0)
    const float4* geo1;    // triangle (b, n.y)
    const float4* geo2;    // triangle (c, n.z)
    const float4* xf_pos;  // (pos, bits(type | flags))
    const float4* xf_rot;  // quaternion xyzw
    const float4* mat0;    // (colour, bits(material))
    const float4* mat1;    // (emission, ior)
    // index BVH: 6 float4 (96 B) per 4-wide node: fp16 child boxes, child refs, fp16 child direction cones
    const float4* inodes;
    // reference BVH: 2 float4 per node + meta
    const float4* rnodes;
    const uint4* rmeta;
    const uint32_t* lca;
    const int32_t* lights;
    const float4* ubox;    // per primitive slot: exact (min) (max) of the reference leaf that starts there
    const float4* planes;  // per plane: (n.xyz, bits(prim id)) (pos.xyz, bits(1 = no rotation))
    const float4* plights; // hw2 dialect: 4 float4 per light (intensity, bits(directed)) (pos) (attenuation) (unit dir)

    uint32_t nprims, nbvh, nnodes, root, iroot, lca_levels, nlights, ref_depth;
    uint32_t iroot_ref[4];  // child references of the index root (k_traverse starts from the children pre_step entered)
    uint32_t width, height, ray_depth, nplanes;
    DevCamera cam;
    float3 bg;
    // homework dialect (scene_host.h Dialect) and the constants that differ between the snapshots
    uint32_t dialect, nplights;
    uint32_t features;  // SceneFeature bits (scene_host.h): which instantiation of k_shade covers the scene
    float eps;         // ray offset: 1e-3 in hw2/hw3 (include/scene.h:60), 1e-4 in hw4/hw5
    float plane_tmax;  // IntersectPlane drops t > 1e5 from hw4 on (hw4 src/primitives.cpp:47); earlier: no limit
    float3 ambient;    // hw2 AMBIENT_LIGHT
};

// Every scalar of DevScene from the host scene (the array pointers are the caller's: HBM slices in c_api.cu,
// host vectors in the test-only host emulation).
inline void fill_dev_scalars(const HostScene& host, DevScene& S) {
    S.nplanes = (uint32_t)(host.flat.planes.size() / 2);
    S.nprims = (uint32_t)host.prims.size(); S.nbvh = host.nbvh; S.nnodes = (uint32_t)host.nodes.size();
    S.root = host.root; S.iroot = host.flat.iroot; S.lca_levels = host.flat.lca_levels;
    for (int c = 0; c < 4; ++c) S.iroot_ref[c] = IREF_NONE;
    if (host.flat.iroot != IREF_NONE && !(host.flat.iroot & IREF_LEAF)) {
        const f4& refs = host.flat.inodes[kIndexNodeF4 * (size_t)(host.flat.iroot & IREF_NODE_MASK) + 3];   // words 12..15 of the node
        memcpy(S.iroot_ref, &refs, sizeof S.iroot_ref);
    }
    S.nlights = (uint32_t)host.lights.size(); S.ref_depth = host.flat.ref_depth;
    S.width = host.cam.width; S.height = host.cam.height; S.ray_depth = host.ray_depth;
    S.cam = dev_camera(host.cam);
    S.bg = make_float3(host.background.x, host.background.y, host.background.z);
    S.nplights = (uint32_t)host.point_lights.size();
    S.dialect = (uint32_t)host.dialect;
    S.features = host.flat.features;
    S.eps = host.dialect <= DIALECT_HW3 ? 1e-3f : 1e-4f;           // hwN include/scene.h `eps`
    S.plane_tmax = host.dialect <= DIALECT_HW3 ? 3.0e38f : 1e5f;   // hw4 src/primitives.cpp:47
    S.ambient = make_float3(host.ambient.x, host.ambient.y, host.ambient.z);
}

// Wavefront path state: three float4 per path and one word for the hit (52 bytes).  Radiance does not travel with
// the path: beta * emission is added to the pixel sum where it is found (k_shade).
struct PathSoA {
    float4* o;      // origin.xyz, bits(sample index)
    float4* d;      // direction.xyz, distance of the closest plane (1e18 = none): closest_dist handed to the BVH
    float4* beta;   // throughput.rgb, bits(pixel index)
};
struct HitSoA {
    uint32_t* id;   // 0xFFFFFFFF = miss, else id of the closest primitive (plane so far, k_traverse overwrites)
};

constexpr uint32_t HIT_MISS = 0xFFFFFFFFu;
constexpr uint32_t HIT_INTERIOR = 1u << 30;

}  // namespace rtc
