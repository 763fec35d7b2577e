// course_device.cuh -- per-pixel device functions of the two deterministic homework dialects (sm_100a):
//   hw1  ray casting: colour of the closest primitive              (hw1 src/scene.cpp:40-56, 167-179)
//   hw2  Whitted: ambient + point / directional lights with shadow rays, mirror reflection, dielectric
//        with the Schlick blend of BOTH branches                   (hw2 src/scene.cpp:262-341)
// Kept apart from the kernels (course_kernels.cu) so that the test-only host compilation (tests/host_emul)
// can run the same code against the reference's images without a GPU.
#pragma once
#include "rt_device.cuh"

namespace rtc {

RT_D SceneHit closest_hit(const DevScene& S, vec3 o, vec3 d) { return scene_intersect<0>(S, o, d, nullptr, nullptr, nullptr); }

// pixel-centre camera ray: Camera::get_to_ray(int x, int y), hw1 src/scene.cpp:30-38 / hw2 src/scene.cpp:229-237.
// `2 * (x + 0.5) / width - 1` and its product with the tangent are evaluated in double and rounded once.
RT_D void centre_ray(const DevScene& S, uint32_t pixel, vec3& o, vec3& d) {
    uint32_t x = pixel % S.width, y = pixel / S.width;
    float nx = (float)((2 * (x + 0.5) / (int)S.width - 1) * (double)S.cam.tan_fov_x);
    float ny = (float)(-1.f * (2 * (y + 0.5) / (int)S.height - 1) * (double)S.cam.tan_fov_y);
    o = mk3(S.cam.pos.x, S.cam.pos.y, S.cam.pos.z);
    d.x = __fadd_rn(__fadd_rn(__fmul_rn(nx, S.cam.right.x), __fmul_rn(ny, S.cam.up.x)), __fmul_rn(1.f, S.cam.forward.x));
    d.y = __fadd_rn(__fadd_rn(__fmul_rn(nx, S.cam.right.y), __fmul_rn(ny, S.cam.up.y)), __fmul_rn(1.f, S.cam.forward.y));
    d.z = __fadd_rn(__fadd_rn(__fmul_rn(nx, S.cam.right.z), __fmul_rn(ny, S.cam.up.z)), __fmul_rn(1.f, S.cam.forward.z));
}

// hw1 Scene::RayTrace: the colour of the closest primitive, the background otherwise (hw1 src/scene.cpp:167-179)
RT_D vec3 raycast_pixel_hw1(const DevScene& S, uint32_t pixel) {
    vec3 o, d;
    centre_ray(S, pixel, o, d);
    SceneHit h = closest_hit(S, o, d);
    vec3 c = mk3(S.bg.x, S.bg.y, S.bg.z);
    if (h.id >= 0) c = ld3(ldg4(S.mat0 + h.id));
    return c;
}

// DotLight::CalcLight / DirectedLight::CalcLight, hw2 src/lights.cpp:7-23
RT_D void calc_light(const DevScene& S, uint32_t l, vec3 p, vec3& colour, vec3& dir, float& dist) {
    float4 a = ldg4(S.plights + 4 * l);
    vec3 intensity = ld3(a);
    if (__float_as_uint(a.w)) {
        colour = intensity;
        dir = ld3(ldg4(S.plights + 4 * l + 3));
        dist = 1e18f;
        return;
    }
    vec3 to = ld3(ldg4(S.plights + 4 * l + 1)) - p;
    vec3 att = ld3(ldg4(S.plights + 4 * l + 2));
    dist = length(to);
    float k = (float)(1. / (double)(att.x + att.y * dist + att.z * dist * dist));  // `1. / float`: a double division
    colour = k * intensity;
    dir = normalize(to);
}

// Scene::RayTrace of hw2 with the recursion turned into a stack of (ray, weight, remaining depth):
// L = sum over the leaves of the reflection / refraction tree of weight * local colour.
constexpr int kWhittedStack = 34;  // depth-first: at most ray_depth + 1 entries are pending
struct Pending {
    vec3 o, d, w;
    uint32_t depth;
};
RT_D vec3 whitted_pixel_hw2(const DevScene& S, uint32_t pixel) {
    Pending st[kWhittedStack];
    int sp = 0;
    vec3 L = mk3(0, 0, 0);
    centre_ray(S, pixel, st[0].o, st[0].d);
    st[0].w = mk3(1, 1, 1);
    st[0].depth = S.ray_depth;
    sp = 1;
    while (sp > 0) {
        Pending r = st[--sp];
        if (r.depth == 0) continue;  // hw2 src/scene.cpp:263-265
        if (sp + 2 > kWhittedStack) continue;  // unreachable while RAY_DEPTH <= 32 (enforced at load and override): never write past st[]
        SceneHit h = closest_hit(S, r.o, r.d);
        if (h.id < 0) { L = L + r.w * mk3(S.bg.x, S.bg.y, S.bg.z); continue; }
        vec3 p = r.o + h.t * r.d;
        vec3 nd = normalize(r.d);
        float4 m0 = ldg4(S.mat0 + h.id);
        vec3 col = ld3(m0);
        uint32_t material = __float_as_uint(m0.w);
        vec3 rdir = reflect_dir(h.n, nd);
        if (material == MAT_DIFFUSE) {
            vec3 sum = mk3(S.ambient.x, S.ambient.y, S.ambient.z);
            for (uint32_t l = 0; l < S.nplights; ++l) {
                vec3 lc, ldir;
                float dist;
                calc_light(S, l, p, lc, ldir, dist);
                float k = dot(ldir, h.n);
                if (k >= 0.f) {  // the light is not behind the surface
                    SceneHit b = closest_hit(S, p + S.eps * ldir, ldir);
                    if (!(b.id >= 0 && b.t <= dist)) sum = sum + k * lc;
                }
            }
            L = L + r.w * (sum * col);
        } else if (material == MAT_METALLIC) {
            st[sp++] = Pending{p + S.eps * rdir, rdir, r.w * col, r.depth - 1};
        } else {  // DIELECTRIC, hw2 src/scene.cpp:300-330
            float eta1 = 1.f, eta2 = ldg4(S.mat1 + h.id).w;
            if (h.interior) { float tmp = eta1; eta1 = eta2; eta2 = tmp; }
            vec3 dir = -nd;
            float dn = dot(h.n, dir);
            // unqualified sqrt / pow on floats are the double versions (hw2 src/scene.cpp:310-329)
            float sin2 = (float)((double)(eta1 / eta2) * sqrt((double)(1.f - dn * dn)));
            if (fabsf(sin2) > 1.f) {  // total internal reflection
                st[sp++] = Pending{p + S.eps * rdir, rdir, r.w, r.depth - 1};
                continue;
            }
            float cos2 = (float)sqrt((double)(1.f - sin2 * sin2));
            float e = eta1 / eta2;
            vec3 fr = e * (-dir) + (e * dn - cos2) * h.n;
            double q0 = (double)((eta1 - eta2) / (eta1 + eta2));
            float r0 = (float)(q0 * q0);
            double m = (double)(1.f - dn), m2 = m * m;
            float refl = (float)((double)r0 + (double)(1.f - r0) * (m2 * m2 * m));
            vec3 wt = (1.f - refl) * r.w;
            if (!h.interior) wt = wt * col;
            st[sp++] = Pending{p + S.eps * fr, fr, wt, r.depth - 1};
            st[sp++] = Pending{p + S.eps * rdir, rdir, refl * r.w, r.depth - 1};
        }
    }
    return L;
}

// hw1 writes the colour as it is: Color::toUInts, hw1 src/color.cpp:10-16 (no tone mapping, no gamma)
RT_D unsigned char flat_u8(float mean) { return (unsigned char)(int)roundf(__fmul_rn(255.f, mean)); }

}  // namespace rtc
