// rt_device.cuh -- device functions of the hw5 hot path for sm_100a: primitive intersection,
// the two BVH traversals, the light/cosine mix distribution and the Philox streams.
// Reference lines are cited per function (paths under /root/reference/hw5).
#pragma once
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <math_constants.h>
#include <stdint.h>

#include "device_scene.h"
#include "scene_host.h"  // PrimType / Material / flag and IREF_* constants (plain enums)
#include "vecmath.h"

namespace rtc {

#define RT_D __device__ __forceinline__
#ifdef __CUDACC__
#define RT_D_COLD static __device__ __noinline__   // rarely taken paths: one out-of-line copy per kernel
#else
#define RT_D_COLD static inline                    // host compilation of this header (tests/host_emul)
#endif

constexpr float kInfF = 1e18f;      // include/bvh.h:9
constexpr float kPi = 3.14159274101257324f;  // (float)acos(-1), include/distributions.h:14
constexpr int kRejectCap = 64;      // light sampling retries (the reference retries forever)
constexpr int kMaxRecords = 24;     // leaf hits kept per ray before falling back to the reference tree walk
constexpr int kIndexStack = 64;
constexpr int kRefStack = 96;

RT_D vec3 ld3(const float4& v) { return mk3(v.x, v.y, v.z); }
RT_D float4 ldg4(const float4* p) { return __ldg(p); }

// ------------------------------------------------------------------------------- Philox4x32-10
// Counter-based streams (DESIGN.md "RNG streams"): key = (seed, 0x52544300),
// counter = (pixel, sample, slot, block).  slot 0 = camera jitter, slot b >= 1 = the b-th hit.
RT_D uint4 philox4x32_10(uint4 c, uint2 k) {
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        uint32_t hi0 = __umulhi(0xD2511F53u, c.x), lo0 = 0xD2511F53u * c.x;
        uint32_t hi1 = __umulhi(0xCD9E8D57u, c.z), lo1 = 0xCD9E8D57u * c.z;
        c = make_uint4(hi1 ^ c.y ^ k.x, lo1, hi0 ^ c.w ^ k.y, lo0);
        k.x += 0x9E3779B9u;
        k.y += 0xBB67AE85u;
    }
    return c;
}
struct Rng {
    uint32_t seed, pixel, sample, slot;
    RT_D uint4 block(uint32_t b) const {
        return philox4x32_10(make_uint4(pixel, sample, slot, b), make_uint2(seed, 0x52544300u));
    }
};
RT_D float u01(uint32_t x) { return (float)(x >> 8) * (1.0f / 16777216.0f); }
RT_D void box_muller(uint32_t x0, uint32_t x1, float& z0, float& z1) {
    float a = (float)((x0 >> 8) + 1u) * (1.0f / 16777216.0f);
    float r = sqrtf(-2.0f * __logf(a));
    // theta in [0, 2pi): evaluate at theta - pi in [-pi, pi), where the fast sin/cos are accurate
    float th = 6.283185307179586f * u01(x1) - 3.14159265358979f;
    float s, c;
    __sincosf(th, &s, &c);
    z0 = -r * c;
    z1 = -r * s;
}
// Distribution::SampleNormal01Vec, src/distributions.cpp:102-110
RT_D vec3 normal_vec(uint4 b) {
    float z0, z1, z2, z3;
    box_muller(b.x, b.y, z0, z1);
    box_muller(b.z, b.w, z2, z3);
    float k = rsqrtf(z0 * z0 + z1 * z1 + z2 * z2);  // a random direction: 2 ulp of rsqrt are immaterial
    return mk3(z0 * k, z1 * k, z2 * k);
}

// ------------------------------------------------------------------------------- primitives
// Two arithmetic flavours.  EXACT (default) keeps IEEE division / sqrt wherever a result decides a
// hit or becomes the reported distance or normal (traversal, final hit, rtc_intersect).  FAST
// (approximate reciprocal / rsqrt, <= 2 ulp) is used only inside the shading estimators
// (light pdf, validity test of a light sample), whose inputs are random anyway.
template <bool FAST> RT_D float rt_div(float a, float b) { return FAST ? __fdividef(a, b) : a / b; }
template <bool FAST> RT_D vec3 rt_div(vec3 a, vec3 b) { return mk3(rt_div<FAST>(a.x, b.x), rt_div<FAST>(a.y, b.y), rt_div<FAST>(a.z, b.z)); }
template <bool FAST> RT_D vec3 rt_normalize(vec3 a) {
    if (!FAST) return normalize(a);
    float k = rsqrtf(dot(a, a));
    return mk3(a.x * k, a.y * k, a.z * k);
}
struct Isect {
    float t;
    vec3 n;
    int interior;
};

// Primitive::IntersectPlane, src/primitives.cpp:55-66
RT_D bool isect_plane(vec3 o, vec3 d, vec3 n, float tmax, Isect& out) {
    float dn = dot(d, n);
    float t = -dot(o, n) / dn;
    if (t > tmax) return false;
    if (t > 0.f) {
        out.t = t;
        out.interior = dn >= 0.f;
        out.n = out.interior ? -n : n;
        return true;
    }
    return false;
}
// Primitive::IntersectBox, src/primitives.cpp:70-117
template <bool FAST = false>
RT_D bool isect_box(vec3 o, vec3 d, vec3 s, Isect& out) {
    vec3 a, b;
    if (FAST) {
        vec3 inv = mk3(__fdividef(1.f, d.x), __fdividef(1.f, d.y), __fdividef(1.f, d.z));
        a = (-s - o) * inv;
        b = (s - o) * inv;
    } else {
        a = (-s - o) / d;
        b = (s - o) / d;
    }
    float t1 = fmaxf(fmaxf(fminf(a.x, b.x), fminf(a.y, b.y)), fminf(a.z, b.z));
    float t2 = fminf(fminf(fmaxf(a.x, b.x), fmaxf(a.y, b.y)), fmaxf(a.z, b.z));
    if (t1 > t2 || t2 < 0.f) return false;
    bool interior = t1 < 0.f;
    float t = interior ? t2 : t1;
    vec3 p = o + t * d;
    vec3 nrm = rt_div<FAST>(p, s);
    if (interior) nrm = -nrm;
    float mx = fmaxf(fmaxf(fabsf(nrm.x), fabsf(nrm.y)), fabsf(nrm.z));
    if (fabsf(nrm.x) != mx) nrm.x = 0.f;
    if (fabsf(nrm.y) != mx) nrm.y = 0.f;
    if (fabsf(nrm.z) != mx) nrm.z = 0.f;
    out.t = t;
    out.n = rt_normalize<FAST>(nrm);
    out.interior = interior;
    return true;
}
// Primitive::IntersectEllipsoid, src/primitives.cpp:120-152.  The reference evaluates the two
// roots in double (unqualified sqrt(float) resolves to ::sqrt(double)) and rounds once; so do we.
RT_D bool isect_ellipsoid(vec3 o, vec3 d, vec3 r, Isect& out) {
    vec3 dr = d / r, orr = o / r;
    float a = __fadd_rn(__fadd_rn(__fmul_rn(dr.x, dr.x), __fmul_rn(dr.y, dr.y)), __fmul_rn(dr.z, dr.z));
    float b = __fmul_rn(2.f, __fadd_rn(__fadd_rn(__fmul_rn(orr.x, dr.x), __fmul_rn(orr.y, dr.y)), __fmul_rn(orr.z, dr.z)));
    float c = __fadd_rn(__fadd_rn(__fadd_rn(__fmul_rn(orr.x, orr.x), __fmul_rn(orr.y, orr.y)), __fmul_rn(orr.z, orr.z)), -1.f);
    float disc = __fadd_rn(__fmul_rn(b, b), -__fmul_rn(__fmul_rn(4.f, a), c));
    if (disc <= 0.f) return false;
    double sq = sqrt((double)disc), den = (double)__fmul_rn(2.f, a);
    float x1 = (float)(((double)(-b) - sq) / den);
    float x2 = (float)(((double)(-b) + sq) / den);
    if (x1 > x2) { float tmp = x1; x1 = x2; x2 = tmp; }
    if (x2 < 0.f) return false;
    bool interior = x1 < 0.f;
    float t = interior ? x2 : x1;
    vec3 p = o + t * d;
    vec3 nrm = normalize(p / (r * r));
    if (interior) nrm = -nrm;
    out.t = t;
    out.n = nrm;
    out.interior = interior;
    return true;
}
// Primitive::IntersectTriangle, src/primitives.cpp:155-174.  Faithful to the reference: the
// plane is the one through the LOCAL ORIGIN with the triangle's normal (IntersectPlane(ray, n)),
// and the three orientation tests then act on that point.
RT_D bool isect_triangle(vec3 o, vec3 d, vec3 a, vec3 b, vec3 c, vec3 n, float& t_out, bool& interior) {
    float dn = dot(d, n);
    float t = -dot(o, n) / dn;
    if (!(t > 0.f) || t > 1e5f) return false;
    vec3 p = o + t * d;
    vec3 pa = p - a;
    if (!(dot(cross(b - a, pa), n) > 0.f)) return false;
    if (!(dot(cross(pa, c - a), n) > 0.f)) return false;
    if (!(dot(cross(c - b, p - b), n) > 0.f)) return false;
    t_out = t;
    interior = dn >= 0.f;
    return true;
}

// glm's quaternion * vector (vecmath.h rotate) without FMA contraction: rotated primitives then see
// bit-identical local rays to the reference's, which matters for grazing ellipsoid hits (the
// discriminant b^2 - 4ac cancels, so ulps in the rotated ray become 1e-3 in t).
RT_D vec3 cross_exact(vec3 a, vec3 b) {
    return mk3(__fsub_rn(__fmul_rn(a.y, b.z), __fmul_rn(b.y, a.z)), __fsub_rn(__fmul_rn(a.z, b.x), __fmul_rn(b.z, a.x)),
               __fsub_rn(__fmul_rn(a.x, b.y), __fmul_rn(b.x, a.y)));
}
RT_D vec3 rotate_exact(quat q, vec3 v) {
    vec3 qv = mk3(q.x, q.y, q.z);
    vec3 uv = cross_exact(qv, v);
    vec3 uuv = cross_exact(qv, uv);
    vec3 s = mk3(__fadd_rn(__fmul_rn(uv.x, q.w), uuv.x), __fadd_rn(__fmul_rn(uv.y, q.w), uuv.y), __fadd_rn(__fmul_rn(uv.z, q.w), uuv.z));
    return mk3(__fadd_rn(v.x, __fmul_rn(s.x, 2.0f)), __fadd_rn(v.y, __fmul_rn(s.y, 2.0f)), __fadd_rn(v.z, __fmul_rn(s.z, 2.0f)));
}
// Ray into the primitive's local frame: rotate(conjugate(rotator), ray + -1*pos), src/primitives.cpp:15
RT_D void to_local(const DevScene& S, uint32_t prim, uint32_t flags, vec3& o, vec3& d) {
    if (flags & PF_IDENT) return;
    vec3 pos = ld3(ldg4(S.xf_pos + prim));
    o = o - pos;
    if (flags & PF_ROT_IDENT) return;
    float4 q4 = ldg4(S.xf_rot + prim);
    quat qc;
    qc.x = -q4.x; qc.y = -q4.y; qc.z = -q4.z; qc.w = q4.w;
    o = rotate_exact(qc, o);
    d = rotate_exact(qc, d);
}
RT_D uint32_t prim_flags(const DevScene& S, uint32_t prim) { return __float_as_uint(__ldg(&S.xf_pos[prim].w)); }

// Scene features (scene_host.h SceneFeature, DevScene::features): k_shade is instruction-cache bound, so it is
// compiled once per feature set and the host picks the smallest instantiation that covers the scene.  A kernel
// built WITHOUT a feature is only ever launched on scenes that do not have it; what it computes for the
// primitives that remain is the same arithmetic as the full version (the rotation code is already skipped per
// primitive through PF_ROT_IDENT, the type switches lose a case).
template <uint32_t FEAT>
RT_D uint32_t prim_flags_for(const DevScene& S, uint32_t prim) {
    uint32_t flags = prim_flags(S, prim);
    if (!(FEAT & FE_ROTATION)) flags |= PF_ROT_IDENT;
    return flags;
}

// distance-only test used during traversal (normal is recomputed once for the winner)
template <bool FAST = false>
RT_D bool prim_hit_t(const DevScene& S, uint32_t prim, vec3 o, vec3 d, float& t) {
    uint32_t flags = prim_flags(S, prim);
    to_local(S, prim, flags, o, d);
    float4 g0 = ldg4(S.geo0 + prim);
    if ((flags & PF_TYPE_MASK) == PT_TRIANGLE) {
        float4 g1 = ldg4(S.geo1 + prim), g2 = ldg4(S.geo2 + prim);
        bool interior;
        return isect_triangle(o, d, ld3(g0), ld3(g1), ld3(g2), mk3(g0.w, g1.w, g2.w), t, interior);
    }
    Isect is;
    bool ok;
    switch (flags & PF_TYPE_MASK) {
        case PT_BOX: ok = isect_box<FAST>(o, d, ld3(g0), is); break;
        case PT_ELLIPSOID: ok = isect_ellipsoid(o, d, ld3(g0), is); break;
        default: ok = isect_plane(o, d, ld3(g0), S.plane_tmax, is); break;
    }
    t = is.t;
    return ok;
}
// Primitive::Intersect, src/primitives.cpp:14-52 (normal back to world space, re-normalised), on rows the caller has
// already fetched: xp = xf_pos[prim] (position, type | flags), g0..g2 = geo0..2[prim].  k_shade issues those loads (and
// the material rows) together as soon as it knows the primitive, instead of flags -> position -> geometry one after
// the other (16 % of its stall samples sat on that chain).
template <bool FAST = false, uint32_t FEAT = FE_ALL, bool FAST_NORMAL = FAST>
RT_D bool prim_intersect_rows(const DevScene& S, uint32_t prim, float4 xp, float4 g0, float4 g1, float4 g2, vec3 o, vec3 d, Isect& out) {
    uint32_t flags = __float_as_uint(xp.w);
    if (!(FEAT & FE_ROTATION)) flags |= PF_ROT_IDENT;
    if (!(flags & PF_IDENT)) {  // to_local
        o = o - ld3(xp);
        if (!(flags & PF_ROT_IDENT)) {
            float4 q4 = ldg4(S.xf_rot + prim);
            quat qc;
            qc.x = -q4.x; qc.y = -q4.y; qc.z = -q4.z; qc.w = q4.w;
            o = rotate_exact(qc, o);
            d = rotate_exact(qc, d);
        }
    }
    bool ok;
    const uint32_t type = flags & PF_TYPE_MASK;
    if (type == PT_TRIANGLE) {
        vec3 n = mk3(g0.w, g1.w, g2.w);
        bool interior;
        ok = isect_triangle(o, d, ld3(g0), ld3(g1), ld3(g2), n, out.t, interior);
        out.interior = interior;
        out.n = interior ? -n : n;
    } else if (type == PT_BOX) {
        ok = isect_box<FAST>(o, d, ld3(g0), out);
    } else if ((FEAT & FE_ELLIPSOID) && type == PT_ELLIPSOID) {
        ok = isect_ellipsoid(o, d, ld3(g0), out);
    } else {
        ok = isect_plane(o, d, ld3(g0), S.plane_tmax, out);
    }
    if (!ok) return false;
    if (!(flags & PF_ROT_IDENT)) {
        float4 q4 = ldg4(S.xf_rot + prim);
        quat q;
        q.x = q4.x; q.y = q4.y; q.z = q4.z; q.w = q4.w;
        out.n = rotate_exact(q, out.n);
    }
    out.n = rt_normalize<FAST_NORMAL>(out.n);
    return true;
}
template <bool FAST = false, uint32_t FEAT = FE_ALL, bool FAST_NORMAL = FAST>
RT_D bool prim_intersect(const DevScene& S, uint32_t prim, vec3 o, vec3 d, Isect& out) {
    const float4 xp = ldg4(S.xf_pos + prim), g0 = ldg4(S.geo0 + prim);
    float4 g1 = make_float4(0.f, 0.f, 0.f, 0.f), g2 = g1;
    if ((__float_as_uint(xp.w) & PF_TYPE_MASK) == PT_TRIANGLE) { g1 = ldg4(S.geo1 + prim); g2 = ldg4(S.geo2 + prim); }
    return prim_intersect_rows<FAST, FEAT, FAST_NORMAL>(S, prim, xp, g0, g1, g2, o, d, out);
}

// ------------------------------------------------------------------------------- boxes
// AABB_t::Intersect = IntersectBox(ray - centre, half), src/bvh.cpp:89-93, with IEEE division:
// used where the reference's own nodes decide (reference-tree walk, LCA culling).
RT_D bool ref_box(const DevScene& S, uint32_t node, vec3 o, vec3 d, float& t_enter, bool& interior, uint32_t& left, uint32_t& right) {
    float4 A = ldg4(S.rnodes + 2 * node), B = ldg4(S.rnodes + 2 * node + 1);
    left = __float_as_uint(A.w);
    right = __float_as_uint(B.w);
    vec3 oc = o - ld3(A), s = ld3(B);
    vec3 a = (-s - oc) / d, b = (s - oc) / d;
    float t1 = fmaxf(fmaxf(fminf(a.x, b.x), fminf(a.y, b.y)), fminf(a.z, b.z));
    float t2 = fminf(fminf(fmaxf(a.x, b.x), fmaxf(a.y, b.y)), fmaxf(a.z, b.z));
    if (t1 > t2 || t2 < 0.f) return false;
    interior = t1 < 0.f;
    t_enter = interior ? t2 : t1;
    return true;
}

struct BestHit {
    float t;
    int id;
};

// ------------------------------------------------------------------------------- reference-tree walk
// BVH_t::Intersect_ (src/bvh.cpp:185-225) made iterative.  The recursion passes to the right
// child the distance found in the LEFT sibling subtree (or its own closest_dist when that
// subtree had no hit); a frame keeps that fallback plus the best hit seen before the frame was
// opened, `cur` is the best hit since.
RT_D BestHit trace_reftree(const DevScene& S, vec3 o, vec3 d, float cd0) {
    struct Frame { uint32_t node; float cdf; float st; int sid; };
    Frame stack[kRefStack];
    int sp = 0;
    BestHit cur{kInfF, -1};
    if (S.nbvh == 0) return cur;
    uint32_t v = S.root;
    float cd = cd0;
    for (;;) {
        float te; bool interior; uint32_t l, r;
        bool descend = false;
        if (ref_box(S, v, o, d, te, interior, l, r) && !(cd < te && !interior)) {
            if (l == 0xFFFFFFFFu) {
                uint4 m = __ldg(S.rmeta + v);
                for (uint32_t i = m.x; i < m.x + m.y; ++i) {
                    float t;
                    if (prim_hit_t(S, i, o, d, t) && t < cur.t) { cur.t = t; cur.id = (int)i; }
                }
            } else if (sp < kRefStack) {
                stack[sp].node = r; stack[sp].cdf = cd; stack[sp].st = cur.t; stack[sp].sid = cur.id;
                ++sp;
                cur.t = kInfF; cur.id = -1;
                v = l;
                descend = true;
            }
        }
        if (descend) continue;
        if (sp == 0) break;
        --sp;
        Frame f = stack[sp];
        cd = (cur.id != -1) ? cur.t : f.cdf;
        if (!(cur.t < f.st)) { cur.t = f.st; cur.id = f.sid; }
        v = f.node;
    }
    return cur;
}

// ------------------------------------------------------------------------------- index traversal
// Lowest common ancestor in the reference tree of the leaves starting at primitive a < b:
// the shallowest inner node whose cut position lies in (a, b].
RT_D uint32_t ref_lca(const DevScene& S, uint32_t a, uint32_t b) {
    uint32_t lo = a + 1, len = b - a;
    uint32_t l = 31 - __clz(len);
    uint32_t n1 = __ldg(S.lca + (size_t)l * S.nbvh + lo);
    uint32_t n2 = __ldg(S.lca + (size_t)l * S.nbvh + (b + 1 - (1u << l)));
    if (n1 == 0xFFFFFFFFu) return n2;
    if (n2 == 0xFFFFFFFFu || n1 == n2) return n1;
    uint32_t d1 = __ldg(&S.rmeta[n1].z), d2 = __ldg(&S.rmeta[n2].z);
    return d2 < d1 ? n2 : n1;
}

struct LeafRec {
    uint32_t key;  // first primitive of the reference leaf (its position in DFS order)
    int id;        // closest primitive inside the leaf
    float t;       // its distance
    float tcull;   // leaf box entry distance, -inf when the origin is inside the box
};

// Replays BVH_t::Intersect_ on the k leaves (sorted by key) that actually produced a hit.
// Leaves without a hit, and subtrees without such leaves, return id = -1 in the reference and
// influence nothing; along a chain of single-child steps closest_dist does not change and the
// boxes shrink, so testing the skip rule at the bottom of each chain (a branching node = an LCA,
// or the leaf) is equivalent to testing it at every node of the chain.
RT_D BestHit replay_reference(const DevScene& S, vec3 o, vec3 d, float cd0, LeafRec* rec, int k) {
    BestHit cur{kInfF, -1};
    if (k == 0) return cur;
    if (k == 1) {
        if (!(cd0 < rec[0].tcull)) { cur.t = rec[0].t; cur.id = rec[0].id; }
        return cur;
    }
    for (int i = 1; i < k; ++i) {  // insertion sort by key
        LeafRec x = rec[i];
        int j = i - 1;
        while (j >= 0 && rec[j].key > x.key) { rec[j + 1] = rec[j]; --j; }
        rec[j + 1] = x;
    }
    struct Frame { int m, j; float cdf; float st; int sid; };
    Frame stack[kMaxRecords];
    int sp = 0, i = 0, j = k;
    float cd = cd0;
    for (;;) {
        bool descend = false;
        if (j - i == 1) {
            if (!(cd < rec[i].tcull) && rec[i].t < cur.t) { cur.t = rec[i].t; cur.id = rec[i].id; }
        } else {
            uint32_t u = ref_lca(S, rec[i].key, rec[j - 1].key);
            float te; bool interior; uint32_t l, r;
            if (ref_box(S, u, o, d, te, interior, l, r) && !(cd < te && !interior)) {
                uint32_t cut = __ldg(&S.rmeta[u].y);
                int m = i + 1;
                while (rec[m].key < cut) ++m;
                stack[sp].m = m; stack[sp].j = j; stack[sp].cdf = cd; stack[sp].st = cur.t; stack[sp].sid = cur.id;
                ++sp;
                cur.t = kInfF; cur.id = -1;
                j = m;
                descend = true;
            }
        }
        if (descend) continue;
        if (sp == 0) break;
        --sp;
        Frame f = stack[sp];
        cd = (cur.id != -1) ? cur.t : f.cdf;
        if (!(cur.t < f.st)) { cur.t = f.st; cur.id = f.sid; }
        i = f.m; j = f.j;
    }
    return cur;
}

// One index-BVH node = 96 bytes: the boxes of its 4 children as fp16 rounded OUTWARD (64 bytes with the refs) + one
// direction cone per child (32 bytes, cone_cull_pair below)
// (min.x[4] min.y[4] min.z[4] max.x[4] | max.y[4] max.z[4] refs[4]), read with two 32-byte loads.
// The traversal is bound by the L1 misses an SM can keep in flight (profiles/r01_experiments.md),
// so node bytes are what counts; conservative boxes only add candidates, and every leaf is
// re-tested against its EXACT float box before its primitives are (leaf_test).
// Slab tests in min/max form with the reciprocal direction.  tc = box entry distance, or -inf when
// the origin is inside (the reference's `interior`).
// Reciprocal direction for the slab tests, clamped to +-1e30: a zero direction component would give
// inf and then inf - inf = NaN in c * inv - o * inv, which the 3-input min/max drop, i.e. the axis would
// not constrain at all and such a ray (about one in 10^7) would walk a whole slab of the tree and hold
// a persistent k_traverse launch for milliseconds.  With a finite reciprocal the test is simply exact.
#ifndef RTC_FAST_RAY_INV
#define RTC_FAST_RAY_INV 1   // measured on B200: k_traverse 11.70 -> 11.56 ms, k_shade 7.14 -> 7.07 ms
#endif
RT_D vec3 ray_inv(vec3 d) {
    const float big = 1e30f;
#if RTC_FAST_RAY_INV && defined(__CUDA_ARCH__)
    // approximate reciprocal (MUFU.RCP, 1 ulp): the slab tests of the index nodes are conservative by more than that
    // and leaf_box re-decides everything inside its 2e-6 band exactly
    return mk3(fminf(fmaxf(__fdividef(1.0f, d.x), -big), big), fminf(fmaxf(__fdividef(1.0f, d.y), -big), big), fminf(fmaxf(__fdividef(1.0f, d.z), -big), big));
#else
    return mk3(fminf(fmaxf(1.0f / d.x, -big), big), fminf(fmaxf(1.0f / d.y, -big), big), fminf(fmaxf(1.0f / d.z, -big), big));
#endif
}
struct NodeVisit {
    uint32_t ref[kNodeWidth];
    bool hit[kNodeWidth];
};
RT_D void slab(float mnx, float mny, float mnz, float mxx, float mxy, float mxz, vec3 inv, vec3 oi, uint32_t ref, bool& hit, float& tc) {
    float x1 = fmaf(mnx, inv.x, -oi.x), x2 = fmaf(mxx, inv.x, -oi.x);
    float y1 = fmaf(mny, inv.y, -oi.y), y2 = fmaf(mxy, inv.y, -oi.y);
    float z1 = fmaf(mnz, inv.z, -oi.z), z2 = fmaf(mxz, inv.z, -oi.z);
    float t1 = fmaxf(fmaxf(fminf(x1, x2), fminf(y1, y2)), fminf(z1, z2));
    float t2 = fminf(fminf(fmaxf(x1, x2), fmaxf(y1, y2)), fmaxf(z1, z2));
    hit = t1 <= t2 && t2 >= 0.f && ref != IREF_NONE;
    tc = t1 < 0.f ? -kInfF : t1;
}
// 32-byte read-only load (LDG.E.256 on sm_100a)
RT_D void ldg8(const float4* p, float4& a, float4& b) {
#ifdef __CUDA_ARCH__
    asm volatile("ld.global.nc.v8.f32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                 : "=f"(a.x), "=f"(a.y), "=f"(a.z), "=f"(a.w), "=f"(b.x), "=f"(b.y), "=f"(b.z), "=f"(b.w)
                 : "l"(p));
#else
    a = p[0];
    b = p[1];
#endif
}
RT_D float2 unpack_half2(float word) {
    uint32_t u = __float_as_uint(word);
    return __half22float2(*reinterpret_cast<const __half2*>(&u));
}
#if RTC_NODE_CENTRE_HALF
// child box = centre +- half: entry/exit per axis are tc -+ h * |inv| with tc = c * inv - o * inv, three
// FFMA and no min/max (the kernel is bound by the ALU pipe, which FMNMX shares with the integer
// bookkeeping).  Against the exact leaf test (slab) the two roundings can move entry/exit by a few ulp of
// t; fp16 rounding of c and h (outward) is three orders of magnitude larger except for boxes whose faces
// are exactly representable in fp16, where a ray within ~1e-6 of grazing a face may be decided the other way.
RT_D void slab_ch(float cx, float cy, float cz, float hx, float hy, float hz, vec3 inv, vec3 oi, uint32_t ref, bool& hit) {
    float tx = fmaf(cx, inv.x, -oi.x), ty = fmaf(cy, inv.y, -oi.y), tz = fmaf(cz, inv.z, -oi.z);
    float ax = fabsf(inv.x), ay = fabsf(inv.y), az = fabsf(inv.z);
    float t1 = fmaxf(fmaxf(fmaf(-hx, ax, tx), fmaf(-hy, ay, ty)), fmaf(-hz, az, tz));
    float t2 = fminf(fminf(fmaf(hx, ax, tx), fmaf(hy, ay, ty)), fmaf(hz, az, tz));
    hit = t1 <= t2 && t2 >= 0.f && ref != IREF_NONE;
}
#endif
// Feasibility cones (bvh_build.cpp Cone): the normalised ray direction as halves, (x, y) and (z, z).
struct ConeDir {
    uint32_t xy, zz;
};
RT_D uint32_t pack_half2(float a, float b) {
    __half2 h = __floats2half2_rn(a, b);
    return *reinterpret_cast<const uint32_t*>(&h);
}
RT_D ConeDir cone_dir(vec3 d) {
    // scale by the largest component first: |d|^2 must neither overflow nor vanish
    float m = fmaxf(fmaxf(fabsf(d.x), fabsf(d.y)), fabsf(d.z));
    vec3 e = d * __fdividef(1.f, m);
    float k = rsqrtf(dot(e, e));  // the result is rounded to 11 bits
    ConeDir c;
    c.xy = pack_half2(e.x * k, e.y * k);
    c.zz = pack_half2(e.z * k, e.z * k);
    return c;  // a zero or non-finite direction gives NaN halves: every comparison below is then false = not culled
}
// children (2j, 2j + 1) of a node: bit 0 / bit 16 set when the child cannot be hit by a ray of this direction,
// |dn . axis| < threshold in half arithmetic (the thresholds carry the rounding slack, bvh_build.cpp emit)
RT_D uint32_t cone_cull_pair(ConeDir dn, float wx, float wy, float wz, float wt) {
#ifdef __CUDA_ARCH__
    const __half2 xy = *reinterpret_cast<const __half2*>(&dn.xy), zz = *reinterpret_cast<const __half2*>(&dn.zz);
    const uint32_t ux = __float_as_uint(wx), uy = __float_as_uint(wy), uz = __float_as_uint(wz), ut = __float_as_uint(wt);
    const __half2 ax = *reinterpret_cast<const __half2*>(&ux), ay = *reinterpret_cast<const __half2*>(&uy);
    const __half2 az = *reinterpret_cast<const __half2*>(&uz), th = *reinterpret_cast<const __half2*>(&ut);
    __half2 dt = __hmul2(ax, __low2half2(xy));
    dt = __hfma2(ay, __high2half2(xy), dt);
    dt = __hfma2(az, zz, dt);
    return __hlt2_mask(__habs2(dt), th) & 0x00010001u;
#else
    // host compilation (tests/host_emul): the same operations, each rounded to half
    auto h = [](float f) { return __half2float(__float2half_rn(f)); };
    const float2 d_xy = unpack_half2(__uint_as_float(dn.xy)), d_zz = unpack_half2(__uint_as_float(dn.zz));
    const float2 ax = unpack_half2(wx), ay = unpack_half2(wy), az = unpack_half2(wz), th = unpack_half2(wt);
    float d0 = h(ax.x * d_xy.x), d1 = h(ax.y * d_xy.x);
    d0 = h(fmaf(ay.x, d_xy.y, d0)); d1 = h(fmaf(ay.y, d_xy.y, d1));
    d0 = h(fmaf(az.x, d_zz.x, d0)); d1 = h(fmaf(az.y, d_zz.x, d1));
    return (fabsf(d0) < th.x ? 1u : 0u) | (fabsf(d1) < th.y ? 0x10000u : 0u);
#endif
}
// one block of 4 children: boxes, refs, cones (ref / hit point at the block's 4 entries of the NodeVisit)
RT_D void index_visit_block(const float4* nd, bool nocone, vec3 inv, vec3 oi, ConeDir dn, uint32_t* ref, bool* hit) {
    float4 q0, q1, q2, q3;
    ldg8(nd, q0, q1);
    ldg8(nd + 2, q2, q3);
    // q0 = min.x[0..3] min.y[0..3] ; q1 = min.z max.x ; q2 = max.y max.z ; q3 = refs
    // (centre/half layout: centre in place of min, half-extent in place of max)
    const float2 ax01 = unpack_half2(q0.x), ax23 = unpack_half2(q0.y), ay01 = unpack_half2(q0.z), ay23 = unpack_half2(q0.w);
    const float2 az01 = unpack_half2(q1.x), az23 = unpack_half2(q1.y), bx01 = unpack_half2(q1.z), bx23 = unpack_half2(q1.w);
    const float2 by01 = unpack_half2(q2.x), by23 = unpack_half2(q2.y), bz01 = unpack_half2(q2.z), bz23 = unpack_half2(q2.w);
    ref[0] = __float_as_uint(q3.x); ref[1] = __float_as_uint(q3.y);
    ref[2] = __float_as_uint(q3.z); ref[3] = __float_as_uint(q3.w);
#if RTC_NODE_CENTRE_HALF
    slab_ch(ax01.x, ay01.x, az01.x, bx01.x, by01.x, bz01.x, inv, oi, ref[0], hit[0]);
    slab_ch(ax01.y, ay01.y, az01.y, bx01.y, by01.y, bz01.y, inv, oi, ref[1], hit[1]);
    slab_ch(ax23.x, ay23.x, az23.x, bx23.x, by23.x, bz23.x, inv, oi, ref[2], hit[2]);
    slab_ch(ax23.y, ay23.y, az23.y, bx23.y, by23.y, bz23.y, inv, oi, ref[3], hit[3]);
#else
    float tc;
    slab(ax01.x, ay01.x, az01.x, bx01.x, by01.x, bz01.x, inv, oi, ref[0], hit[0], tc);
    slab(ax01.y, ay01.y, az01.y, bx01.y, by01.y, bz01.y, inv, oi, ref[1], hit[1], tc);
    slab(ax23.x, ay23.x, az23.x, bx23.x, by23.x, bz23.x, inv, oi, ref[2], hit[2], tc);
    slab(ax23.y, ay23.y, az23.y, bx23.y, by23.y, bz23.y, inv, oi, ref[3], hit[3], tc);
#endif
#if RTC_NODE_CONES
    // axis.x[0..3] axis.y[0..3] | axis.z[0..3] threshold[0..3]; a node without cones (IREF_NOCONE in the reference that
    // led here) is tested against all-zero thresholds = nothing culled, and one scattered 32-byte load is saved
    float4 q4 = make_float4(0.f, 0.f, 0.f, 0.f), q5 = q4;
    if (!nocone) ldg8(nd + 4, q4, q5);
    const uint32_t c01 = cone_cull_pair(dn, q4.x, q4.z, q5.x, q5.z), c23 = cone_cull_pair(dn, q4.y, q4.w, q5.y, q5.w);
    hit[0] = hit[0] && !(c01 & 1u); hit[1] = hit[1] && !(c01 >> 16);
    hit[2] = hit[2] && !(c23 & 1u); hit[3] = hit[3] && !(c23 >> 16);
#else
    (void)dn;
#endif
}
RT_D NodeVisit index_visit(const DevScene& S, uint32_t node, vec3 inv, vec3 oi, ConeDir dn) {
    const float4* nd = S.inodes + kIndexNodeF4 * (size_t)(node & IREF_NODE_MASK);
    const bool nocone = (node & IREF_NOCONE) != 0;
    NodeVisit v;
#pragma unroll
    for (uint32_t blk = 0; blk < kNodeWidth / 4; ++blk) index_visit_block(nd + kIndexBlockF4 * blk, nocone, inv, oi, dn, v.ref + 4 * blk, v.hit + 4 * blk);
    return v;
}
// closest primitive of one reference leaf (strict <: the first one wins ties, src/bvh.cpp:206-211)
RT_D void leaf_best(const DevScene& S, uint32_t ref, vec3 o, vec3 d, float& bt, int& bid, uint32_t* tests) {
    uint32_t first = ref & 0xFFFFFFu, count = ((ref >> 24) & 0x3Fu) + 1;
    bt = kInfF;
    bid = -1;
    for (uint32_t p = first; p < first + count; ++p) {
        float t;
        if (prim_hit_t(S, p, o, d, t) && t < bt) { bt = t; bid = (int)p; }
    }
    if (tests) *tests += count;
}

// AABB_t::Intersect of a reference LEAF from its stored corners, in the reference's own arithmetic
// (src/bvh.cpp:89-93: s = 0.5 (max - min), centre = 0.5 (max + min), IntersectBox(ray - centre, s) with IEEE
// divisions, src/primitives.cpp:70-97): hit and the entry distance (-inf when the origin is inside the box).
RT_D_COLD void leaf_box_reference(vec3 mn, vec3 mx, vec3 o, vec3 d, bool& hit, float& tc) {  // rare: kept out of line
    const vec3 s = 0.5f * (mx - mn), c = 0.5f * (mx + mn);
    const vec3 oc = o - c;
    const vec3 a = (-s - oc) / d, b = (s - oc) / d;
    const float t1 = fmaxf(fmaxf(fminf(a.x, b.x), fminf(a.y, b.y)), fminf(a.z, b.z));
    const float t2 = fminf(fminf(fmaxf(a.x, b.x), fmaxf(a.y, b.y)), fmaxf(a.z, b.z));
    hit = !(t1 > t2) && !(t2 < 0.f);
    tc = t1 < 0.f ? -kInfF : t1;
}

// Leaf box test = the reference's decision at FMA cost: the min/max * (1/d) slab form first; its rounding error is
// a few ulp of its operands, so a result further than 2e-6 * (|o/d| + |t|) from every decision boundary (t1 = t2,
// t2 = 0, t1 = 0) is the reference's result as well, and only a ray inside that band (it grazes a face or starts
// on one) pays for leaf_box_reference (IEEE divisions were 5 % of k_traverse when every candidate took them).
RT_D void leaf_box(vec3 mn, vec3 mx, vec3 o, vec3 d, vec3 inv, vec3 oi, bool& hit, float& tc) {
    float x1 = fmaf(mn.x, inv.x, -oi.x), x2 = fmaf(mx.x, inv.x, -oi.x);
    float y1 = fmaf(mn.y, inv.y, -oi.y), y2 = fmaf(mx.y, inv.y, -oi.y);
    float z1 = fmaf(mn.z, inv.z, -oi.z), z2 = fmaf(mx.z, inv.z, -oi.z);
    float t1 = fmaxf(fmaxf(fminf(x1, x2), fminf(y1, y2)), fminf(z1, z2));
    float t2 = fminf(fminf(fmaxf(x1, x2), fmaxf(y1, y2)), fmaxf(z1, z2));
    const float band = 2e-6f * (fabsf(oi.x) + fabsf(oi.y) + fabsf(oi.z) + fabsf(t1) + fabsf(t2));
#ifdef RTC_LEAF_BOX_FAST_ONLY   // A/B: never take the exact path (the pre-session-3 behaviour)
    const bool clear = band == band || true;
#else
    const bool clear = fabsf(t2 - t1) > band && fabsf(t2) > band && fabsf(t1) > band;  // NaN / inf: not clear
#endif
    if (!clear) { leaf_box_reference(mn, mx, o, d, hit, tc); return; }
    hit = t1 <= t2 && t2 >= 0.f;
    tc = t1 < 0.f ? -kInfF : t1;
}

// One candidate leaf: the EXACT box of the reference leaf first (a single untransformed triangle
// has min/max of its vertices as its reference AABB, src/bvh.cpp:53-64; other leaves keep theirs in
// ubox) -- the fp16 child boxes of the index nodes only ever ADD candidates, so the set of leaves that pass here
// is the set BVH_t::Intersect_ would reach (unless the ray grazes an ANCESTOR's face within an ulp) -- then its
// primitives.  Returns false when the ray misses the exact box.
RT_D bool leaf_test(const DevScene& S, uint32_t ref, vec3 o, vec3 d, vec3 inv, vec3 oi, float& bt, int& bid, float& tc,
                    uint32_t* tests) {
    const uint32_t first = ref & 0xFFFFFFu;
    const bool fast = (ref & IREF_FAST) != 0;
    bt = kInfF;
    bid = -1;
    float4 g0 = make_float4(0.f, 0.f, 0.f, 0.f), g1 = g0, g2 = g0;
    vec3 mn, mx;
    if (fast) {
        g0 = ldg4(S.geo0 + first); g1 = ldg4(S.geo1 + first); g2 = ldg4(S.geo2 + first);
        mn = mk3(fminf(fminf(g0.x, g1.x), g2.x), fminf(fminf(g0.y, g1.y), g2.y), fminf(fminf(g0.z, g1.z), g2.z));
        mx = mk3(fmaxf(fmaxf(g0.x, g1.x), g2.x), fmaxf(fmaxf(g0.y, g1.y), g2.y), fmaxf(fmaxf(g0.z, g1.z), g2.z));
    } else {
        mn = ld3(ldg4(S.ubox + 2 * (size_t)first));
        mx = ld3(ldg4(S.ubox + 2 * (size_t)first + 1));
    }
    bool hitbox;
    leaf_box(mn, mx, o, d, inv, oi, hitbox, tc);
    if (!hitbox) return false;
    if (fast) {
        float t; bool interior;
        if (isect_triangle(o, d, ld3(g0), ld3(g1), ld3(g2), mk3(g0.w, g1.w, g2.w), t, interior)) { bt = t; bid = (int)first; }
        if (tests) ++*tests;
    } else {
        leaf_best(S, ref, o, d, bt, bid, tests);
    }
    return true;
}

// All reference leaves whose AABB the ray touches, via the index BVH; primitives of a touched
// leaf are tested at once and only leaves with a hit are recorded.  Returns false when more
// than kMaxRecords leaves produced hits (caller falls back to trace_reftree).
// (Straight-line form; the render path runs the same steps from the persistent kernel
// k_traverse in rt_kernels.cu.)
RT_D bool collect_leaf_hits(const DevScene& S, vec3 o, vec3 d, LeafRec* rec, int& k, uint32_t* visits, uint32_t* tests) {
    k = 0;
    if (S.iroot == IREF_NONE) return true;
    vec3 inv = ray_inv(d);
    vec3 oi = o * inv;
    const ConeDir dn = cone_dir(d);
    uint32_t stack[kIndexStack];
    int sp = 0;
    uint32_t ref = S.iroot;
    for (;;) {
        if (ref & IREF_LEAF) {
            float bt, tc; int bid;
            if (leaf_test(S, ref, o, d, inv, oi, bt, bid, tc, tests) && bid >= 0) {
                if (k == kMaxRecords) return false;
                rec[k].key = ref & 0xFFFFFFu; rec[k].id = bid; rec[k].t = bt; rec[k].tcull = tc;
                ++k;
            }
            if (sp == 0) break;
            ref = stack[--sp];
            continue;
        }
        if (visits) ++*visits;
        NodeVisit v = index_visit(S, ref, inv, oi, dn);
        bool have = false;
#pragma unroll
        for (int c = 0; c < (int)kNodeWidth; ++c) {
            if (!v.hit[c]) continue;
            if (!have) { ref = v.ref[c]; have = true; continue; }
            if (sp + 1 > kIndexStack) return false;
            stack[sp++] = v.ref[c];
        }
        if (!have) {
            if (sp == 0) break;
            ref = stack[--sp];
        }
    }
    return true;
}

// Closest plane (planes are stored last and are not part of the BVH), src/scene.cpp:50-66.
// Planes without rotation use the world-space form t = -dot(o - pos, n) / dot(d, n), which is
// what Primitive::Intersect + IntersectPlane evaluate for an identity rotator.
template <uint32_t FEAT = FE_ALL>
RT_D void closest_plane(const DevScene& S, vec3 o, vec3 d, float& closest, int& id) {
    closest = kInfF;
    id = -1;
    for (uint32_t i = 0; i < S.nplanes; ++i) {
        float4 a = ldg4(S.planes + 2 * i), b = ldg4(S.planes + 2 * i + 1);
        uint32_t prim = __float_as_uint(a.w);
        float t;
        bool ok;
        if (!(FEAT & FE_ROTATION) || __float_as_uint(b.w)) {
            vec3 n = ld3(a);
            t = -dot(o - ld3(b), n) / dot(d, n);
            ok = t > 0.f && !(t > S.plane_tmax);
        } else {  // rotated plane: ray into the plane's frame (src/primitives.cpp:15), plane code only
            vec3 lo = o, ld = d;
            to_local(S, prim, prim_flags(S, prim), lo, ld);
            Isect is;
            ok = isect_plane(lo, ld, ld3(a), S.plane_tmax, is);
            t = is.t;
        }
        if (ok && t < closest) { closest = t; id = (int)prim; }
    }
}

struct SceneHit {
    int id;  // -1 = miss
    float t;
    vec3 n;
    int interior;
};

// Scene::RayIntersection, src/scene.cpp:46-77
template <int MODE>
RT_D SceneHit scene_intersect(const DevScene& S, vec3 o, vec3 d, uint32_t* visits, uint32_t* tests, uint32_t* fallbacks) {
    SceneHit h;
    h.id = -1; h.t = 0.f; h.n = mk3(0, 0, 0); h.interior = 0;
    float closest;
    closest_plane(S, o, d, closest, h.id);
    BestHit b;
    if (MODE == 1) {
        b = trace_reftree(S, o, d, closest);
    } else {
        LeafRec rec[kMaxRecords];
        int k;
        if (collect_leaf_hits(S, o, d, rec, k, visits, tests)) b = replay_reference(S, o, d, closest, rec, k);
        else {
            if (fallbacks) ++*fallbacks;
            b = trace_reftree(S, o, d, closest);
        }
    }
    if (b.id != -1 && b.t < closest) h.id = b.id;
    if (h.id >= 0) {
        Isect is;
        prim_intersect(S, (uint32_t)h.id, o, d, is);
        h.t = is.t; h.n = is.n; h.interior = is.interior;
    }
    return h;
}

// Primitive::Intersect restricted to what a light can be (box or ellipsoid): same arithmetic as
// prim_intersect<true>, without the triangle / plane code (k_shade is instruction-cache bound).
template <uint32_t FEAT = FE_ALL>
RT_D bool light_intersect(const DevScene& S, uint32_t prim, bool is_box, vec3 o, vec3 d, Isect& out) {
    uint32_t flags = prim_flags_for<FEAT>(S, prim);
    to_local(S, prim, flags, o, d);
    vec3 g0 = ld3(ldg4(S.geo0 + prim));
    bool ok = (is_box || !(FEAT & FE_ELLIPSOID)) ? isect_box<true>(o, d, g0, out) : isect_ellipsoid(o, d, g0, out);
    if (!ok) return false;
    if (!(flags & PF_ROT_IDENT)) {
        float4 q4 = ldg4(S.xf_rot + prim);
        quat q;
        q.x = q4.x; q.y = q4.y; q.z = q4.z; q.w = q4.w;
        out.n = rotate(q, out.n);
    }
    out.n = rt_normalize<true>(out.n);
    return true;
}

// ------------------------------------------------------------------------------- distributions
// Distribution::SampleCosine, src/distributions.cpp:144-159
RT_D vec3 sample_cosine(const Rng& g, vec3 n) {
    vec3 dir = normal_vec(g.block(1)) + n;
    if (dot(dir, n) <= 1e-8f) return n;
    float dd = dot(dir, dir);
    if (dd <= 1e-8f) return n;  // length(dir) <= 1e-4
    float k = rsqrtf(dd);
    return mk3(dir.x * k, dir.y * k, dir.z * k);
}
// Distribution::SampleBox, src/distributions.cpp:227-269
template <uint32_t FEAT = FE_ALL>
RT_D vec3 sample_box(const DevScene& S, uint32_t prim, const Rng& g, vec3 x) {
    vec3 s = ld3(ldg4(S.geo0 + prim));
    vec3 pos = ld3(ldg4(S.xf_pos + prim));
    float4 q4 = make_float4(0.f, 0.f, 0.f, 1.f);
    if (FEAT & FE_ROTATION) q4 = ldg4(S.xf_rot + prim);
    quat q; q.x = q4.x; q.y = q4.y; q.z = q4.z; q.w = q4.w;
    float wx = s.x * s.x, wy = s.y * s.y, wz = s.z * s.z;
    vec3 smp = mk3(0, 0, 0);
    for (int j = 0; j < kRejectCap; ++j) {
        uint4 A = g.block(2 + 2 * j), B = g.block(3 + 2 * j);
        float u = u01(A.x);
        float side = u01(A.y) <= 0.5f ? 1.f : -1.f;
        u *= wx + wy + wz;
        float c1 = 2.f * u01(A.z) - 1.f, c2 = 2.f * u01(A.w) - 1.f, c3 = 2.f * u01(B.x) - 1.f;
        vec3 pnt = mk3(c1 * s.x, c2 * s.y, c3 * s.z);
        if (u < wx) pnt.x = side * s.x;
        else if (u < wx + wy) pnt.y = side * s.y;
        else pnt.z = side * s.z;
        vec3 on_box = ((FEAT & FE_ROTATION) ? rotate(q, pnt) : pnt) + pos;  // rotate(identity, v) == v exactly
        smp = rt_normalize<true>(on_box - x);
        Isect is;
        if (light_intersect<FEAT>(S, prim, true, x, smp, is)) break;
    }
    return smp;
}
// Distribution::SampleEllipsoid, src/distributions.cpp:318-338
RT_D vec3 sample_ellipsoid(const DevScene& S, uint32_t prim, const Rng& g, vec3 x) {
    vec3 r = ld3(ldg4(S.geo0 + prim));
    vec3 pos = ld3(ldg4(S.xf_pos + prim));
    float4 q4 = ldg4(S.xf_rot + prim);
    quat q; q.x = q4.x; q.y = q4.y; q.z = q4.z; q.w = q4.w;
    vec3 smp = mk3(0, 0, 0);
    for (int j = 0; j < kRejectCap; ++j) {
        vec3 k = normal_vec(g.block(2 + 2 * j));
        vec3 on = rotate(q, r * k) + pos;
        smp = normalize(on - x);
        Isect is;
        if (light_intersect(S, prim, false, x, smp, is)) break;
    }
    return smp;
}
// Distribution::SampleMix, src/distributions.cpp:385-399
// The coin of Distribution::SampleMix for the shading at slot `g.slot`: true = a light is sampled, false = the cosine lobe.
RT_D bool mix_picks_light(const DevScene& S, const Rng& g) { return S.nlights != 0 && !(u01(g.block(0).x) <= 0.5f); }
// `known`: -1 = toss the coin here; 0 / 1 = the caller already knows it came up cosine / light (k_shade keeps the two
// kinds of rays in different warps, rt_kernels.cu) -- the cosine side then never computes block 0.
template <uint32_t FEAT = FE_ALL>
RT_D vec3 mix_sample(const DevScene& S, const Rng& g, vec3 x, vec3 n, int known = -1) {
    if (known == 0) return sample_cosine(g, n);
    uint4 b0 = g.block(0);
    float flip = u01(b0.x);
    if (known < 0 && (S.nlights == 0 || flip <= 0.5f)) return sample_cosine(g, n);
    float fid = u01(b0.y);
    uint32_t id = (uint32_t)floorf(fid * (float)S.nlights);
    uint32_t prim = (uint32_t)__ldg(S.lights + id);
    if (!(FEAT & FE_ELLIPSOID) || (prim_flags(S, prim) & PF_TYPE_MASK) == PT_BOX) return sample_box<FEAT>(S, prim, g, x);
    return sample_ellipsoid(S, prim, g, x);
}
// PdfPointBox / PdfPointEllipsoid, src/distributions.cpp:271-287, 340-347
RT_D float pdf_point(const DevScene& S, uint32_t prim, bool is_box, float dist2, vec3 y, vec3 nrm, vec3 d) {
    vec3 r = ld3(ldg4(S.geo0 + prim));
    float p_y;
    if (is_box) {
        p_y = 1.f / (8.f * (r.x * r.x + r.y * r.y + r.z * r.z));
    } else {
        vec3 pos = ld3(ldg4(S.xf_pos + prim));
        float4 q4 = ldg4(S.xf_rot + prim);
        quat qc; qc.x = -q4.x; qc.y = -q4.y; qc.z = -q4.z; qc.w = q4.w;
        vec3 n = rotate(qc, y - pos) / r;
        p_y = 1.f / (4.f * kPi * length(mk3(n.x * r.y * r.z, r.x * n.y * r.z, r.x * r.y * n.z)));
    }
    return __fdividef(p_y * dist2, fabsf(dot(d, nrm)));
}
// PdfBox / PdfEllipsoid + GetPointsForPdf, src/distributions.cpp:170-198, 289-312, 349-372.
// The reference intersects the light twice: from x, and again from the point 1e-4 behind the first hit.
//  * BOX: the two hits are the entry and the exit of ONE slab computation (outside: both count;
//    inside: only the exit; the second hit is dropped when the chord is shorter than 1e-4), so the
//    box is intersected once -- k_shade spent a quarter of its time in this function.
//  * ELLIPSOID: evaluated exactly as the reference does, with two intersections.  For directions that
//    graze the ellipsoid the float discriminant b^2 - 4ac is cancellation noise, the reference's two
//    roots are then off by ~1e-3 and its pdf several times smaller than the analytic value; a
//    "cleaner" one-pass evaluation is measurably darker than the reference (4 sigma on lights_mix).
template <uint32_t FEAT = FE_ALL>
RT_D float pdf_light(const DevScene& S, uint32_t prim, vec3 x, vec3 d) {
    const uint32_t flags = prim_flags_for<FEAT>(S, prim);
    if ((FEAT & FE_ELLIPSOID) && (flags & PF_TYPE_MASK) != PT_BOX) {
        Isect i1;
        if (!light_intersect(S, prim, false, x, d, i1)) return 1e-9f;
        if (i1.t <= 1e-8f) return 1e-9f;
        vec3 p1 = x + i1.t * d;
        vec3 v1 = p1 - x;
        float sum = pdf_point(S, prim, false, dot(v1, v1), p1, i1.n, d);
        float step = i1.t + 1e-4f;
        Isect i2;
        if (light_intersect(S, prim, false, x + step * d, d, i2)) {
            float t2 = i2.t + step;
            vec3 p2 = x + t2 * d;
            vec3 v2 = p2 - x;
            sum += pdf_point(S, prim, false, dot(v2, v2), p2, i2.n, d);
        }
        return sum;
    }
    vec3 lo = x, ld = d;
    to_local(S, prim, flags, lo, ld);
    const vec3 g = ld3(ldg4(S.geo0 + prim));
    const vec3 inv = mk3(__fdividef(1.f, ld.x), __fdividef(1.f, ld.y), __fdividef(1.f, ld.z));
    const vec3 a = (-g - lo) * inv, b = (g - lo) * inv;
    const float t_in = fmaxf(fmaxf(fminf(a.x, b.x), fminf(a.y, b.y)), fminf(a.z, b.z));
    const float t_out = fminf(fminf(fmaxf(a.x, b.x), fmaxf(a.y, b.y)), fmaxf(a.z, b.z));
    if (t_in > t_out || t_out < 0.f) return 1e-9f;
    const bool inside = t_in < 0.f;
    const float t_first = inside ? t_out : t_in;
    if (t_first <= 1e-8f) return 1e-9f;
    float4 q4 = make_float4(0.f, 0.f, 0.f, 1.f);
    if (!(flags & PF_ROT_IDENT)) q4 = ldg4(S.xf_rot + prim);
    quat q; q.x = q4.x; q.y = q4.y; q.z = q4.z; q.w = q4.w;
    const float dd = dot(d, d);
    const float p_y = __fdividef(1.f, 8.f * (g.x * g.x + g.y * g.y + g.z * g.z));
    const vec3 ginv = mk3(__fdividef(1.f, g.x), __fdividef(1.f, g.y), __fdividef(1.f, g.z));
    float sum = 0.f;
#pragma unroll
    for (int which = 0; which < 2; ++which) {
        const float t = which == 0 ? t_first : t_out;
        if (which == 1 && (inside || t_out - (t_in + 1e-4f) < 0.f)) break;
        vec3 nl = (lo + t * ld) * ginv;  // face normal as Primitive::IntersectBox finds it (p / s, largest component)
        float mx = fmaxf(fmaxf(fabsf(nl.x), fabsf(nl.y)), fabsf(nl.z));
        nl = mk3(fabsf(nl.x) != mx ? 0.f : nl.x, fabsf(nl.y) != mx ? 0.f : nl.y, fabsf(nl.z) != mx ? 0.f : nl.z);
        nl = rt_normalize<true>(nl);
        vec3 nw = (flags & PF_ROT_IDENT) ? nl : rt_normalize<true>(rotate(q, nl));
        sum += __fdividef(p_y * (t * t * dd), fabsf(dot(d, nw)));
    }
    return sum;
}
// Distribution::PdfMix, src/distributions.cpp:401-416
template <uint32_t FEAT = FE_ALL>
RT_D float mix_pdf(const DevScene& S, vec3 x, vec3 n, vec3 d) {
    float sum = fmaxf(0.f, 1.f / kPi * dot(d, n));
    if (S.nlights > 0) {
        float prim_sum = 0.f;
        for (uint32_t i = 0; i < S.nlights; ++i) prim_sum += pdf_light<FEAT>(S, (uint32_t)__ldg(S.lights + i), x, d);
        prim_sum *= 1.f / (float)S.nlights;
        sum = 0.5f * sum + 0.5f * prim_sum;
    }
    return sum;
}

// Camera::GetToRay, src/scene.cpp:180-187, without FMA contraction (bit-exact with the reference)
RT_D void camera_ray(const DevCamera& C, uint32_t width, uint32_t height, float x, float y, vec3& o, vec3& d) {
    float nx = __fmul_rn(__fadd_rn(__fdiv_rn(__fmul_rn(2.f, x), (float)width), -1.f), C.tan_fov_x);
    float ny = __fmul_rn(__fmul_rn(-1.f, __fadd_rn(__fdiv_rn(__fmul_rn(2.f, y), (float)height), -1.f)), C.tan_fov_y);
    o = mk3(C.pos.x, C.pos.y, C.pos.z);
    d.x = __fadd_rn(__fadd_rn(__fmul_rn(nx, C.right.x), __fmul_rn(ny, C.up.x)), __fmul_rn(1.f, C.forward.x));
    d.y = __fadd_rn(__fadd_rn(__fmul_rn(nx, C.right.y), __fmul_rn(ny, C.up.y)), __fmul_rn(1.f, C.forward.y));
    d.z = __fadd_rn(__fadd_rn(__fmul_rn(nx, C.right.z), __fmul_rn(ny, C.up.z)), __fmul_rn(1.f, C.forward.z));
}
// through the scene's own camera
RT_D void camera_ray(const DevScene& S, float x, float y, vec3& o, vec3& d) { camera_ray(S.cam, S.width, S.height, x, y, o, d); }

// GetReflection, src/scene.cpp:79-81
RT_D vec3 reflect_dir(vec3 n, vec3 dir) { return dir - (2.0f * n) * dot(n, dir); }

// ------------------------------------------------------------------------------- thin lens
// Shirley-Chiu concentric map of (u, v) in [0, 1)^2 onto the unit disk, without FMA contraction (the oracle restates it
// in C).  The angle is carried in units of pi, th = angle / pi in [-1/4, 3/4], and sin / cos (pi th) are evaluated in
// double and rounded once to float: sincospi on the device (no argument-reduction table), sin / cos of the double
// product pi th in the host builds (tests/host_emul, the oracle).  The two double results differ by an ulp of a double
// at most, so the float lens points are the same unless one lies within that of a float rounding boundary.
RT_D void concentric_disk(float u, float v, float& lx, float& ly) {
    const float sx = __fadd_rn(__fmul_rn(2.f, u), -1.f), sy = __fadd_rn(__fmul_rn(2.f, v), -1.f);
    if (sx == 0.f && sy == 0.f) { lx = 0.f; ly = 0.f; return; }
    float rad, th;
    if (fabsf(sx) > fabsf(sy)) { rad = sx; th = __fmul_rn(0.25f, __fdiv_rn(sy, sx)); }
    else { rad = sy; th = __fadd_rn(0.5f, -__fmul_rn(0.25f, __fdiv_rn(sx, sy))); }
    float s, c;
#ifdef __CUDA_ARCH__
    double sd, cd;
    sincospi((double)th, &sd, &cd);
    s = (float)sd;
    c = (float)cd;
#else
    s = (float)sin(3.141592653589793 * (double)th);
    c = (float)cos(3.141592653589793 * (double)th);
#endif
    lx = __fmul_rn(rad, c);
    ly = __fmul_rn(rad, s);
}
// The lens step of a camera sample (DESIGN.md "Thin lens"): (o, d) from camera_ray, b = the sample's slot-0 block, whose
// .x / .y gave the jitter; .z / .w pick the lens point (lx, ly).  With e = lx right + ly up the ray starts at o + r e and
// runs along d - (r / f) e: every ray of the sample passes through o + f d, and d keeps its forward coefficient 1.
RT_D void lens_ray(const DevCamera& C, DevLens L, uint4 b, vec3& o, vec3& d) {
    float lx, ly;
    concentric_disk(u01(b.z), u01(b.w), lx, ly);
    const vec3 e = mk3(__fadd_rn(__fmul_rn(lx, C.right.x), __fmul_rn(ly, C.up.x)), __fadd_rn(__fmul_rn(lx, C.right.y), __fmul_rn(ly, C.up.y)),
                       __fadd_rn(__fmul_rn(lx, C.right.z), __fmul_rn(ly, C.up.z)));
    o = mk3(__fadd_rn(o.x, __fmul_rn(L.r, e.x)), __fadd_rn(o.y, __fmul_rn(L.r, e.y)), __fadd_rn(o.z, __fmul_rn(L.r, e.z)));
    d = mk3(__fadd_rn(d.x, -__fmul_rn(L.r_over_f, e.x)), __fadd_rn(d.y, -__fmul_rn(L.r_over_f, e.y)),
            __fadd_rn(d.z, -__fmul_rn(L.r_over_f, e.z)));
}
// The camera ray of a sample at film position (x, y): camera_ray, then, LENS, lens_ray with the sample's slot-0 block b
template <bool LENS>
RT_D void camera_sample(const DevCamera& C, uint32_t width, uint32_t height, float x, float y, uint4 b, DevLens L, vec3& o, vec3& d) {
    camera_ray(C, width, height, x, y, o, d);
    if (LENS) lens_ray(C, L, b, o, d);
}

// ------------------------------------------------------------------------------- per-pixel candidate leaves
// All camera rays of a pixel start at C.pos and differ only by their jitter, so one conservative traversal of the index
// tree with the pixel's whole beam of directions (pixel_candidates) finds every leaf the index traversal of any of its
// rays can reach.  A camera ray then tests those leaves exactly (leaf_test) and replays the reference over the ones with
// a hit (camera_path in rt_kernels.cu), with no node visit and no traverse-queue record.  Since the list is a superset
// of what the ray's own traversal reaches and the exact leaf_test decides, the set of hit leaves and so the id are the
// same (DESIGN.md "Camera rays from per-pixel candidate lists").
//
// A pixel whose beam reaches more than kMaxRecords leaves, or at whose nodes k_traverse could run out of stack, is
// marked kPixelTraverse: its rays take pre_step and k_traverse as every other ray does.  A thin lens gives every sample its own origin;
// lens renders build no lists (measured slower than the index traversal: DESIGN.md "Thin lens").
constexpr uint32_t kPixelTraverse = 0xFFFFFFFFu;
// k_traverse's per-lane stack (rt_kernels.cu): inner-node stack from the bottom, noted leaves from the top
constexpr int kStackWords = 56;
// Slack of the beam's cone test against cone_cull_pair's half arithmetic: the ray's direction rounded to half (2^-11
// relative), one product and two fused sums each rounded to half (2^-11 of |ax dx| + |ay dy| + |az dz| <= |axis| <= 1.001
// each) stay below 4 * 2^-11 * 1.001 = 1.96e-3 together; the float work of cone_dir adds ~1e-6.  Twice that is kept.
constexpr float kBeamConeSlack = 1.f / 256.f;
// Relative slack of the beam's slab test against the per-ray slab_ch (approximate reciprocal, 1-2 ulp; fma of the centre
// and the half-extent, one ulp each): a few 2^-23 of (|centre| + |half| + |origin|) / |d|.  1e-5 is ~40 times that.
constexpr float kBeamBoxSlack = 1e-5f;

// The directions camera_ray makes for the jittered samples of pixel (x, y) through camera C.  Every step of camera_ray
// (correctly rounded products, sums, one division) is monotone in its input, so each direction component is monotone in
// fx and in fy separately, and its range over the pixel is spanned by the four corner samples: jitter u = 0 and
// u = 1 - 2^-24, the largest u01 (plus hw3's half pixel).  The range is exact for float directions, no widening needed.
struct Beam {
    vec3 o;        // common origin
    vec3 lo, hi;   // per axis: least and greatest direction component of any sample
    vec3 c;        // unit direction the cone test measures from
    float r;       // bound on |normalize(d) - c| over the pixel's samples
};
RT_D Beam pixel_beam(const DevCamera& C, uint32_t width, uint32_t height, uint32_t dialect, uint32_t x, uint32_t y) {
    const float umax = (float)0xFFFFFFu * (1.0f / 16777216.0f);
    float fx[2] = {__fadd_rn((float)x, 0.f), __fadd_rn((float)x, umax)}, fy[2] = {__fadd_rn((float)y, 0.f), __fadd_rn((float)y, umax)};
    if (dialect == DIALECT_HW3)
        for (int i = 0; i < 2; ++i) { fx[i] = __fadd_rn(fx[i], 0.5f); fy[i] = __fadd_rn(fy[i], 0.5f); }
    Beam B;
    vec3 dn[4], sum = mk3(0.f, 0.f, 0.f);
    for (int i = 0; i < 4; ++i) {
        vec3 d;
        camera_ray(C, width, height, fx[i & 1], fy[i >> 1], B.o, d);
        B.lo = i ? mk3(fminf(B.lo.x, d.x), fminf(B.lo.y, d.y), fminf(B.lo.z, d.z)) : d;
        B.hi = i ? mk3(fmaxf(B.hi.x, d.x), fmaxf(B.hi.y, d.y), fmaxf(B.hi.z, d.z)) : d;
        dn[i] = normalize(d);
        sum = sum + dn[i];
    }
    // the directions lie on the plane camera_ray maps the pixel to; on that plane {p : angle(p, c) <= a} is convex for
    // a < 90 degrees, so the angle to c, and with it |normalize(d) - c|, is greatest at a corner (1e-5: float rounding)
    B.c = normalize(sum);
    B.r = 0.f;
    for (int i = 0; i < 4; ++i) B.r = fmaxf(B.r, length(dn[i] - B.c));
    B.r += 1e-5f;
    return B;
}
// Slab entry / exit distances of one axis over the beam, widened by the slack of the per-ray test: (-inf, inf) when the
// beam's direction interval holds 0 or a component so small that ray_inv clamps it.
RT_D void beam_axis(float mn, float mx, float o, float lo, float hi, float slack, float& t_in, float& t_out) {
    if (!(fminf(fabsf(lo), fabsf(hi)) >= 1e-20f) || (lo < 0.f) != (hi < 0.f)) { t_in = -kInfF; t_out = kInfF; return; }
    const float il = 1.f / lo, ih = 1.f / hi;
    const float a = mn - o, b = mx - o;
    const float m = slack * (fabsf(mn) + fabsf(mx) + 2.f * fabsf(o)) * fmaxf(fabsf(il), fabsf(ih));
    t_in = fminf(fminf(a * il, a * ih), fminf(b * il, b * ih)) - m;
    t_out = fmaxf(fmaxf(a * il, a * ih), fmaxf(b * il, b * ih)) + m;
}
// The child boxes of one block of 4 children (centre / half-extent halves, index_visit_block's layout) and their cones,
// against the whole beam: bit c set when child c may be hit by some ray of the beam.  A child is dropped only when every
// direction of the beam fails slab_ch (interval slab test, NaN keeps the child) or every one is culled by cone_cull_pair.
RT_D uint32_t beam_visit_block(const float4* nd, bool nocone, const Beam& B) {
    const float4 q0 = ldg4(nd), q1 = ldg4(nd + 1), q2 = ldg4(nd + 2), q3 = ldg4(nd + 3);
    const float2 c[3][2] = {{unpack_half2(q0.x), unpack_half2(q0.y)}, {unpack_half2(q0.z), unpack_half2(q0.w)}, {unpack_half2(q1.x), unpack_half2(q1.y)}};
    const float2 h[3][2] = {{unpack_half2(q1.z), unpack_half2(q1.w)}, {unpack_half2(q2.x), unpack_half2(q2.y)}, {unpack_half2(q2.z), unpack_half2(q2.w)}};
    const uint32_t ref[4] = {__float_as_uint(q3.x), __float_as_uint(q3.y), __float_as_uint(q3.z), __float_as_uint(q3.w)};
    const float o[3] = {B.o.x, B.o.y, B.o.z}, lo[3] = {B.lo.x, B.lo.y, B.lo.z}, hi[3] = {B.hi.x, B.hi.y, B.hi.z};
    float4 q4 = make_float4(0.f, 0.f, 0.f, 0.f), q5 = q4;
#if RTC_NODE_CONES
    if (!nocone) { q4 = ldg4(nd + 4); q5 = ldg4(nd + 5); }
#else
    (void)nocone;
#endif
    const float2 ax[2] = {unpack_half2(q4.x), unpack_half2(q4.y)}, ay[2] = {unpack_half2(q4.z), unpack_half2(q4.w)};
    const float2 az[2] = {unpack_half2(q5.x), unpack_half2(q5.y)}, th[2] = {unpack_half2(q5.z), unpack_half2(q5.w)};
    uint32_t mask = 0;
    for (int i = 0; i < 4; ++i) {
        if (ref[i] == IREF_NONE) continue;
        auto pick = [i](const float2* v) { return (i & 1) ? v[i >> 1].y : v[i >> 1].x; };
        float t1 = -kInfF, t2 = kInfF;
        for (int a = 0; a < 3; ++a) {
            const float cc = pick(c[a]), hh = pick(h[a]);
#if RTC_NODE_CENTRE_HALF
            const float mn = cc - hh, mx = cc + hh;
#else
            const float mn = cc, mx = hh;
#endif
            float ti, to;
            beam_axis(mn, mx, o[a], lo[a], hi[a], kBeamBoxSlack, ti, to);
            t1 = fmaxf(t1, ti);
            t2 = fminf(t2, to);
        }
        if (t1 > t2 || t2 < 0.f) continue;
        const float wx = pick(ax), wy = pick(ay), wz = pick(az), thr = pick(th);
        const float len = sqrtf(wx * wx + wy * wy + wz * wz);
        if (fabsf(B.c.x * wx + B.c.y * wy + B.c.z * wz) + B.r * len + kBeamConeSlack < thr) continue;
        mask |= 1u << i;
    }
    return mask;
}
// The candidate leaves of pixel (x, y) into out[0 .. n) (any order; refs as in the index tree); returns n, or
// kPixelTraverse.  `visits` (optional) counts the nodes visited.
//   * More than kMaxRecords candidates: kPixelTraverse (a ray that could need more records takes k_traverse's fallback).
//   * k_traverse overflows a lane only when, before a visit, its inner-node stack holds more than kStackWords -
//     (2 kNodeWidth - 1) entries.  Before it visits node u a ray holds at most sum over u's ancestors a of (inner children
//     of a the ray enters - 1), and a ray enters a subset of what the beam enters; `pend` carries that sum for the beam,
//     and a pixel where it can reach the limit is kPixelTraverse.
RT_D uint32_t pixel_candidates(const DevScene& S, const Beam& B, uint32_t* out, uint32_t* visits) {
    if (S.iroot == IREF_NONE) return kPixelTraverse;
    if (S.iroot & IREF_LEAF) { out[0] = S.iroot; return 1u; }
    uint32_t stk[kIndexStack], pst[kIndexStack];
    int sp = 0;
    uint32_t n = 0, node = S.iroot, pend = 0;
    for (;;) {
        if ((int)pend + (int)(2 * kNodeWidth - 1) > kStackWords) return kPixelTraverse;
        if (visits) ++*visits;
        const float4* nd = S.inodes + kIndexNodeF4 * (size_t)(node & IREF_NODE_MASK);
        const bool nocone = (node & IREF_NOCONE) != 0;
        uint32_t inner = 0;
        const int sp0 = sp;
        for (uint32_t blk = 0; blk < kNodeWidth / 4; ++blk) {
            const float4* bd = nd + kIndexBlockF4 * blk;
            const uint32_t m = beam_visit_block(bd, nocone, B);
            const float4 q3 = ldg4(bd + 3);
            const uint32_t ref[4] = {__float_as_uint(q3.x), __float_as_uint(q3.y), __float_as_uint(q3.z), __float_as_uint(q3.w)};
            for (int i = 0; i < 4; ++i) {
                if (!(m >> i & 1u)) continue;
                if (ref[i] & IREF_LEAF) {
                    if (n == (uint32_t)kMaxRecords) return kPixelTraverse;
                    out[n++] = ref[i];
                } else {
                    if (sp == kIndexStack) return kPixelTraverse;
                    stk[sp++] = ref[i];
                    ++inner;
                }
            }
        }
        for (int j = sp0; j < sp; ++j) pst[j] = pend + (inner > 0 ? inner - 1 : 0);
        if (sp == 0) break;
        --sp;
        node = stk[sp];
        pend = pst[sp];
    }
    return n;
}

}  // namespace rtc
