// bvh_build.cpp -- Scene::InitScene on the host: primitive order, the reference's SAH BVH, the
// light list, then OUR acceleration data (index BVH over the reference's leaves + an LCA table)
// and the flattening into float4 arrays for HBM.
//
// Why two trees.  The reference's traversal result depends on its BVH topology: a primitive is
// tested only if the ray passes the AABB test of every ancestor, where a node is skipped when
// `closest_dist < t_enter && !interior` (src/bvh.cpp:185-198) and closest_dist is the hit
// distance found in the left sibling subtree.  Because IntersectTriangle intersects the plane
// through the LOCAL ORIGIN (src/primitives.cpp:155-157), hit points do not lie inside the AABBs
// and that skipping rule changes results, so a drop-in replacement has to reproduce it.  On the
// dragon scenes every triangle has POSITION 0 0 0, the sort keys are all equal, and the
// resulting tree is nearly useless for culling (~1100 node visits per primary ray on 10k
// triangles).  We therefore keep the reference tree only as the DEFINITION of the result and
// find the leaves a ray touches with a second, spatially good BVH (index BVH); the reference
// recursion is then replayed on just those leaves, using lowest-common-ancestor queries on
// the reference tree (DESIGN.md "Traversal").
#include <algorithm>
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <cmath>
#include <cstring>
#include <future>
#include <thread>
#include <numeric>
#include <stdexcept>

#include "scene_host.h"

namespace rtc {

static const float kInf = 1e18f;  // include/bvh.h:9

static Aabb empty_box() { return Aabb{{kInf, kInf, kInf}, {-kInf, -kInf, -kInf}}; }
static void grow(Aabb& b, vec3 p) {  // AABB_t::Extend(Point) src/bvh.cpp:29-34
    b.mx.x = std::max(b.mx.x, p.x); b.mn.x = std::min(b.mn.x, p.x);
    b.mx.y = std::max(b.mx.y, p.y); b.mn.y = std::min(b.mn.y, p.y);
    b.mx.z = std::max(b.mx.z, p.z); b.mn.z = std::min(b.mn.z, p.z);
}
static void grow(Aabb& b, const Aabb& o) { grow(b, o.mx); grow(b, o.mn); }  // src/bvh.cpp:36-39
static float surface(const Aabb& b) {                                        // src/bvh.cpp:23-27
    vec3 d = b.mx - b.mn;
    return 2.f * (d.x * d.y + d.x * d.z + d.y * d.z);
}

Aabb aabb_of_primitive(const Primitive& p) {
    vec3 lo, hi;
    if (p.type == PT_TRIANGLE) {
        lo = mk3(std::min({p.d0.x, p.d1.x, p.d2.x}), std::min({p.d0.y, p.d1.y, p.d2.y}), std::min({p.d0.z, p.d1.z, p.d2.z}));
        hi = mk3(std::max({p.d0.x, p.d1.x, p.d2.x}), std::max({p.d0.y, p.d1.y, p.d2.y}), std::max({p.d0.z, p.d1.z, p.d2.z}));
    } else if (p.type == PT_BOX || p.type == PT_ELLIPSOID) {
        lo = -1.f * p.d0;
        hi = p.d0;
    } else {
        throw std::runtime_error("aabb_of_primitive: primitive type has no bounding box");
    }
    Aabb b = empty_box();
    for (int corner = 0; corner < 8; ++corner) {
        vec3 v = mk3((corner & 1) ? hi.x : lo.x, (corner & 2) ? hi.y : lo.y, (corner & 4) ? hi.z : lo.z);
        grow(b, rotate(p.rot, v));
    }
    b.mn = b.mn + p.pos;
    b.mx = b.mx + p.pos;
    return b;
}

// ---------------------------------------------------------------------------------------------
// Reference-order SAH BVH (BVH_t::InitTree, src/bvh.cpp:105-179).  Works on a permutation of
// primitive indices; std::sort / std::partition are the very library routines the reference
// calls, with an equivalent comparator, so equal keys end up in the same order as there.
namespace {
// levels of the two tree builds whose halves run concurrently: 2^levels tasks at most (RTC_BUILD_THREADS=1: serial)
int build_parallel_levels() {
    unsigned threads = std::thread::hardware_concurrency();
    if (const char* v = std::getenv("RTC_BUILD_THREADS")) threads = (unsigned)std::atoi(v);
    int levels = 0;
    while (levels < 5 && (2u << levels) <= threads) ++levels;
    return levels;
}

struct RefBuilder {
    std::vector<int32_t>& perm;
    const std::vector<Aabb>& box;         // per original primitive
    const std::vector<Primitive>& prims;  // original order
    std::vector<float> cost;

    void sort_axis(uint32_t first, uint32_t last, int axis) {
        const Primitive* P = prims.data();
        std::sort(perm.begin() + first, perm.begin() + last,
                  [P, axis](int32_t a, int32_t b) { return idx(P[a].pos, axis) < idx(P[b].pos, axis); });
    }

    // Appends the subtree of perm[first, last) to `out` in creation (pre-)order and returns the index of its root.
    // The two halves of a node are independent (disjoint ranges of perm and cost): for the top `par` levels they are
    // built concurrently into vectors of their own and appended left-then-right, which is exactly the order -- and
    // therefore the node numbering -- of the reference's serial recursion.
    uint32_t build(std::vector<RefNode>& out, uint32_t first, uint32_t last, int par) {
        Aabb all = empty_box();
        for (uint32_t i = first; i < last; ++i) grow(all, box[perm[i]]);
        uint32_t me = (uint32_t)out.size();
        out.push_back(RefNode{all, UINT32_MAX, UINT32_MAX, first, last - first});
        if (last - first == 1) return me;

        float best[3] = {kInf, kInf, kInf};
        uint32_t where[3] = {0, 0, 0};
        for (int axis = 0; axis < 3; ++axis) {
            sort_axis(first, last, axis);
            // cost[cut] = S(first..cut-1) * (cut-first) + S(cut..last-1) * (last-cut)
            Aabb left = box[perm[first]];
            for (uint32_t cut = first + 1; cut < last; ++cut) {
                cost[cut] = surface(left) * (cut - first);
                grow(left, box[perm[cut]]);
            }
            Aabb right = empty_box();
            for (uint32_t cut = last - 1; cut > first; --cut) {
                grow(right, box[perm[cut]]);
                cost[cut] += surface(right) * (last - cut);
            }
            for (uint32_t cut = first + 1; cut < last; ++cut)
                if (cost[cut] < best[axis]) { best[axis] = cost[cut]; where[axis] = cut; }
        }
        float optimum = std::min({best[0], best[1], best[2]});
        float leaf_cost = surface(all) * (last - first);
        if (optimum >= leaf_cost) return me;

        uint32_t cut = 0;
        for (int axis = 0; axis < 3; ++axis) {
            if (optimum == best[axis]) {
                sort_axis(first, last, axis);  // re-sort: moves equal keys again, exactly as the reference does
                cut = where[axis];
                break;
            }
        }
        // No cut costs less than kInf, but the leaf costs more (or is NaN): boxes whose surface areas reach 1e18.  The
        // reference then builds an empty child and recurses on the same range until its stack overflows.
        if (cut == 0) throw std::runtime_error("the SAH finds no cut below 1e18 for a BVH node that is too costly as a leaf (primitive boxes too large)");
        if (par > 0 && last - first >= 4096) {
            std::vector<RefNode> lhs, rhs;
            auto other = std::async(std::launch::async, [&] { build(lhs, first, cut, par - 1); });
            build(rhs, cut, last, par - 1);
            other.get();
            for (std::vector<RefNode>* half : {&lhs, &rhs}) {
                const uint32_t off = (uint32_t)out.size();
                (half == &lhs ? out[me].left : out[me].right) = off;
                for (RefNode n : *half) {
                    if (n.left != UINT32_MAX) { n.left += off; n.right += off; }
                    out.push_back(n);
                }
            }
            return me;
        }
        uint32_t l = build(out, first, cut, 0);
        out[me].left = l;
        uint32_t r = build(out, cut, last, 0);
        out[me].right = r;
        return me;
    }
};

// ---------------------------------------------------------------------------------------------
// Index BVH: a SAH tree over the reference's LEAVES ("units"), built binary and collapsed to 4-wide nodes.  Every unit keeps
// exactly the AABB the reference stores for that leaf; traversal reports all units whose AABB
// the ray touches (no ordering, no early out -- see the header comment).
// Feasibility cone of a set of reference leaves: every ray that can produce a hit in the set has its direction
// within `alpha` of +axis or of -axis.  Why such a cone exists: Primitive::IntersectTriangle intersects the plane
// through the ORIGIN (src/primitives.cpp:155-157), so triangle T = (a, b, c) with unit normal n is rendered as
// T' = T - (a.n) n, while BVH_t::Intersect_ still demands that the ray touches the AABB of the real T
// (src/bvh.cpp:194-198).  A ray through a point of T' and a point x of a box that contains T has direction
// (a.n) n + (x - q), q in T: within asin(diag(box) / |a.n|) of +-n.  alpha >= pi/2 means "no restriction".
struct Cone {
    double ax = 0, ay = 0, az = 1, alpha = 4.0;
    bool open() const { return !(alpha < 1.5707); }
};
static Cone merge_cones(const Cone& a, const Cone& b) {
    if (a.open() || b.open()) return Cone{};
    double dt = a.ax * b.ax + a.ay * b.ay + a.az * b.az;
    const double sgn = dt < 0 ? -1.0 : 1.0;  // +-axis describe the same double cone: take the closer one
    dt = std::min(1.0, std::fabs(dt));
    const double bx = sgn * b.ax, by = sgn * b.ay, bz = sgn * b.az;
    const double gamma = std::acos(dt);
    if (gamma + b.alpha <= a.alpha) return a;
    if (gamma + a.alpha <= b.alpha) return Cone{bx, by, bz, b.alpha};
    Cone r;
    r.alpha = 0.5 * (gamma + a.alpha + b.alpha) * (1.0 + 1e-9) + 1e-9;
    if (r.open()) return Cone{};
    // axis: a's axis turned towards b's by (alpha_new - a.alpha), inside the plane of the two (slerp)
    const double tt = (r.alpha - a.alpha) / gamma;
    const double sg = std::sin(gamma);
    const double wa = std::sin((1.0 - tt) * gamma) / sg, wb = std::sin(tt * gamma) / sg;
    r.ax = wa * a.ax + wb * bx; r.ay = wa * a.ay + wb * by; r.az = wa * a.az + wb * bz;
    const double len = std::sqrt(r.ax * r.ax + r.ay * r.ay + r.az * r.az);
    r.ax /= len; r.ay /= len; r.az /= len;
    return r;
}
// cone of one reference leaf holding prims[first .. first + count) inside `box`
static Cone cone_of_leaf(const std::vector<Primitive>& prims, uint32_t first, uint32_t count, const Aabb& box) {
    const double ex = (double)box.mx.x - box.mn.x, ey = (double)box.mx.y - box.mn.y, ez = (double)box.mx.z - box.mn.z;
    double scale = 0;
    for (float v : {box.mn.x, box.mn.y, box.mn.z, box.mx.x, box.mx.y, box.mx.z}) scale = std::max(scale, (double)std::fabs(v));
    // generous slack for the float arithmetic of the slab test and of the orientation tests
    const double diag = std::sqrt(ex * ex + ey * ey + ez * ez) * 1.001 + 1e-5 * scale + 1e-30;
    if (!(diag < 1e30)) return Cone{};
    Cone all;
    bool have = false;
    for (uint32_t i = first; i < first + count; ++i) {
        const Primitive& p = prims[i];
        const bool ident = p.rot.x == 0.f && p.rot.y == 0.f && p.rot.z == 0.f && p.rot.w == 1.f && p.pos.x == 0.f &&
                           p.pos.y == 0.f && p.pos.z == 0.f;
        if (p.type != PT_TRIANGLE || !ident) return Cone{};
        const double ux = (double)p.d1.x - p.d0.x, uy = (double)p.d1.y - p.d0.y, uz = (double)p.d1.z - p.d0.z;
        const double vx = (double)p.d2.x - p.d0.x, vy = (double)p.d2.y - p.d0.y, vz = (double)p.d2.z - p.d0.z;
        double nx = uy * vz - uz * vy, ny = uz * vx - ux * vz, nz = ux * vy - uy * vx;
        const double len = std::sqrt(nx * nx + ny * ny + nz * nz);
        if (!(len > 1e-30)) return Cone{};  // degenerate triangle: its float normal is noise
        nx /= len; ny /= len; nz /= len;
        const double h = std::fabs(p.d0.x * nx + p.d0.y * ny + p.d0.z * nz);
        // the device tests with the FLOAT normal (normalize(cross) in float, relative error ~1e-6 per
        // component, far more for slivers): its plane offset and direction differ from ours by that much
        const double sliver = 4e-7 * (std::sqrt(ux * ux + uy * uy + uz * uz) * std::sqrt(vx * vx + vy * vy + vz * vz)) / len;
        const double ratio = (diag + sliver * (h + scale)) / h;
        if (!(ratio < 0.999)) return Cone{};
        Cone c{nx, ny, nz, std::asin(ratio) + sliver};
        all = have ? merge_cones(all, c) : c;
        have = true;
        if (all.open()) return Cone{};
    }
    return have ? all : Cone{};
}

struct Unit {
    Aabb box;
    uint32_t first, count;
    vec3 centre;
    bool fast;  // a single untransformed triangle: its box is min/max of its vertices
    Cone cone;
};
// float -> IEEE half bits, round to nearest even (finite inputs; overflow gives infinity)
static uint16_t half_bits_rn(float f) {
    uint32_t x;
    std::memcpy(&x, &f, 4);
    const uint32_t sign = (x >> 16) & 0x8000u;
    x &= 0x7FFFFFFFu;
    if (x >= 0x47800000u) return (uint16_t)(sign | 0x7C00u);           // >= 65536 (or inf/nan) -> inf
    if (x < 0x38800000u) {                                             // subnormal half (or zero)
        if (x < 0x33000000u) return (uint16_t)sign;
        const uint32_t shift = 113u - (x >> 23);
        const uint32_t mant = (x & 0x7FFFFFu) | 0x800000u;
        uint32_t h = mant >> (shift + 13);
        const uint32_t rem = mant & ((1u << (shift + 13)) - 1u), half = 1u << (shift + 12);
        if (rem > half || (rem == half && (h & 1u))) ++h;
        return (uint16_t)(sign | h);
    }
    uint32_t h = ((x - 0x38000000u) >> 13);
    const uint32_t rem = x & 0x1FFFu;
    if (rem > 0x1000u || (rem == 0x1000u && (h & 1u))) ++h;
    return (uint16_t)(sign | h);
}
static float half_to_float(uint16_t h) {
    const uint32_t sign = (uint32_t)(h & 0x8000u) << 16, e = (h >> 10) & 0x1Fu, m = h & 0x3FFu;
    float f;
    if (e == 0) f = std::ldexp((float)m, -24);
    else if (e == 31) f = m ? NAN : INFINITY;
    else f = std::ldexp((float)(m | 0x400u), (int)e - 25);
    return sign ? -f : f;
}
// the largest half <= f (down) / the smallest half >= f (up): conservative child boxes
static uint16_t half_down(float f) {
    uint16_t h = half_bits_rn(f);
    if (half_to_float(h) > f) h = (h & 0x8000u) ? (uint16_t)(h + 1) : (h == 0 ? (uint16_t)0x8001u : (uint16_t)(h - 1));
    return h;
}
static uint16_t half_up(float f) {
    uint16_t h = half_bits_rn(f);
    if (half_to_float(h) < f) h = (h & 0x8000u) ? (h == 0x8000u ? (uint16_t)0x0001u : (uint16_t)(h - 1)) : (uint16_t)(h + 1);
    return h;
}

struct IndexBuilder {
    const std::vector<Unit>& units;
    std::vector<f4>& out;  // kIndexNodeF4 f4 (96 bytes) per 4-wide node
    std::vector<float> rarea;
    double slack = 0;  // absolute inflation of every child half-extent: 2^-20 of the scene size (set by HostScene::init)

    static uint32_t leaf_ref(const Unit& u) { return IREF_LEAF | (u.fast ? IREF_FAST : 0u) | ((u.count - 1) << 24) | u.first; }
    static f4 bits4(uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
        f4 r;
        std::memcpy(&r.x, &a, 4); std::memcpy(&r.y, &b, 4); std::memcpy(&r.z, &c, 4); std::memcpy(&r.w, &d, 4);
        return r;
    }
    Aabb bound(uint32_t lo, uint32_t hi) const {
        Aabb b = empty_box();
        for (uint32_t i = lo; i < hi; ++i) grow(b, units[sorted[0][i]].box);
        return b;
    }
    // Unit ids ordered by (centre[axis], id), one array per axis; a range [lo, hi) holds the same SET of units in all
    // three, so a node sweeps each axis without sorting and a split only has to partition the other two arrays
    // stably (O(n) per level instead of three sorts per node: 2.2 s -> 0.9 s for 100k units, same tree bit for bit).
    std::vector<uint32_t> sorted[3];
    std::vector<uint32_t> scratch;
    std::vector<uint8_t> left_side;
    void prepare() {
        const uint32_t n = (uint32_t)units.size();
        for (int axis = 0; axis < 3; ++axis) {
            sorted[axis].resize(n);
            std::iota(sorted[axis].begin(), sorted[axis].end(), 0u);
            std::sort(sorted[axis].begin(), sorted[axis].end(), [&](uint32_t a, uint32_t b) {
                float ca = idx(units[a].centre, axis), cb = idx(units[b].centre, axis);
                return ca < cb || (ca == cb && a < b);
            });
        }
        scratch.resize(n);
        left_side.assign(n, 0);
    }
    struct Bin {
        Aabb box[2];
        uint32_t ref[2];
        Cone cone[2];
    };
    std::vector<Bin> tmp;
    // Appends the binary subtree of the units in [lo, hi) to `out` (pre-order); returns its child reference (a leaf
    // reference, or the index of its root in `out`) and the feasibility cone of the subtree.  As in RefBuilder the two
    // sides of a split touch disjoint ranges of every array, and the top `par` levels build them concurrently.
    uint32_t build(std::vector<Bin>& out, uint32_t lo, uint32_t hi, uint32_t depth, Cone& cone, int par) {
        if (hi - lo == 1) { cone = units[sorted[0][lo]].cone; return leaf_ref(units[sorted[0][lo]]); }
        // Split cost = sum over the two sides of P(a random ray enters the side) * units in it, with
        // P = surface of the box * fraction of directions inside the feasibility cone.  Candidate orders: the
        // unit centres along x, y, z (|axis.x|, |axis.y|, |axis.z| of the units' cones as three more orders would group
        // faces of one orientation where the surface folds back on itself; measured: the greedy cost never profits,
        // 5.35 vs 5.32 visits, and forced 2-means orientation splits below 64 .. 4096 units make it worse:
        // profiles/r01_experiments.md).  The cone factor itself: 5.54 -> 5.32 index node visits per random ray.
        auto frac = [&](const Cone& c) -> float { return c.open() ? 1.f : (float)(1.0 - std::cos(c.alpha)); };
        float best = 3.0e38f;
        int best_axis = -1;
        uint32_t best_cut = 0;
        for (int axis = 0; axis < 3; ++axis) {
            const std::vector<uint32_t>& order = sorted[axis];
            Aabb r = empty_box();
            Cone rc;
            for (uint32_t i = hi - 1; i > lo; --i) {
                const Unit& u = units[order[i]];
                grow(r, u.box);
                rc = (i == hi - 1) ? u.cone : merge_cones(rc, u.cone);
                rarea[i] = surface(r) * frac(rc);
            }
            Aabb l = empty_box();
            Cone lc;
            for (uint32_t i = lo + 1; i < hi; ++i) {
                const Unit& u = units[order[i - 1]];
                grow(l, u.box);
                lc = (i == lo + 1) ? u.cone : merge_cones(lc, u.cone);
                float c = surface(l) * frac(lc) * (i - lo) + rarea[i] * (hi - i);
                if (c < best) { best = c; best_axis = axis; best_cut = i; }
            }
        }
        if (best_axis < 0) {  // every candidate cost was NaN/inf (degenerate boxes): split in the middle
            best_axis = 2;
            best_cut = lo + (hi - lo) / 2;
        }
        // the left side is the head of the winning order; the other two orders are partitioned stably around it
        for (uint32_t i = lo; i < best_cut; ++i) left_side[sorted[best_axis][i]] = 1;
        for (int axis = 0; axis < 3; ++axis) {
            if (axis == best_axis) continue;
            std::vector<uint32_t>& order = sorted[axis];
            uint32_t nl = lo, nr = 0;
            for (uint32_t i = lo; i < hi; ++i) {
                if (left_side[order[i]]) order[nl++] = order[i];
                else scratch[lo + nr++] = order[i];
            }
            std::copy(scratch.begin() + lo, scratch.begin() + lo + nr, order.begin() + nl);
        }
        for (uint32_t i = lo; i < best_cut; ++i) left_side[sorted[best_axis][i]] = 0;
        // binary node in a temporary tree; emit() collapses it to 4-wide nodes afterwards
        uint32_t me = (uint32_t)out.size();
        out.push_back(Bin{});
        Aabb lb = bound(lo, best_cut), rb = bound(best_cut, hi);
        Cone lc, rc;
        uint32_t lref, rref;
        if (par > 0 && hi - lo >= 4096) {
            std::vector<Bin> lhs, rhs;
            auto other = std::async(std::launch::async, [&] { lref = build(lhs, lo, best_cut, depth + 1, lc, par - 1); });
            rref = build(rhs, best_cut, hi, depth + 1, rc, par - 1);
            other.get();
            for (std::vector<Bin>* half : {&lhs, &rhs}) {
                const uint32_t off = (uint32_t)out.size();
                uint32_t& top = half == &lhs ? lref : rref;
                if (!(top & IREF_LEAF)) top += off;
                for (Bin b : *half) {
                    for (uint32_t& r : b.ref) if (!(r & IREF_LEAF)) r += off;
                    out.push_back(b);
                }
            }
        } else {
            lref = build(out, lo, best_cut, depth + 1, lc, 0);
            rref = build(out, best_cut, hi, depth + 1, rc, 0);
        }
        out[me] = Bin{{lb, rb}, {lref, rref}, {lc, rc}};
        cone = merge_cones(lc, rc);
        return me;
    }

    uint32_t wide_depth = 0;

    // ---- optimal collapse of the binary tree into 4-wide nodes (dynamic programme over the binary tree).
    // Visiting a wide node costs the same whatever it holds, so the quantity to minimise is the expected number of
    // wide nodes a random ray enters: sum over wide nodes of P(enter) = surface of its box * fraction of directions
    // inside its cone.  best[n][k-1] = least such sum for the subtree of binary node n when it may occupy at most k
    // slots of its parent's wide node: either one slot (n becomes a wide node itself: P(n) + its own best use of W
    // slots), or the slots are shared between its two children.  A leaf costs nothing in any number of slots.
    static constexpr int W = (int)kNodeWidth;
    struct Plan {
        float cost[W];
        uint8_t left[W];  // slots given to the left child when the subtree is spread over k slots; 0 = "n is one wide node"
    };
    std::vector<Plan> plan;
    float entered(const Aabb& box, const Cone& cone) const {
        return surface(box) * (cone.open() ? 1.f : (float)(1.0 - std::cos(cone.alpha)));
    }
    float plan_cost(uint32_t ref, int k) const { return (ref & IREF_LEAF) ? 0.f : plan[ref].cost[k - 1]; }
    void make_plan() {
        plan.assign(tmp.size(), Plan{});
        // children have larger indices than their parent (build() pushes the parent first): a reverse sweep sees them first
        for (size_t n = tmp.size(); n-- > 0;) {
            const Bin& b = tmp[n];
            Plan& p = plan[n];
            float share[W + 1];      // share[k] = least cost of spreading n's two children over at most k >= 2 slots
            uint8_t share_left[W + 1];
            for (int k = 2; k <= W; ++k) {
                share[k] = 3.0e38f; share_left[k] = 1;
                for (int i = 1; i < k; ++i) {
                    float c = plan_cost(b.ref[0], i) + plan_cost(b.ref[1], k - i);
                    if (c < share[k]) { share[k] = c; share_left[k] = (uint8_t)i; }
                }
                if (k > 2 && share[k - 1] <= share[k]) { share[k] = share[k - 1]; share_left[k] = share_left[k - 1]; }
            }
            Aabb whole = b.box[0];
            grow(whole, b.box[1]);
            float self = entered(whole, merge_cones(b.cone[0], b.cone[1])) + share[W];
            if (!(self < 3.0e38f)) self = 3.0e38f;
            p.cost[0] = self; p.left[0] = 0;
            for (int k = 2; k <= W; ++k) {
                if (share[k] < self) { p.cost[k - 1] = share[k]; p.left[k - 1] = share_left[k]; }
                else { p.cost[k - 1] = self; p.left[k - 1] = 0; }
            }
        }
    }
    struct Slot { Aabb box; uint32_t ref; Cone cone; };
    // the slots the subtree under (box, ref, cone) occupies when it is given k of them
    void spread(const Slot& s, int k, std::vector<Slot>& slots) const {
        if ((s.ref & IREF_LEAF) || k == 1 || plan[s.ref].left[k - 1] == 0) { slots.push_back(s); return; }
        const Bin& b = tmp[s.ref];
        // find the k' <= k the plan actually used (share[k] may have been inherited from k - 1)
        int i = plan[s.ref].left[k - 1];
        int j = k - i;
        spread(Slot{b.box[0], b.ref[0], b.cone[0]}, i, slots);
        spread(Slot{b.box[1], b.ref[1], b.cone[1]}, j, slots);
    }

    // Emits the wide node of binary node `b` (and, recursively, of every slot that stays an inner node).
    uint32_t emit(uint32_t b, uint32_t depth) {
        wide_depth = std::max(wide_depth, depth);
        if (plan.empty()) make_plan();
        std::vector<Slot> slots;
        {
            // the node's own W slots: the best split between its two children
            const Bin& bn = tmp[b];
            int best_i = 1 | (1 << 4);
            float best = 3.0e38f;
            for (int k = 2; k <= W; ++k)
                for (int i = 1; i < k; ++i) {
                    float c = plan_cost(bn.ref[0], i) + plan_cost(bn.ref[1], k - i);
                    if (c < best) { best = c; best_i = i | ((k - i) << 4); }
                }
            spread(Slot{bn.box[0], bn.ref[0], bn.cone[0]}, best_i & 15, slots);
            spread(Slot{bn.box[1], bn.ref[1], bn.cone[1]}, best_i >> 4, slots);
        }
        uint32_t me = (uint32_t)(out.size() / kIndexNodeF4);
        out.resize(out.size() + kIndexNodeF4, f4{0, 0, 0, 0});
        bool any_cone = false;
        // one block of 4 children after the other (a node of width 8 is two blocks of the same layout)
        for (int blk = 0; blk < W / 4; ++blk) {
            uint16_t hv[6][4];
            uint16_t cv[4][4] = {{0, 0, 0, 0}, {0, 0, 0, 0}, {0, 0, 0, 0}, {0, 0, 0, 0}};  // axis x, y, z, threshold; all 0 = never culled
            uint32_t refs[4];
            for (int i = 0; i < 4; ++i) {
                const int si = 4 * blk + i;  // slot of the node = child i of block blk
                bool used = si < (int)slots.size();
                // unused slot: a far-away point box and the IREF_NONE marker
                Aabb bx = used ? slots[si].box : Aabb{{60000.f, 60000.f, 60000.f}, {60000.f, 60000.f, 60000.f}};
#if RTC_NODE_CENTRE_HALF
                // centre rounded to the nearest half, half-extent rounded UP so that [c - h, c + h] covers the box
                const float mn[3] = {bx.mn.x, bx.mn.y, bx.mn.z}, mx[3] = {bx.mx.x, bx.mx.y, bx.mx.z};
                for (int a = 0; a < 3; ++a) {
                    uint16_t c16 = half_bits_rn(0.5f * (mn[a] + mx[a]));
                    double c = (double)half_to_float(c16);
                    // + slack: the device evaluates fma(c, 1/d, -(o * 1/d)) -+ h |1/d|, whose rounding is a few ulp of
                    // |o / d| and |c / d|, i.e. a few 2^-24 of the scene size in world units; the child boxes must stay
                    // conservative even when a face is exactly representable in fp16 (no rounding margin of its own)
                    double need = std::max((double)mx[a] - c, c - (double)mn[a]) + slack;
                    float nf = (float)need;
                    if ((double)nf < need) nf = std::nextafter(nf, INFINITY);
                    hv[a][i] = c16;
                    hv[3 + a][i] = half_up(nf);
                    if ((c16 & 0x7C00u) == 0x7C00u || !(need <= 65504.0)) { hv[a][i] = 0; hv[3 + a][i] = 0x7C00u; }  // beyond fp16: always visited
                }
#else
                hv[0][i] = half_down(bx.mn.x); hv[1][i] = half_down(bx.mn.y); hv[2][i] = half_down(bx.mn.z);
                hv[3][i] = half_up(bx.mx.x); hv[4][i] = half_up(bx.mx.y); hv[5][i] = half_up(bx.mx.z);
#endif
                if (used && !slots[si].cone.open()) {
                    // The device culls the child when |dn . axis| < threshold, dn = normalised ray direction, all in
                    // half precision: the axis components round to nearest (error <= 8.7e-4 in the dot product), dn
                    // likewise, three half products / sums add <= 2.5e-3; the threshold gives 8e-3 away and is
                    // rounded down.  A threshold that ends up <= 0 leaves the child unrestricted.
                    const Cone& c = slots[si].cone;
                    const double thr = std::cos(std::min(c.alpha + 2e-3, 1.5707963)) - 8e-3;
                    if (thr > 0) {
                        cv[0][i] = half_bits_rn((float)c.ax); cv[1][i] = half_bits_rn((float)c.ay); cv[2][i] = half_bits_rn((float)c.az);
                        cv[3][i] = half_down((float)thr);
                        if (cv[3][i] & 0x8000u) cv[3][i] = 0;
                        if (cv[3][i] != 0) any_cone = true;
                    }
                }
                refs[i] = IREF_NONE;
                if (used) refs[i] = (slots[si].ref & IREF_LEAF) ? slots[si].ref : emit(slots[si].ref, depth + 1);
            }
            uint32_t w[16];
            for (int r = 0; r < 6; ++r) {
                w[2 * r] = (uint32_t)hv[r][0] | ((uint32_t)hv[r][1] << 16);
                w[2 * r + 1] = (uint32_t)hv[r][2] | ((uint32_t)hv[r][3] << 16);
            }
            for (int i = 0; i < 4; ++i) w[12 + i] = refs[i];
            for (int q = 0; q < 4; ++q) out[kIndexNodeF4 * me + kIndexBlockF4 * blk + q] = bits4(w[4 * q], w[4 * q + 1], w[4 * q + 2], w[4 * q + 3]);
#if RTC_NODE_CONES
            // q4 = axis.x[0..3] axis.y[0..3] ; q5 = axis.z[0..3] threshold[0..3]  (halves, two children per word)
            uint32_t cw[8];
            for (int r = 0; r < 4; ++r) {
                cw[2 * r] = (uint32_t)cv[r][0] | ((uint32_t)cv[r][1] << 16);
                cw[2 * r + 1] = (uint32_t)cv[r][2] | ((uint32_t)cv[r][3] << 16);
            }
            out[kIndexNodeF4 * me + kIndexBlockF4 * blk + 4] = bits4(cw[0], cw[1], cw[2], cw[3]);
            out[kIndexNodeF4 * me + kIndexBlockF4 * blk + 5] = bits4(cw[4], cw[5], cw[6], cw[7]);
#endif
        }
        return any_cone ? me : (me | IREF_NOCONE);
    }
};
}  // namespace

static f4 pack(vec3 v, uint32_t bits) {
    f4 r{v.x, v.y, v.z, 0.f};
    std::memcpy(&r.w, &bits, 4);
    return r;
}

namespace {
// RTC_TIMING=1: phase times of the host scene build on stderr
struct PhaseTimer {
    bool on = std::getenv("RTC_TIMING") != nullptr;
    std::chrono::steady_clock::time_point t0 = std::chrono::steady_clock::now();
    void lap(const char* what) {
        if (!on) return;
        auto t1 = std::chrono::steady_clock::now();
        std::fprintf(stderr, "[rtc timing] %-28s %8.1f ms\n", what, std::chrono::duration<double, std::milli>(t1 - t0).count());
        t0 = t1;
    }
};
}  // namespace

void HostScene::init() {
    PhaseTimer timer;
    const uint32_t n = (uint32_t)prims.size();
    if (n >= IREF_MAX_PRIMS) throw std::runtime_error("scene has more than 2^24 primitives");

    // ---- Scene::InitBVH (src/scene.cpp:16-21): non-planes first (std::partition order)
    std::vector<Primitive> original = prims;
    std::vector<int32_t> perm(n);
    std::iota(perm.begin(), perm.end(), 0);
    const Primitive* P = original.data();
    nbvh = (uint32_t)(std::partition(perm.begin(), perm.end(), [P](int32_t i) { return P[i].type != PT_PLANE; }) - perm.begin());

    nodes.clear();
    root = 0;
    if (nbvh > 0) {
        std::vector<Aabb> boxes(n, empty_box());
        for (uint32_t i = 0; i < n; ++i)
            if (original[i].type != PT_PLANE) boxes[i] = aabb_of_primitive(original[i]);
        nodes.reserve(2 * (size_t)nbvh);
        RefBuilder rb{perm, boxes, original, std::vector<float>((size_t)nbvh + 1, 0.f)};
        root = rb.build(nodes, 0, nbvh, build_parallel_levels());
    }
    for (uint32_t i = 0; i < n; ++i) prims[i] = original[perm[i]];
    timer.lap("reference BVH (RefBuilder)");

    // ---- Scene::InitDistribution (src/scene.cpp:27-40)
    lights.clear();
    for (uint32_t i = 0; i < n; ++i) {
        const Primitive& p = prims[i];
        if (!(p.emission.x > 0 || p.emission.y > 0 || p.emission.z > 0)) continue;
        if (p.type == PT_BOX || p.type == PT_ELLIPSOID) lights.push_back((int32_t)i);
    }

    // ---- flatten primitives
    FlatScene& F = flat;
    F = FlatScene();
    F.geo0.resize(n); F.geo1.resize(n); F.geo2.resize(n);
    F.xf_pos.resize(n); F.xf_rot.resize(n); F.mat0.resize(n); F.mat1.resize(n);
    for (uint32_t i = 0; i < n; ++i) {
        const Primitive& p = prims[i];
        uint32_t flags = (uint32_t)p.type & PF_TYPE_MASK;
        bool rot_ident = p.rot.x == 0.f && p.rot.y == 0.f && p.rot.z == 0.f && p.rot.w == 1.f;
        bool pos_zero = p.pos.x == 0.f && p.pos.y == 0.f && p.pos.z == 0.f;
        if (rot_ident) flags |= PF_ROT_IDENT;
        if (rot_ident && pos_zero) flags |= PF_IDENT;
        if (!rot_ident) F.features |= FE_ROTATION;
        if (p.type == PT_ELLIPSOID) F.features |= FE_ELLIPSOID;
        if (p.material != MAT_DIFFUSE) F.features |= FE_SPECULAR;
        if (p.type == PT_TRIANGLE) {
            // n = normalize(cross(b - a, c - a)), src/primitives.cpp:156 -- same float operations,
            // evaluated once here instead of once per intersection test
            vec3 nrm = normalize(cross(p.d1 - p.d0, p.d2 - p.d0));
            F.geo0[i] = f4{p.d0.x, p.d0.y, p.d0.z, nrm.x};
            F.geo1[i] = f4{p.d1.x, p.d1.y, p.d1.z, nrm.y};
            F.geo2[i] = f4{p.d2.x, p.d2.y, p.d2.z, nrm.z};
        } else {
            F.geo0[i] = f4{p.d0.x, p.d0.y, p.d0.z, 0.f};
            F.geo1[i] = f4{0, 0, 0, 0};
            F.geo2[i] = f4{0, 0, 0, 0};
        }
        F.xf_pos[i] = pack(p.pos, flags);
        F.xf_rot[i] = f4{p.rot.x, p.rot.y, p.rot.z, p.rot.w};
        F.mat0[i] = pack(p.col, (uint32_t)p.material);
        F.mat1[i] = f4{p.emission.x, p.emission.y, p.emission.z, p.ior};
    }
    F.lights = lights;
    for (const PointLight& l : point_lights) {  // hw2: DirectedLight keeps glm::normalize(dir), hw2 src/lights.cpp:20-23
        vec3 nd = l.directed ? normalize(l.dir) : mk3(0, 0, 0);
        F.plights.push_back(pack(l.intensity, l.directed ? 1u : 0u));
        F.plights.push_back(pack(l.pos, 0));
        F.plights.push_back(pack(l.att, 0));
        F.plights.push_back(pack(nd, 0));
    }
    for (uint32_t i = nbvh; i < n; ++i) {  // planes sit behind the BVH primitives (src/scene.cpp:17-19)
        const Primitive& p = prims[i];
        bool rot_ident = p.rot.x == 0.f && p.rot.y == 0.f && p.rot.z == 0.f && p.rot.w == 1.f;
        F.planes.push_back(pack(p.d0, i));
        F.planes.push_back(pack(p.pos, rot_ident ? 1u : 0u));
    }

    timer.lap("flatten primitives");
    // ---- reference tree: centre/half boxes (AABB_t::Intersect, src/bvh.cpp:89-93), depth, cuts
    const uint32_t nn = (uint32_t)nodes.size();
    F.rnodes.resize(2 * (size_t)nn);
    F.rmeta.resize(nn);
    std::vector<uint32_t> depth(nn, 0);
    std::vector<Unit> units;
    if (nn > 0) {
        std::vector<uint32_t> stack{root};
        while (!stack.empty()) {
            uint32_t v = stack.back();
            stack.pop_back();
            const RefNode& nd = nodes[v];
            vec3 half = 0.5f * (nd.box.mx - nd.box.mn);
            vec3 centre = 0.5f * (nd.box.mx + nd.box.mn);
            F.rnodes[2 * v] = pack(centre, nd.left);
            F.rnodes[2 * v + 1] = pack(half, nd.right);
            F.ref_depth = std::max(F.ref_depth, depth[v]);
            if (nd.left == UINT32_MAX) {
                F.rmeta[v] = u4{nd.first, nd.count, depth[v], 0};
                if (nd.count > IREF_MAX_LEAF_PRIMS) throw std::runtime_error("a BVH leaf holds more than 64 primitives");
                if (nd.count > 0) {
                    const Primitive& p0 = prims[nd.first];
                    bool ident = p0.rot.x == 0.f && p0.rot.y == 0.f && p0.rot.z == 0.f && p0.rot.w == 1.f &&
                                 p0.pos.x == 0.f && p0.pos.y == 0.f && p0.pos.z == 0.f;
                    bool fast = nd.count == 1 && p0.type == PT_TRIANGLE && ident;
                    units.push_back(Unit{nd.box, nd.first, nd.count, 0.5f * (nd.box.mx + nd.box.mn), fast,
                                         cone_of_leaf(prims, nd.first, nd.count, nd.box)});
                }
            } else {
                F.rmeta[v] = u4{nd.first, nodes[nd.right].first, depth[v], 0};
                depth[nd.left] = depth[nd.right] = depth[v] + 1;
                stack.push_back(nd.right);
                stack.push_back(nd.left);
            }
        }
    }
    std::sort(units.begin(), units.end(), [](const Unit& a, const Unit& b) { return a.first < b.first; });
    F.units = (uint32_t)units.size();
    F.ubox.assign(2 * (size_t)n, f4{0, 0, 0, 0});
    for (const Unit& u : units) {
        F.ubox[2 * (size_t)u.first] = f4{u.box.mn.x, u.box.mn.y, u.box.mn.z, 0.f};
        F.ubox[2 * (size_t)u.first + 1] = f4{u.box.mx.x, u.box.mx.y, u.box.mx.z, 0.f};
    }

    timer.lap("reference nodes, units, cones");
    // ---- index BVH
    F.inodes.clear();
    F.iroot = IREF_NONE;
    if (!units.empty()) {
        IndexBuilder ib{units, F.inodes, std::vector<float>(units.size() + 1, 0.f)};
        double extent = std::max({std::fabs((double)cam.pos.x), std::fabs((double)cam.pos.y), std::fabs((double)cam.pos.z)});
        for (const Unit& u : units)
            for (float v : {u.box.mn.x, u.box.mn.y, u.box.mn.z, u.box.mx.x, u.box.mx.y, u.box.mx.z})
                if (std::isfinite(v)) extent = std::max(extent, (double)std::fabs(v));
        ib.slack = extent * (1.0 / 1048576.0);
        ib.prepare();
        timer.lap("index BVH: presort");
        Cone whole;
        uint32_t broot = ib.build(ib.tmp, 0, (uint32_t)units.size(), 0, whole, build_parallel_levels());
        timer.lap("index BVH: sweep build");
        F.iroot = (broot & IREF_LEAF) ? broot : ib.emit(broot, 1);
        timer.lap("index BVH: collapse + emit");
        F.index_depth = ib.wide_depth;
    }

    // ---- LCA table: for a cut position c (boundary between primitive c-1 and c) the inner node
    // that splits there; range-min by depth over positions gives the lowest common ancestor of
    // two leaves.  lca[l * nbvh + c] = shallowest node among positions c .. c + 2^l - 1.
    F.lca.clear();
    F.lca_levels = 0;
    if (nbvh > 1) {
        uint32_t levels = 1;
        while ((1u << levels) < nbvh) ++levels;
        F.lca_levels = levels;
        F.lca.assign((size_t)levels * nbvh, UINT32_MAX);
        for (uint32_t v = 0; v < nn; ++v)
            if (nodes[v].left != UINT32_MAX) F.lca[F.rmeta[v].y] = v;
        auto dep = [&](uint32_t v) { return v == UINT32_MAX ? UINT32_MAX : depth[v]; };
        for (uint32_t l = 1; l < levels; ++l) {
            const uint32_t* prev = &F.lca[(size_t)(l - 1) * nbvh];
            uint32_t* cur = &F.lca[(size_t)l * nbvh];
            uint32_t half = 1u << (l - 1);
            for (uint32_t c = 0; c < nbvh; ++c) {
                uint32_t a = prev[c], b = (c + half < nbvh) ? prev[c + half] : UINT32_MAX;
                cur[c] = dep(b) < dep(a) ? b : a;
            }
        }
    }
    timer.lap("LCA table");
}

}  // namespace rtc
