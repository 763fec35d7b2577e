// rt_kernels.cu -- kernels of the wavefront integrator and the batch "probe" kernels behind
// rtc_intersect, rtc_mix_pdf, ... (sm_100a).
//
// One bounce of Scene::RayTrace =
//   pre_step    (fused into the kernel that creates the ray: k_generate, k_shade; k_pre for the probes) closest
//               plane + the root of the index BVH; rays that touch no root child are finished, the others are
//               queued (warp-aggregated atomics) together with the root children they enter, for
//   k_traverse  persistent warps that pull rays from that queue; every lane refills itself as soon as its ray is
//               done: all reference leaves a ray touches, then the replay of the reference recursion;
//   k_shade     recomputes the hit of the winning primitive (normal, interior), applies the material, writes
//               surviving paths compacted into the next queue.
#include <cassert>

#include "rt_device.cuh"
#include "rt_kernels.h"

namespace rtc {

static_assert(kNodeWidth == 4, "a traverse-queue entry carries the 4 root children a ray enters");
constexpr unsigned kFullMask = 0xFFFFFFFFu;
#ifndef RTC_TRAVERSE_CHUNK
#define RTC_TRAVERSE_CHUNK 64
#endif
#ifndef RTC_TRAVERSE_CHUNK_DIV
#define RTC_TRAVERSE_CHUNK_DIV 4
#endif
#ifndef RTC_TRAVERSE_CHUNK_MAX
#define RTC_TRAVERSE_CHUNK_MAX 512   // B200 sweep (full frame / share of one GPU of eight, Mpaths/s): fixed 32: 1969 / 1809, fixed 128: 1996 / 1819, fixed 512: 1983 / 1638, guided 32..256: 2007 / 1817, 64..256: 2008 / 1822, 64..512: 2011 / 1823
#endif
constexpr uint32_t kChunk = RTC_TRAVERSE_CHUNK;   // queue slots a warp reserves per atomic (at least)

// Wavefront state (paths, hits, queues) is written once and read once per bounce: 1.4 GB per k_shade launch
// streams through a 126 MB L2 that should keep the 34 MB of BVH nodes and triangles k_traverse gathers from.
// Every state access is marked evict-first (ld.global.cs / st.global.cs; +0.5 % measured, RTC_NO_STREAM_STATE
// restores plain accesses for A/B runs).
#ifndef RTC_NO_STREAM_STATE
#define WF_LD(ptr) __ldcs(ptr)
#define WF_ST(ptr, v) __stcs(ptr, v)
#else
#define WF_LD(ptr) (*(ptr))
#define WF_ST(ptr, v) (*(ptr) = (v))
#endif

// Planes (src/scene.cpp:50-66) and the root of the index BVH for one fresh ray: cd = closest_dist
// handed to BVH_t::Intersect, id = the plane hit so far; returns whether the ray touches any
// child box of the index root (only those rays are queued for k_traverse).
// Returns 0 when the ray touches no child box of the index root, else the mask of the root's children it enters
// (bit c = child c; a single-leaf tree reports bit 0): k_traverse starts from those children instead of visiting
// the root a second time.
template <uint32_t FEAT = FE_ALL>
RT_D uint32_t pre_step(const DevScene& S, vec3 o, vec3 d, float& cd, uint32_t& id) {
    int pid;
    closest_plane<FEAT>(S, o, d, cd, pid);
    id = pid < 0 ? HIT_MISS : (uint32_t)pid;
    if (S.iroot == IREF_NONE) return 0u;
    if (S.iroot & IREF_LEAF) {
        float te; bool interior; uint32_t l, r;
        return ref_box(S, S.root, o, d, te, interior, l, r) ? 1u : 0u;
    }
    vec3 inv = ray_inv(d);
    NodeVisit v = index_visit(S, S.iroot, inv, o * inv, cone_dir(d));
    uint32_t m = 0;
#pragma unroll
    for (uint32_t c = 0; c < kNodeWidth; ++c) m |= v.hit[c] ? (1u << c) : 0u;
    return m;
}
// Traverse-queue entry: the path slot in the low 28 bits (a batch holds at most 2^28 paths), the entered root
// children in the high 4.
constexpr uint32_t kTqSlotBits = 28;
constexpr uint32_t kTqSlotMask = (1u << kTqSlotBits) - 1u;
// warp-aggregated append of slot `i` to the traverse queue; call with the full warp converged
// one traverse-queue entry (rt_kernels.h kTraverseQueueWords)
RT_D void tq_store(uint32_t* tq, uint32_t at, uint32_t entry, vec3 o, vec3 d, float cd) {
    float4* rec = reinterpret_cast<float4*>(tq) + 2 * (size_t)at;
    WF_ST(rec, make_float4(o.x, o.y, o.z, __uint_as_float(entry)));
    WF_ST(rec + 1, make_float4(d.x, d.y, d.z, cd));
}
RT_D void enqueue(uint32_t rootmask, uint32_t i, vec3 o, vec3 d, float cd, uint32_t* tq, uint32_t* tq_count, uint32_t lane) {
    const bool enters = rootmask != 0;
    unsigned mask = __ballot_sync(kFullMask, enters);
    if (mask) {
        uint32_t base = 0;
        if (lane == 0) base = atomicAdd(tq_count, (uint32_t)__popc(mask));
        base = __shfl_sync(kFullMask, base, 0);
        const uint32_t entry = i | (rootmask << kTqSlotBits);
        if (enters) tq_store(tq, base + __popc(mask & ((1u << lane) - 1u)), entry, o, d, cd);
    }
}

// A path queue has two ends (round 2).  A surviving path is written to the FRONT when the mix distribution of its next
// shading will sample the cosine lobe, to the BACK (slots cap - 1, cap - 2, ...) when it will sample a light: the coin is
// a pure function of (seed, pixel, sample, bounce), so it can be tossed when the ray is made.  k_shade then walks the
// front and the back in whole warps, and a warp runs ONE of the two sampling codes instead of both with half its lanes
// masked (k_shade was bound by issue slots at 20 of 32 lanes).  q[0] = paths at the front, q[1] = paths at the back.
struct QueueView {
    uint32_t n_front, n_back, front_padded, total;   // total = both parts rounded up to whole warps
};
RT_D QueueView queue_view(const uint32_t* q) {
    QueueView v;
    v.n_front = q[0]; v.n_back = q[1];
    v.front_padded = (v.n_front + 31u) & ~31u;
    v.total = v.front_padded + ((v.n_back + 31u) & ~31u);
    return v;
}
// virtual index (thread's position in the walk) -> slot; returns false for the padding lanes
RT_D bool queue_slot(const QueueView& v, uint32_t at, uint32_t cap, uint32_t& slot, bool& back) {
    back = at >= v.front_padded;
    const uint32_t j = back ? at - v.front_padded : at;
    slot = back ? cap - 1u - j : j;
    return j < (back ? v.n_back : v.n_front);
}

// ------------------------------------------------------------------------------- generate
// Scene::Sample's jitter + Camera::GetToRay (src/scene.cpp:189-200) for the camera path of (pixel, sample), stored
// in slot i, and its pre_step; returns the root children the ray enters (o, d, cd: what the traverse queue takes).
RT_D uint32_t camera_path(const DevScene& S, PathSoA P, HitSoA H, uint32_t i, uint32_t pixel, uint32_t sample, uint32_t seed,
                          vec3& o, vec3& d, float& cd) {
    uint32_t x = pixel % S.width, y = pixel / S.width;
    Rng g{seed, pixel, sample, 0};
    uint4 b = g.block(0);
    float fx = __fadd_rn((float)x, u01(b.x)), fy = __fadd_rn((float)y, u01(b.y));
    // hw3's Camera::GetToRay(float, float) still adds the half pixel of its integer ancestor
    // (hw3 src/scene.cpp:186-187): its jittered samples cover [x + 0.5, x + 1.5)
    if (S.dialect == DIALECT_HW3) { fx = __fadd_rn(fx, 0.5f); fy = __fadd_rn(fy, 0.5f); }
    camera_ray(S, fx, fy, o, d);
    uint32_t id;
    const uint32_t enters = pre_step(S, o, d, cd, id);
    WF_ST(P.o + i, make_float4(o.x, o.y, o.z, __uint_as_float(sample)));
    WF_ST(P.d + i, make_float4(d.x, d.y, d.z, cd));
    WF_ST(P.beta + i, make_float4(1.f, 1.f, 1.f, __uint_as_float(pixel)));
    WF_ST(H.id + i, id);
    return enters;
}
// One thread per path.  Path ids run sample-major over the image: consecutive threads = consecutive pixels of a row.
__global__ void __launch_bounds__(256) k_generate(DevScene S, PathSoA P, HitSoA H, uint32_t* q, uint32_t* tq, uint32_t* tq_count,
                                                   uint64_t first_path, uint32_t count, uint32_t seed, uint32_t sample_begin) {
    const uint32_t npix = S.width * S.height;
    const uint32_t lane = threadIdx.x & 31;
    const uint32_t rounded = (count + 31u) & ~31u;
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < rounded; i += gridDim.x * blockDim.x) {
        uint32_t enters = 0;
        vec3 o = mk3(0, 0, 0), d = mk3(0, 0, 0);
        float cd = 0.f;
        if (i < count) {
            uint64_t pid = first_path + i;
            uint32_t sample = sample_begin + (uint32_t)(pid / npix);
            uint32_t pixel = (uint32_t)(pid % npix);
            enters = camera_path(S, P, H, i, pixel, sample, seed, o, d, cd);
        }
        enqueue(enters, i, o, d, cd, tq, tq_count, lane);
    }
    if (blockIdx.x == 0 && threadIdx.x == 0) q[0] = count;
}
// The same over a pixel list (adaptive sampling): path id p is pixel plist[p % npix] and sample sample_first +
// 2 (p / npix) -- every other sample, so that one call renders the even or the odd samples of a range.
__global__ void __launch_bounds__(256) k_generate_list(DevScene S, PathSoA P, HitSoA H, uint32_t* q, uint32_t* tq, uint32_t* tq_count,
                                                        uint64_t first_path, uint32_t count, uint32_t seed, const uint32_t* plist,
                                                        uint32_t npix, uint32_t sample_first) {
    const uint32_t lane = threadIdx.x & 31;
    const uint32_t rounded = (count + 31u) & ~31u;
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < rounded; i += gridDim.x * blockDim.x) {
        uint32_t enters = 0;
        vec3 o = mk3(0, 0, 0), d = mk3(0, 0, 0);
        float cd = 0.f;
        if (i < count) {
            uint64_t pid = first_path + i;
            uint32_t sample = sample_first + 2u * (uint32_t)(pid / npix);
            uint32_t pixel = plist[pid % npix];
            enters = camera_path(S, P, H, i, pixel, sample, seed, o, d, cd);
        }
        enqueue(enters, i, o, d, cd, tq, tq_count, lane);
    }
    if (blockIdx.x == 0 && threadIdx.x == 0) q[0] = count;
}

// ------------------------------------------------------------------------------- extend, step 1
// pre_step as a kernel of its own: only the probe path (rtc_intersect) needs it -- in a render the
// step is fused into the kernel that creates the ray (k_generate, k_shade).
__global__ void __launch_bounds__(256) k_pre(DevScene S, PathSoA P, HitSoA H, const uint32_t* qcount, uint32_t* tq,
                                              uint32_t* tq_count) {
    const uint32_t count = *qcount;
    const uint32_t lane = threadIdx.x & 31;
    const uint32_t rounded = (count + 31u) & ~31u;
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < rounded; i += gridDim.x * blockDim.x) {
        uint32_t enters = 0;
        vec3 o = mk3(0, 0, 0), d = mk3(0, 0, 0);
        float cd = 0.f;
        if (i < count) {
            uint32_t id;
            const float4 d4 = WF_LD(P.d + i);
            o = ld3(WF_LD(P.o + i)); d = ld3(d4);
            enters = pre_step(S, o, d, cd, id);
            WF_ST(P.d + i, make_float4(d4.x, d4.y, d4.z, cd));
            WF_ST(H.id + i, id);
        }
        enqueue(enters, i, o, d, cd, tq, tq_count, lane);
    }
}

// ------------------------------------------------------------------------------- extend, step 2
// BVH_t::Intersect (src/bvh.cpp:181-225) for the queued rays: index-BVH traversal collecting the
// reference leaves with a hit, then the replay of the reference recursion (rt_device.cuh).
//
// Persistent warps with a per-warp task scheduler.  The traversal reports ALL touched leaves in
// any order, so the three kinds of work of a ray are decoupled: VISIT one inner node (children
// that are leaves are only noted down), test one noted LEAF, FINISH the ray (replay + store);
// idle lanes REFILL from the queue (FINISH and REFILL share an iteration: a lane that stores its result takes its
// next ray at once).  Every iteration the warp votes and executes the kind most
// lanes are ready for, which keeps lanes busy although rays need between one and several
// hundred node visits.  `cursor` hands out queue slots, kChunk per atomic.
// (The traversal stack of a lane in shared memory, word w of thread t at [w][t], was measured slower than local memory:
// profiles/r02_experiments.md.)
// FINISH and REFILL as one kind of scheduler work: measured on B200 11.52 -> 10.90 ms (the two used to cost a vote and a
// partly filled warp iteration each: 5.3 M + 5.4 M iterations per frame at 15.7 / 17.7 lanes)
constexpr int kStackWords = 56;  // per lane: inner-node stack from the bottom, noted leaves from the top
#define STK(i) stk[i]
constexpr uint32_t kNone = 0xFFFFFFFFu;
#ifndef RTC_LEAF_FIRST
#define RTC_LEAF_FIRST 8
#endif
#ifndef RTC_VISIT_QUORUM
#define RTC_VISIT_QUORUM 16   // sweep on B200 with cone nodes: 10: 20.2, 12: 19.7, 14: 19.3, 16: 19.05 ms/step (64-byte nodes: 14 was best)
#endif
constexpr int kVisitQuorum = RTC_VISIT_QUORUM;

#ifndef RTC_TRAVERSE_MIN_BLOCKS
#define RTC_TRAVERSE_MIN_BLOCKS 7   // 72 registers; 5 / 6 / 8 blocks (84 / 79 / 64 registers): 12.96 / 11.73 / 12.75 ms against 11.56
#endif
template <bool STATS>
__global__ void __launch_bounds__(128, RTC_TRAVERSE_MIN_BLOCKS) k_traverse(DevScene S, PathSoA P, HitSoA H, const uint32_t* tq, const uint32_t* tq_count,
                                                   uint32_t* cursor, unsigned long long* stats) {
    const uint32_t total = *tq_count;
    const uint32_t lane = threadIdx.x & 31;
    const uint32_t lt_mask = (1u << lane) - 1u;
    uint32_t pool_base = 0, pool_left = 0;  // warp-uniform
    bool exhausted = false;                 // warp-uniform: the queue has no more slots for this warp
    bool active = false, overflow = false;
    uint32_t ray = 0, node = kNone;
    vec3 o = mk3(0, 0, 0), d = mk3(0, 0, 0), inv = mk3(0, 0, 0), oi = mk3(0, 0, 0);
    ConeDir dn{0u, 0u};
    float cd0 = 0.f;
    int sp = 0, nl = 0, k = 0;
    uint32_t stk[kStackWords];
    LeafRec rec[kMaxRecords];
    uint32_t visits = 0, tests = 0, fallbacks = 0;
    uint32_t iters[4] = {0, 0, 0, 0}, busy[4] = {0, 0, 0, 0};  // STATS: warp iterations and participating lanes per kind

    enum { kVisit, kLeaf, kFinish, kRefill };
    for (;;) {
        const bool room = sp + nl + (2 * (int)kNodeWidth - 1) <= kStackWords;  // a visit notes up to W leaves and pushes up to W - 1 nodes
        const bool canV = active && node != kNone && room;
        const unsigned mV = __ballot_sync(kFullMask, canV);
        const int nV = __popc(mV);
        int kind = kVisit;
        bool canL = false, canF = false, canR = false;
        unsigned mR = 0;
        int nR = 0;
        if (nV < kVisitQuorum) {  // full vote only when visiting would leave too many lanes idle
            // a lane whose stack is full of inner nodes (no noted leaf to free room) gives up and takes the
            // reference walk in FINISH; checked here only: such a lane is not in mV, so the vote comes
            if (active && node != kNone && !room && nl == 0) { overflow = true; node = kNone; sp = 0; }
            canL = active && nl > 0;
            canF = active && node == kNone && nl == 0;
            canR = !active && (pool_left > 0 || !exhausted);
            const unsigned mL = __ballot_sync(kFullMask, canL), mF = __ballot_sync(kFullMask, canF);
            mR = __ballot_sync(kFullMask, canR);
            if (!(mV | mL | mF | mR)) break;
            const int nL = __popc(mL), nF = __popc(mF);
            nR = __popc(mR);
            // lanes holding noted leaves are served before the plain majority vote once there are enough
            // of them (threshold swept on B200: profiles/r01_experiments.md)
            // FINISH and REFILL are one kind of work: a lane whose ray is done stores its result and takes the next ray in
            // the same iteration (kind kFinish stands for both)
            const int nT = __popc(mF | mR);
            if (nL >= RTC_LEAF_FIRST) kind = kLeaf;
            else if (nV >= nL && nV >= nT) kind = kVisit;
            else if (nL >= nT) kind = kLeaf;
            else kind = kFinish;
        }

        if (STATS) {  // warp-execution efficiency of the scheduler: lanes that take part in this iteration
            const bool part = kind == kVisit ? canV : kind == kLeaf ? canL : kind == kFinish ? canF : canR;
            const int n = __popc(__ballot_sync(kFullMask, part));
#pragma unroll
            for (int q = 0; q < 4; ++q) if (kind == q) { iters[q] += 1; busy[q] += (uint32_t)n; }
        }
        if (kind == kVisit) {
            // ---- VISIT: one inner node per ready lane; leaf children are only noted
            if (canV) {
                if (STATS) ++visits;
                NodeVisit v = index_visit(S, node, inv, oi, dn);
                const int spm = sp > 0 ? sp - 1 : 0;
                const uint32_t top = STK(spm);
                uint32_t next = kNone;
#pragma unroll
                for (int c = 0; c < (int)kNodeWidth; ++c) {
                    const bool leaf = (v.ref[c] & IREF_LEAF) != 0;
                    if (v.hit[c] && leaf) {  // note the leaf, test it later
                        ++nl;
                        STK(kStackWords - nl) = v.ref[c];
                    }
                    const bool inner = v.hit[c] && !leaf;
                    if (inner && next != kNone) { STK(sp) = v.ref[c]; ++sp; }
                    next = (inner && next == kNone) ? v.ref[c] : next;
                }
                const bool pop = next == kNone && sp > 0;
                node = pop ? top : next;
                sp = pop ? spm : sp;
            }
        } else if (kind == kLeaf) {
            // ---- LEAF: one noted reference leaf per ready lane
            if (canL) {
                const uint32_t ref = STK(kStackWords - nl);
                --nl;
                float bt, tc; int bid;
                if (leaf_test(S, ref, o, d, inv, oi, bt, bid, tc, STATS ? &tests : nullptr) && bid >= 0) {
                    if (k == kMaxRecords) { overflow = true; node = kNone; sp = 0; nl = 0; }
                    else { rec[k].key = ref & 0xFFFFFFu; rec[k].id = bid; rec[k].t = bt; rec[k].tcull = tc; ++k; }
                }
            }
        } else {
          if (kind == kFinish) {   // (always: FINISH and REFILL are one kind of scheduler work, the vote never picks kRefill)
            // ---- FINISH: replay of the reference recursion, store the winner
            if (canF) {
                BestHit b;
                if (overflow) { b = trace_reftree(S, o, d, cd0); ++fallbacks; }
                else b = replay_reference(S, o, d, cd0, rec, k);
                if (b.id != -1 && b.t < cd0) WF_ST(H.id + ray, (uint32_t)b.id);  // src/scene.cpp:68-74
                active = false;
            }
            canR = !active && (pool_left > 0 || !exhausted);
            mR = __ballot_sync(kFullMask, canR);
            nR = __popc(mR);
            if (STATS) { iters[kRefill] += 1; busy[kRefill] += (uint32_t)nR; }
          }
            // ---- REFILL idle lanes from the queue (the lanes that just finished among them)
            if (pool_left == 0) {
                uint32_t base = 0;
#if RTC_TRAVERSE_CHUNK_MAX > RTC_TRAVERSE_CHUNK
                // guided chunks: large while much of the queue is left (fewer atomic round trips: 10.89 -> 10.76 ms at 128
                // slots per atomic), down to kChunk towards its end (a warp that sits on many unserved slots while the
                // others run dry lengthens the tail of the launch: 512 slots cost 40 % at the share of one GPU of eight).
                // `pool_base` is where this warp's last chunk ended: a slightly stale view of the cursor, good enough here.
                const uint32_t left = total > pool_base ? total - pool_base : 0u;
                const uint32_t take = min(max(left / ((uint32_t)RTC_TRAVERSE_CHUNK_DIV * gridDim.x * (blockDim.x / 32u)), kChunk), (uint32_t)RTC_TRAVERSE_CHUNK_MAX);
#else
                const uint32_t take = kChunk;
#endif
                if (lane == 0) base = atomicAdd(cursor, take);
                base = __shfl_sync(kFullMask, base, 0);
                if (base >= total) exhausted = true;
                else { pool_base = base; pool_left = min(take, total - base); }
            }
            uint32_t rank = __popc(mR & lt_mask);
            uint32_t serve = min((uint32_t)nR, pool_left);
            if (canR && rank < serve) {
                // the entry IS the ray: one coalesced round trip (consecutive ranks read consecutive 32-byte records)
                const float4* rec32 = reinterpret_cast<const float4*>(tq) + 2 * (size_t)(pool_base + rank);
                const float4 o4 = WF_LD(rec32), d4 = WF_LD(rec32 + 1);
                const uint32_t entry = __float_as_uint(o4.w);
                ray = entry & kTqSlotMask;
                o = ld3(o4);
                d = ld3(d4);
                cd0 = d4.w;
                inv = ray_inv(d);
                oi = o * inv;
                dn = cone_dir(d);
                sp = 0; nl = 0; k = 0; overflow = false;
                active = true;
                node = kNone;
                if (S.iroot & IREF_LEAF) {  // single-leaf tree
                    nl = 1;
                    STK(kStackWords - 1) = S.iroot;
                } else {
                    // the root was visited when the ray was made (pre_step): start from the children it entered.
                    // (Measured on B200: 6.56 instead of 7.56 visits per ray and the same 11.65 ms -- the root visit of
                    // freshly loaded lanes shares its warp iteration and its cache line with everybody else's.)
#pragma unroll
                    for (int c = 0; c < 4; ++c) {
                        const uint32_t ref = S.iroot_ref[c];
                        if (!((entry >> (kTqSlotBits + c)) & 1u)) continue;
                        if (ref & IREF_LEAF) { ++nl; STK(kStackWords - nl) = ref; }
                        else if (node == kNone) node = ref;
                        else { STK(sp) = ref; ++sp; }
                    }
                }
            }
            pool_base += serve;
            pool_left -= serve;
        }
    }
    if (fallbacks) atomicAdd(stats + 5, (unsigned long long)fallbacks);
    if (STATS) {
        if (visits) atomicAdd(stats + 4, (unsigned long long)visits);
        if (tests) atomicAdd(stats + 6, (unsigned long long)tests);
        if (lane == 0) {
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                atomicAdd(stats + 8 + q, (unsigned long long)iters[q]);
                atomicAdd(stats + 12 + q, (unsigned long long)busy[q]);
            }
        }
    }
}

// The node-by-node twin (RTC_TRAVERSAL_REFTREE): planes + the reference's own tree, one thread per ray.
__global__ void __launch_bounds__(128) k_extend_reftree(DevScene S, PathSoA P, HitSoA H, const uint32_t* q, uint32_t cap) {
    const QueueView view = queue_view(q);
    for (uint32_t at = blockIdx.x * blockDim.x + threadIdx.x; at < view.total; at += gridDim.x * blockDim.x) {
        uint32_t i; bool back;
        if (!queue_slot(view, at, cap, i, back)) continue;
        vec3 o = ld3(WF_LD(P.o + i)), d = ld3(WF_LD(P.d + i));
        float closest;
        int id;
        closest_plane(S, o, d, closest, id);
        BestHit b = trace_reftree(S, o, d, closest);
        if (b.id != -1 && b.t < closest) id = b.id;
        WF_ST(H.id + i, id < 0 ? HIT_MISS : (uint32_t)id);
    }
}

// ------------------------------------------------------------------------------- shade
// beta * emission of one hit into the pixel sum: ONE 16-byte reduction (REDG.E.ADD.F32x4) on the library's own
// float4-per-pixel buffer, folded into the caller's 3-float buffer when the frame's batches are done (k_fold).
RT_D void deposit(float4* accum4, uint32_t pixel, vec3 L) {
#ifdef __CUDA_ARCH__
    asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(accum4 + pixel), "f"(L.x), "f"(L.y), "f"(L.z), "f"(0.f) : "memory");
#endif
}

// Scene::RayTrace's material switch (src/scene.cpp:96-177) for one bounce, recursion unrolled:
// L = sum_k beta_k * E_k.  Surviving paths are written compacted (warp ballot + one atomic per
// warp) into the next queue; every hit adds its beta * emission to the pixel sum at once (deposit).
#ifndef RTC_SHADE_THREADS
#define RTC_SHADE_THREADS 128
#endif
// blocks per SM: the full kernel runs best at 6 (80 registers, 40 B spilled); the instantiations without rotation and
// ellipsoid code fit 64 registers without spilling and gain from 8 (shade 8.3 -> 7.5 ms; 9 / 10 / 12 blocks spill and
// lose again): profiles/r01_experiments.md
#ifndef RTC_SHADE_MIN_BLOCKS_FULL
#define RTC_SHADE_MIN_BLOCKS_FULL 6
#endif
#ifndef RTC_SHADE_MIN_BLOCKS_LEAN
#define RTC_SHADE_MIN_BLOCKS_LEAN 9   // round 2 (52-byte state, two-ended queues): 7 / 8 / 9 blocks: 7.17 / 6.74 / 6.62 ms
#endif
// HW3 = the hw3 snapshot's diffuse term (hw3 src/scene.cpp:238-249): a direction uniform on the hemisphere
// around the normal, weight 2 C cos; every other line of the switch is common to hw3, hw4 and hw5.
// FEAT = the scene features this instantiation supports (rt_device.cuh prim_flags_for): the kernel is bound by
// instruction fetch, and the course's dragon scenes use a third of its code (no rotation, no ellipsoid, diffuse).
template <bool HW3, uint32_t FEAT>
__global__ void __launch_bounds__(RTC_SHADE_THREADS, (FEAT & (FE_ROTATION | FE_ELLIPSOID)) ? RTC_SHADE_MIN_BLOCKS_FULL : RTC_SHADE_MIN_BLOCKS_LEAN) k_shade(DevScene S, PathSoA P, HitSoA H, PathSoA N, HitSoA HN, const uint32_t* qin,
                                                uint32_t* qout, uint32_t* tq, uint32_t* tq_count, float4* accum4, uint32_t bounce,
                                                uint32_t seed, uint32_t cap) {
    const QueueView view = queue_view(qin);
    const uint32_t lane = threadIdx.x & 31;
    const float eps = S.eps;
    // camera paths (bounce 1) arrive unsorted; from then on the end of the queue a path sits at tells its coin
    const bool sorted_in = bounce > 1 && !HW3;
    // the paths written here are shaded with sampling at bounce + 1 only if that is below RAY_DEPTH
    const bool sort_out = !HW3 && S.nlights != 0 && bounce + 1 < S.ray_depth;
    for (uint32_t at = blockIdx.x * blockDim.x + threadIdx.x; at < view.total; at += gridDim.x * blockDim.x) {
        bool alive = false;
        vec3 no = mk3(0, 0, 0), nd = mk3(0, 0, 0), beta = mk3(0, 0, 0);
        uint32_t pixel = 0, sample = 0;
        uint32_t i; bool back;
        if (queue_slot(view, at, cap, i, back)) {
            const float4 b4 = WF_LD(P.beta + i), o4 = WF_LD(P.o + i);
            beta = ld3(b4);
            pixel = __float_as_uint(b4.w); sample = __float_as_uint(o4.w);
            uint32_t prim = WF_LD(H.id + i);
            Isect is;
            vec3 o = ld3(o4), d = ld3(WF_LD(P.d + i));
            vec3 L;   // what this hit adds to the pixel: beta * (background | emission)
            // every row of the winner at once (one round trip instead of flags -> position -> geometry -> material)
            float4 xp = make_float4(0.f, 0.f, 0.f, 0.f), g0 = xp, g1 = xp, g2 = xp, m0 = xp, m1 = xp;
            if (prim != HIT_MISS) {
                xp = ldg4(S.xf_pos + prim); g0 = ldg4(S.geo0 + prim); g1 = ldg4(S.geo1 + prim); g2 = ldg4(S.geo2 + prim);
                m0 = ldg4(S.mat0 + prim); m1 = ldg4(S.mat1 + prim);
            }
            if (prim == HIT_MISS || !prim_intersect_rows<false, FEAT, true>(S, prim, xp, g0, g1, g2, o, d, is)) {  // exact t, rsqrt normal
                L = beta * mk3(S.bg.x, S.bg.y, S.bg.z);  // src/scene.cpp:92-94
            } else {
                bool interior = is.interior != 0;
                vec3 normal = is.n;
                vec3 p = o + is.t * d;
                vec3 col = ld3(m0);
                L = beta * ld3(m1);
                uint32_t material = __float_as_uint(m0.w);
                if (bounce < S.ray_depth) {
                    Rng g{seed, pixel, sample, bounce};
                    if (HW3 && material == MAT_DIFFUSE) {
                        vec3 dir = normal_vec(g.block(1));
                        float cs = dot(dir, normal);
                        if (cs < 0.f) { dir = -dir; cs = -cs; }
                        beta = beta * mk3(col.x * (2.f * cs), col.y * (2.f * cs), col.z * (2.f * cs));
                        no = p + eps * dir; nd = dir;
                        alive = true;
                    } else if (material == MAT_DIFFUSE) {
                        vec3 p_outer = p + eps * normal;
                        vec3 dir = mix_sample<FEAT>(S, g, p_outer, normal, sorted_in ? (back ? 1 : 0) : -1);
                        float cs = dot(dir, normal);
                        if (cs > 0.f) {
                            float pw = mix_pdf<FEAT>(S, p_outer, normal, dir);
                            const float inv_pi = 1.f / kPi;
                            vec3 w = mk3(col.x * inv_pi, col.y * inv_pi, col.z * inv_pi);
                            float k2 = __fdividef(1.f, pw);
                            beta = beta * mk3(w.x * cs * k2, w.y * cs * k2, w.z * cs * k2);
                            no = p + eps * dir; nd = dir;
                            alive = true;
                        }
                    } else if (!(FEAT & FE_SPECULAR)) {
                        // unreachable: the host launches this instantiation only for all-diffuse scenes
                    } else if (material == MAT_METALLIC) {
                        vec3 rd = reflect_dir(normal, normalize(d));
                        beta = beta * col;
                        no = p + eps * rd; nd = rd;
                        alive = true;
                    } else {  // DIELECTRIC, src/scene.cpp:130-170
                        float eta1 = 1.f, eta2 = m1.w;
                        if (interior) { float tmp = eta1; eta1 = eta2; eta2 = tmp; }
                        vec3 nd_in = normalize(d);
                        vec3 dir = -nd_in;
                        float dn = dot(normal, dir);
                        float sin2 = eta1 / eta2 * sqrtf(fmaxf(0.f, 1.f - dn * dn));
                        bool reflect = fabsf(sin2) > 1.f;
                        if (!reflect) {
                            float q0 = (eta1 - eta2) / (eta1 + eta2);
                            float r0 = q0 * q0;
                            float m = 1.f - dn;
                            float m2 = m * m;
                            float r = r0 + (1.f - r0) * (m2 * m2 * m);
                            reflect = u01(g.block(0).x) < r;
                        }
                        if (reflect) {
                            vec3 rd = reflect_dir(normal, nd_in);
                            no = p + eps * rd; nd = rd;
                        } else {
                            float cos2 = sqrtf(1.f - sin2 * sin2);
                            float e = eta1 / eta2;
                            vec3 fr = e * (-dir) + (e * dn - cos2) * normal;
                            no = p + eps * fr; nd = fr;
                            if (!interior) beta = beta * col;
                        }
                        alive = true;
                    }
                }
            }
            if (L.x != 0.f || L.y != 0.f || L.z != 0.f) deposit(accum4, pixel, L);
        }
        unsigned mask = __ballot_sync(kFullMask, alive);
        if (mask) {
            // Both queue reservations are in flight while the next ray's pre_step is computed: the results of the two
            // atomics are first needed by the stores at the very end (12 % of the kernel's stall samples sat on them
            // when each was awaited where it was issued).
            const uint32_t lt = (1u << lane) - 1u;
            // which end of the next queue: the coin of the NEXT shading (slot bounce + 1), tossed now
            bool to_back = false;
            if (sort_out && alive) to_back = mix_picks_light(S, Rng{seed, pixel, sample, bounce + 1});
            const unsigned bmask = __ballot_sync(kFullMask, to_back), fmask = mask & ~bmask;
            unsigned long long both = 0;   // one 64-bit reservation: front count in the low word, back count in the high word
            uint32_t tbase = 0;
            if (lane == 0) both = atomicAdd(reinterpret_cast<unsigned long long*>(qout),
                                            (unsigned long long)__popc(fmask) | ((unsigned long long)__popc(bmask) << 32));
            // first part of the next Scene::RayIntersection, while the ray is still in registers
            float cd = 0.f;
            uint32_t id = HIT_MISS, enters = 0;
            if (alive) enters = pre_step<FEAT>(S, no, nd, cd, id);
            const unsigned emask = __ballot_sync(kFullMask, enters != 0);
            if (emask && lane == 0) tbase = atomicAdd(tq_count, (uint32_t)__popc(emask));
            both = __shfl_sync(kFullMask, both, 0);
            const uint32_t dst = to_back ? cap - 1u - ((uint32_t)(both >> 32) + __popc(bmask & lt))
                                         : (uint32_t)both + __popc(fmask & lt);
            if (alive) {
                WF_ST(N.o + dst, make_float4(no.x, no.y, no.z, __uint_as_float(sample)));
                WF_ST(N.d + dst, make_float4(nd.x, nd.y, nd.z, cd));
                WF_ST(N.beta + dst, make_float4(beta.x, beta.y, beta.z, __uint_as_float(pixel)));
                WF_ST(HN.id + dst, id);
            }
            if (emask) {
                tbase = __shfl_sync(kFullMask, tbase, 0);
                if (enters) tq_store(tq, tbase + __popc(emask & lt), dst | (enters << kTqSlotBits), no, nd, cd);
            }
        }
    }
}

// totals: stats[0] += paths, stats[1] += rays, stats[3] += 1 batch, stats[7] += rays sent to k_traverse
__global__ void k_tally(const uint32_t* q, const uint32_t* tqc, uint32_t ray_depth, unsigned long long* stats) {
    unsigned long long rays = 0, queued = 0;
    for (uint32_t b = 0; b < ray_depth; ++b) { rays += q[2 * b] + q[2 * b + 1]; queued += tqc[b]; }
    // one k_tally per batch on each lane's own stream: two of them may run at the same time
    atomicAdd(stats + 0, (unsigned long long)q[0]);
    atomicAdd(stats + 1, rays);
    atomicAdd(stats + 3, 1ull);
    atomicAdd(stats + 7, queued);
}

// Scene::Render's per-pixel tail (src/scene.cpp:201, 227-228, 247): mean, AcesTonemap,
// GammaCorrected, Color::toUInts (src/color.cpp:26-49)
RT_D float aces(float x) {
    const float a = 2.51f, b = 0.03f, c = 2.43f, d = 0.59f, e = 0.14f;
    float num = __fmul_rn(x, __fadd_rn(__fmul_rn(a, x), b));
    float den = __fadd_rn(__fmul_rn(x, __fadd_rn(__fmul_rn(c, x), d)), e);
    float y = __fdiv_rn(num, den);
    y = (y < 1.f) ? y : 1.f;   // std::min(1.f, y): NaN -> 1
    y = (y < 0.f) ? 0.f : y;   // std::max(y, 0.f)
    return y;
}
RT_D unsigned char to_u8(float y) {
    float g = powf(y, 0.454545468f);  // (float)(1. / 2.2)
    return (unsigned char)(int)roundf(__fmul_rn(255.f, g));
}
// the frame's float4 pixel sums into the caller's 3-floats-per-pixel buffer (rtc_render_accumulate ADDS)
__global__ void __launch_bounds__(256) k_fold(const float4* accum4, float* accum, uint32_t npix) {
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < npix; i += gridDim.x * blockDim.x) {
        const float4 v = accum4[i];
        accum[3 * (size_t)i + 0] += v.x;
        accum[3 * (size_t)i + 1] += v.y;
        accum[3 * (size_t)i + 2] += v.z;
    }
}
__global__ void __launch_bounds__(256) k_resolve(const float* accum, float inv_samples, uint32_t nvalues, uint8_t* out) {
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < nvalues; i += gridDim.x * blockDim.x)
        out[i] = to_u8(aces(__fmul_rn(inv_samples, accum[i])));
}
// Multi-device Scene::Render, last step on the first device: the per-device pixel sums (each device rendered its share
// of the samples) are read where they lie -- peer pointers over NVLink -- summed in device order, and resolved to
// 8 bits in the same pass (src/scene.cpp:201, 227-228, 247); `sum` (optional) keeps the float total.
__global__ void __launch_bounds__(256) k_resolve_peers(PeerAccums A, float inv_samples, uint32_t nvalues, uint8_t* out, float* sum) {
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < nvalues; i += gridDim.x * blockDim.x) {
        float v = A.p[0][i];
        for (int r = 1; r < A.n; ++r) v += A.p[r][i];
        if (sum) sum[i] = v;
        out[i] = to_u8(aces(__fmul_rn(inv_samples, v)));
    }
}
__global__ void __launch_bounds__(256) k_tonemap(const float* rgb, uint32_t nvalues, uint8_t* out) {
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < nvalues; i += gridDim.x * blockDim.x)
        out[i] = to_u8(aces(rgb[i]));
}

// ------------------------------------------------------------------------------- adaptive sampling (rtc_render_adaptive)
// The display value to_u8 rounds, taken before rounding
RT_D float display(float v) { return powf(aces(v), 0.454545468f); }
// e_p of one pixel: the mean over r, g, b of |D(mean of the even samples) - D(mean of the odd samples)|
RT_D float half_error(float4 A, float4 B, float inv_a, float inv_b) {
    const float er = fabsf(display(__fmul_rn(A.x, inv_a)) - display(__fmul_rn(B.x, inv_b)));
    const float eg = fabsf(display(__fmul_rn(A.y, inv_a)) - display(__fmul_rn(B.y, inv_b)));
    const float eb = fabsf(display(__fmul_rn(A.z, inv_a)) - display(__fmul_rn(B.z, inv_b)));
    return __fdiv_rn(__fadd_rn(__fadd_rn(er, eg), eb), 3.f);
}
// One warp per active tile; pixel k of the tile (row-major within the tile) is on lane k % 32, so a lane holds
// pixels (x, y) and (x, y + 4).  ADAPTIVE_FIRST lists every tile of a shard (tiles_in unused), ADAPTIVE_DECIDE computes
// the tile error E from the half sums (n samples: inv_a = 1 / ceil(n/2), inv_b = 1 / floor(n/2)) and keeps the tile
// while !(E < tau), ADAPTIVE_LAST keeps none.  Every visited tile records n; a kept tile is appended to tiles_out and
// its in-image pixels, row by row, to pixels_out (counts_out[0] tiles, counts_out[1] pixels; one atomic per warp).
// ADAPTIVE_FIRST lists the ntiles tiles of one shard of the frame: the w-th is tile shard + w nshards (the whole frame
// is shard 0 of 1; a multi-device render gives device d of D the shard (d, D)).
__global__ void __launch_bounds__(128) k_adaptive_tiles(const float4* A, const float4* B, uint32_t width, uint32_t height,
                                                         const uint32_t* tiles_in, uint32_t ntiles, uint32_t n, float inv_a,
                                                         float inv_b, float tau, int mode, uint32_t* tile_n, uint32_t* tiles_out,
                                                         uint32_t* pixels_out, uint32_t* counts_out, uint32_t shard,
                                                         uint32_t nshards) {
    const uint32_t lane = threadIdx.x & 31;
    const uint32_t tiles_x = (width + kAdaptiveTile - 1) / kAdaptiveTile;
    const uint32_t warps = (gridDim.x * blockDim.x) >> 5;
    for (uint32_t w = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; w < ntiles; w += warps) {   // warp-uniform
        const uint32_t tile = mode == ADAPTIVE_FIRST ? shard + w * nshards : tiles_in[w];
        const uint32_t x = (tile % tiles_x) * kAdaptiveTile + (lane & 7u), y0 = (tile / tiles_x) * kAdaptiveTile + (lane >> 3);
        const bool v0 = x < width && y0 < height, v1 = x < width && y0 + 4u < height;
        const uint32_t p0 = y0 * width + x, p1 = p0 + 4u * width;
        const unsigned m0 = __ballot_sync(kFullMask, v0), m1 = __ballot_sync(kFullMask, v1);
        bool keep = mode != ADAPTIVE_LAST;
        if (mode == ADAPTIVE_DECIDE) {
            float e = 0.f;
            if (v0) e = half_error(A[p0], B[p0], inv_a, inv_b);
            if (v1) e = __fadd_rn(e, half_error(A[p1], B[p1], inv_a, inv_b));
#pragma unroll
            for (int off = 16; off > 0; off >>= 1) e = __fadd_rn(e, __shfl_xor_sync(kFullMask, e, off));
            const float E = __fdiv_rn(e, (float)(__popc(m0) + __popc(m1)));
            keep = !(E < tau);   // a NaN error keeps the tile
        }
        if (lane == 0) tile_n[tile] = n;
        if (keep) {
            uint32_t tbase = 0, pbase = 0;
            if (lane == 0) {
                tbase = atomicAdd(counts_out, 1u);
                pbase = atomicAdd(counts_out + 1, (uint32_t)(__popc(m0) + __popc(m1)));
                tiles_out[tbase] = tile;
            }
            pbase = __shfl_sync(kFullMask, pbase, 0);
            const unsigned lt = (1u << lane) - 1u;
            if (v0) pixels_out[pbase + __popc(m0 & lt)] = p0;
            if (v1) pixels_out[pbase + __popc(m0) + __popc(m1 & lt)] = p1;
        }
    }
}
// The tile (row-major over the frame) of pixel i
RT_D uint32_t tile_of(uint32_t i, uint32_t width, uint32_t tiles_x) {
    return (i / width / kAdaptiveTile) * tiles_x + (i % width) / kAdaptiveTile;
}
// Pixel i of an adaptive image: it took n samples, a / b are its even / odd sums; out = to_u8(aces(1/n * (a + b)))
// (k_resolve's expression); optionally halves (a.rgb, b.rgb per pixel) and spp (n).
RT_D void resolve_adaptive_pixel(uint32_t i, float4 a, float4 b, uint32_t n, uint8_t* out, float* halves, uint32_t* spp) {
    const float inv = __fdiv_rn(1.f, (float)n);
    out[3 * (size_t)i + 0] = to_u8(aces(__fmul_rn(inv, __fadd_rn(a.x, b.x))));
    out[3 * (size_t)i + 1] = to_u8(aces(__fmul_rn(inv, __fadd_rn(a.y, b.y))));
    out[3 * (size_t)i + 2] = to_u8(aces(__fmul_rn(inv, __fadd_rn(a.z, b.z))));
    if (halves) {
        float* h = halves + 6 * (size_t)i;
        h[0] = a.x; h[1] = a.y; h[2] = a.z; h[3] = b.x; h[4] = b.y; h[5] = b.z;
    }
    if (spp) spp[i] = n;
}
// The image of an adaptive render: pixel i took tile_n[its tile] samples, A / B hold its even / odd sums
__global__ void __launch_bounds__(256) k_resolve_adaptive(const float4* A, const float4* B, const uint32_t* tile_n, uint32_t width,
                                                           uint32_t npix, uint8_t* out, float* halves, uint32_t* spp) {
    const uint32_t tiles_x = (width + kAdaptiveTile - 1) / kAdaptiveTile;
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < npix; i += gridDim.x * blockDim.x)
        resolve_adaptive_pixel(i, A[i], B[i], tile_n[tile_of(i, width, tiles_x)], out, halves, spp);
}
// The same for a multi-device adaptive render, on the first device: tile t was rendered by device t % P.n, whose
// half sums and tile counts are read where they lie (peer pointers over NVLink, or copies on this device)
__global__ void __launch_bounds__(256) k_resolve_adaptive_peers(PeerHalves P, uint32_t width, uint32_t npix, uint8_t* out,
                                                                 float* halves, uint32_t* spp) {
    const uint32_t tiles_x = (width + kAdaptiveTile - 1) / kAdaptiveTile;
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < npix; i += gridDim.x * blockDim.x) {
        const uint32_t t = tile_of(i, width, tiles_x), d = t % (uint32_t)P.n;
        resolve_adaptive_pixel(i, P.a[d][i], P.b[d][i], P.tile_n[d][t], out, halves, spp);
    }
}

// ------------------------------------------------------------------------------- denoising (rtc_denoise, rtc_render_denoised)
// Non-local means on the even / odd half sums (Rousselle, Knaus and Zwicker 2012; DESIGN.md "Denoising").  Per pixel
// with n >= 2 samples: u = 1/n (A + B) (resolve_adaptive_pixel's floats), D = display(u) and, per channel, the variance
// estimate V = ((display(A / ceil(n/2)) - display(B / floor(n/2))) / 2)^2 (k_adaptive_tiles' half means).  rgb, when
// given (the filter is not run), gets resolve_adaptive_pixel's image of u.  One pixel: a / b its even / odd sums, the
// outputs point at its own u (3 floats), D, V and rgb (3 bytes, or null).
RT_D void denoise_prep_pixel(const float a[3], const float b[3], uint32_t n, float* u, float4* D, float4* V, uint8_t* rgb) {
    const float inv = __fdiv_rn(1.f, (float)n), inv_a = __fdiv_rn(1.f, (float)((n + 1) / 2)), inv_b = __fdiv_rn(1.f, (float)(n / 2));
    float uc[3], dc[3], vc[3];
#pragma unroll
    for (int c = 0; c < 3; ++c) {
        uc[c] = __fmul_rn(inv, __fadd_rn(a[c], b[c]));
        dc[c] = display(uc[c]);
        const float e = __fmul_rn(__fsub_rn(display(__fmul_rn(a[c], inv_a)), display(__fmul_rn(b[c], inv_b))), 0.5f);
        vc[c] = __fmul_rn(e, e);
        u[c] = uc[c];
        if (rgb) rgb[c] = to_u8(aces(uc[c]));
    }
    *D = make_float4(dc[0], dc[1], dc[2], 0.f);
    *V = make_float4(vc[0], vc[1], vc[2], 0.f);
}
__global__ void __launch_bounds__(256) k_denoise_prep(const float* halves, const uint32_t* spp, uint32_t npix, float* u, float4* D,
                                                       float4* V, uint8_t* rgb) {
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < npix; i += gridDim.x * blockDim.x) {
        const float* h = halves + 6 * (size_t)i;
        const float a[3] = {h[0], h[1], h[2]}, b[3] = {h[3], h[4], h[5]};
        denoise_prep_pixel(a, b, spp[i], u + 3 * (size_t)i, D + i, V + i, rgb ? rgb + 3 * (size_t)i : nullptr);
    }
}
// The same for the rows [row0, row0 + npix / width) of a multi-device adaptive render, straight from the owners' half sums
// (k_resolve_adaptive_peers' ownership: tile t is device t % P.n's).  P.a / P.b point at those rows' first pixel, P.tile_n
// at whole tile-count arrays; u, D and V are band-local.  rgb, when given, gets the image of the pixels
// [rgb_first, rgb_first + rgb_count) of the band.
__global__ void __launch_bounds__(256) k_denoise_prep_peers(PeerHalves P, uint32_t width, uint32_t row0, uint32_t npix, float* u,
                                                             float4* D, float4* V, uint8_t* rgb, uint32_t rgb_first, uint32_t rgb_count) {
    const uint32_t tiles_x = (width + kAdaptiveTile - 1) / kAdaptiveTile;
    for (uint32_t j = blockIdx.x * blockDim.x + threadIdx.x; j < npix; j += gridDim.x * blockDim.x) {
        const uint32_t t = tile_of(row0 * width + j, width, tiles_x), d = t % (uint32_t)P.n;
        const float4 fa = P.a[d][j], fb = P.b[d][j];
        const float a[3] = {fa.x, fa.y, fa.z}, b[3] = {fb.x, fb.y, fb.z};
        const bool out = rgb && j - rgb_first < rgb_count;
        denoise_prep_pixel(a, b, P.tile_n[d][t], u + 3 * (size_t)j, D + j, V + j, out ? rgb + 3 * (size_t)(j - rgb_first) : nullptr);
    }
}
// One block filters a kDenoiseTileW x kDenoiseTileH tile of pixels.  It stages D and the smoothed V (the mean of V over
// the (2S+1)^2 box around the pixel) of the tile and its apron of R + F (coordinates clamped to the image: patches repeat
// the edge pixels) and u of the tile and its apron of R (NaN
// outside the image, so that such neighbours fail the finiteness test), then walks the (2R+1)^2 offsets: per offset
// the distance term of every pixel of the tile plus F, a row box sum of width 2F+1, and per pixel the column box sum,
// the weight and the weighted sums in registers.  Two barriers per offset; each thread owns two pixels of a column.
// The grid covers the tile rows [tile_row0, tile_row0 + gridDim.y) (a band of a multi-device filter; the whole frame is
// (0, 0)); u, D and V hold the image rows [buf_row0, min(H, band end + kDenoiseApron)), mean and rgb the band's rows.
constexpr int kDnR = kDenoiseRadius, kDnF = kDenoisePatch, kDnS = kDenoiseVarRadius, kDnA = kDnR + kDnF;
static_assert(kDenoiseApron == kDnA + kDnS, "k_denoise_nlm: the rows a block reads beyond its tile");
constexpr int kDnTW = kDenoiseTileW, kDnTH = kDenoiseTileH, kDnThreads = 256, kDnRows = kDnThreads / kDnTW;
constexpr int kDnSW = kDnTW + 2 * kDnA, kDnSH = kDnTH + 2 * kDnA;   // D, V staging
constexpr int kDnUW = kDnTW + 2 * kDnR, kDnUH = kDnTH + 2 * kDnR;   // u staging
constexpr int kDnEW = kDnTW + 2 * kDnF, kDnEH = kDnTH + 2 * kDnF;   // distance terms of one offset
constexpr int kDnPix = kDnTH / kDnRows;                              // pixels per thread
static_assert(kDnTW == 32 && kDnTH % kDnRows == 0, "k_denoise_nlm: a warp per tile row");
constexpr size_t kDenoiseSmemFloats = 6 * (size_t)kDnSW * kDnSH + 3 * (size_t)kDnUW * kDnUH + kDnEW * kDnEH + kDnTW * kDnEH;
__global__ void __launch_bounds__(kDnThreads) k_denoise_nlm(const float* u, const float4* D, const float4* V, uint32_t width,
                                                             uint32_t height, uint32_t tile_row0, uint32_t buf_row0, float k2,
                                                             float* mean, uint8_t* rgb) {
    extern __shared__ float smem[];
    float* sD = smem;                              // [3][kDnSH][kDnSW]
    float* sV = sD + 3 * kDnSW * kDnSH;            // [3][kDnSH][kDnSW]
    float* sU = sV + 3 * kDnSW * kDnSH;            // [3][kDnUH][kDnUW]
    float* sT = sU + 3 * kDnUW * kDnUH;            // [kDnEH][kDnEW]
    float* sH = sT + kDnEW * kDnEH;                // [kDnEH][kDnTW]
    const int x0 = blockIdx.x * kDnTW, y0 = (tile_row0 + blockIdx.y) * kDnTH, W = (int)width, H = (int)height;
    const int band0 = tile_row0 * kDnTH, r0 = (int)buf_row0;
    // the rows read below: D and the centres of V's boxes within A of the tile, V's boxes S further, u within R
    assert(max(y0 - kDnA - kDnS, 0) >= r0 &&
           min(y0 + kDnTH + kDnA + kDnS, H) <= min(min((int)(tile_row0 + gridDim.y) * kDnTH, H) + kDenoiseApron, H));
    for (int i = threadIdx.x; i < kDnSW * kDnSH; i += kDnThreads) {
        const int gx = min(max(x0 - kDnA + i % kDnSW, 0), W - 1), gy = min(max(y0 - kDnA + i / kDnSW, 0), H - 1);
        const float4 d = D[(size_t)(gy - r0) * W + gx];
        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);   // V smoothed over the (2S+1)^2 box around (gx, gy), clamped
        for (int oy = -kDnS; oy <= kDnS; ++oy)
            for (int ox = -kDnS; ox <= kDnS; ++ox) {
                const float4 t = V[(size_t)(min(max(gy + oy, 0), H - 1) - r0) * W + min(max(gx + ox, 0), W - 1)];
                v.x += t.x; v.y += t.y; v.z += t.z;
            }
        constexpr float inv_box = 1.f / ((2 * kDnS + 1) * (2 * kDnS + 1));
        v.x *= inv_box; v.y *= inv_box; v.z *= inv_box;
        sD[i] = d.x; sD[i + kDnSW * kDnSH] = d.y; sD[i + 2 * kDnSW * kDnSH] = d.z;
        sV[i] = v.x; sV[i + kDnSW * kDnSH] = v.y; sV[i + 2 * kDnSW * kDnSH] = v.z;
    }
    for (int i = threadIdx.x; i < kDnUW * kDnUH; i += kDnThreads) {
        const int gx = x0 - kDnR + i % kDnUW, gy = y0 - kDnR + i / kDnUW;
        const bool in = gx >= 0 && gx < W && gy >= 0 && gy < H;
#pragma unroll
        for (int c = 0; c < 3; ++c) sU[i + c * kDnUW * kDnUH] = in ? u[3 * ((size_t)(gy - r0) * W + gx) + c] : __int_as_float(0x7fc00000);
    }
    __syncthreads();
    const int tx = threadIdx.x % kDnTW, ty = threadIdx.x / kDnTW;
    float sw[kDnPix], su[kDnPix][3];
#pragma unroll
    for (int j = 0; j < kDnPix; ++j) sw[j] = su[j][0] = su[j][1] = su[j][2] = 0.f;
    const float inv_patch = 1.f / (3.f * (2 * kDnF + 1) * (2 * kDnF + 1));
    for (int dy = -kDnR; dy <= kDnR; ++dy) {
        for (int dx = -kDnR; dx <= kDnR; ++dx) {
            // distance term of extended pixel e (the tile plus F): p + o at staging (ey + R, ex + R), q + o shifted by (dy, dx)
            for (int e = threadIdx.x; e < kDnEW * kDnEH; e += kDnThreads) {
                const int ip = (e / kDnEW + kDnR) * kDnSW + e % kDnEW + kDnR, iq = ip + dy * kDnSW + dx;
                float t = 0.f;
#pragma unroll
                for (int c = 0; c < 3; ++c) {
                    const float dp = sD[ip + c * kDnSW * kDnSH], dq = sD[iq + c * kDnSW * kDnSH];
                    const float vp = sV[ip + c * kDnSW * kDnSH], vq = sV[iq + c * kDnSW * kDnSH];
                    const float num = (dp - dq) * (dp - dq) - kDenoiseAlpha * (vp + fminf(vp, vq));
                    t += __fdividef(num, kDenoiseEps + k2 * (vp + vq));
                }
                sT[e] = t;
            }
            __syncthreads();
            for (int e = threadIdx.x; e < kDnTW * kDnEH; e += kDnThreads) {
                const float* row = sT + (e / kDnTW) * kDnEW + e % kDnTW;
                float s = 0.f;
#pragma unroll
                for (int o = 0; o <= 2 * kDnF; ++o) s += row[o];
                sH[e] = s;
            }
            __syncthreads();
#pragma unroll
            for (int j = 0; j < kDnPix; ++j) {
                const int ly = ty + j * kDnRows;
                float s = 0.f;
#pragma unroll
                for (int o = 0; o <= 2 * kDnF; ++o) s += sH[(ly + o) * kDnTW + tx];
                const int iq = (ly + kDnR + dy) * kDnUW + tx + kDnR + dx;
                const float qr = sU[iq], qg = sU[iq + kDnUW * kDnUH], qb = sU[iq + 2 * kDnUW * kDnUH];
                if (isfinite(qr) && isfinite(qg) && isfinite(qb)) {
                    const float w = __expf(-fmaxf(0.f, s * inv_patch));
                    sw[j] += w;
                    su[j][0] += w * qr; su[j][1] += w * qg; su[j][2] += w * qb;
                }
            }
        }
    }
#pragma unroll
    for (int j = 0; j < kDnPix; ++j) {
        const int x = x0 + tx, y = y0 + ty + j * kDnRows;
        if (x >= W || y >= H) continue;
        const int ip = (ty + j * kDnRows + kDnR) * kDnUW + tx + kDnR;
        float up[3] = {sU[ip], sU[ip + kDnUW * kDnUH], sU[ip + 2 * kDnUW * kDnUH]};
        const bool finite = isfinite(up[0]) && isfinite(up[1]) && isfinite(up[2]);   // else it passes through
        const size_t i = (size_t)(y - band0) * W + x;
#pragma unroll
        for (int c = 0; c < 3; ++c) {
            const float v = finite ? __fdiv_rn(su[j][c], sw[j]) : up[c];
            mean[3 * i + c] = v;
            rgb[3 * i + c] = to_u8(aces(v));
        }
    }
}

// ------------------------------------------------------------------------------- scene arena, device-built tail
// Levels >= 1 of the LCA range-minimum table (bvh_build.cpp: lca[l][c] = the shallower of lca[l-1][c] and
// lca[l-1][c + 2^(l-1)]) from level 0, which is uploaded; one launch per level.
__global__ void __launch_bounds__(256) k_expand_lca_level(const uint32_t* prev, uint32_t* cur, const uint4* rmeta, uint32_t n, uint32_t half) {
    for (uint32_t c = blockIdx.x * blockDim.x + threadIdx.x; c < n; c += gridDim.x * blockDim.x) {
        const uint32_t a = prev[c], b = (c + half < n) ? prev[c + half] : 0xFFFFFFFFu;
        const uint32_t da = a == 0xFFFFFFFFu ? 0xFFFFFFFFu : rmeta[a].z, db = b == 0xFFFFFFFFu ? 0xFFFFFFFFu : rmeta[b].z;
        cur[c] = db < da ? b : a;
    }
}
// exact boxes of the leaves that have one: (slot, min, max) triples scattered into the (zeroed) per-slot array
__global__ void __launch_bounds__(256) k_expand_boxes(const float4* sparse, uint32_t n, float4* ubox) {
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const uint32_t slot = __float_as_uint(sparse[3 * i].x);
        ubox[2 * (size_t)slot] = sparse[3 * i + 1];
        ubox[2 * (size_t)slot + 1] = sparse[3 * i + 2];
    }
}
// per-primitive rows (position | flags, or the two material rows) from the palette of distinct rows that was uploaded
__global__ void __launch_bounds__(256) k_expand_palette(const float4* palette, const uint16_t* index, uint32_t n, float4* out0, float4* out1) {
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const uint32_t row = index[i];
        if (out1) { out0[i] = palette[2 * row]; out1[i] = palette[2 * row + 1]; }
        else out0[i] = palette[row];
    }
}
__global__ void __launch_bounds__(256) k_fill_identity_rotations(float4* rot, uint32_t n) {
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) rot[i] = make_float4(0.f, 0.f, 0.f, 1.f);
}

// ------------------------------------------------------------------------------- probes
// rtc_intersect: rays given as 3 floats each -> the float4 queue layout of the render path, and
// back from primitive ids to (t, normal, interior) by re-intersecting the winner.
__global__ void k_pack_rays(long n, const float* o, const float* d, PathSoA P, uint32_t* q) {
    for (long i = blockIdx.x * (long)blockDim.x + threadIdx.x; i < n; i += (long)gridDim.x * blockDim.x) {
        P.o[i] = make_float4(o[3 * i], o[3 * i + 1], o[3 * i + 2], 0.f);
        P.d[i] = make_float4(d[3 * i], d[3 * i + 1], d[3 * i + 2], 0.f);
    }
    if (blockIdx.x == 0 && threadIdx.x == 0) q[0] = (uint32_t)n;
}
__global__ void k_unpack_hits(DevScene S, long n, PathSoA P, HitSoA H, int32_t* id, float* t, float* nrm, int32_t* interior) {
    for (long i = blockIdx.x * (long)blockDim.x + threadIdx.x; i < n; i += (long)gridDim.x * blockDim.x) {
        uint32_t prim = H.id[i];
        Isect is;
        is.t = 0.f; is.n = mk3(0, 0, 0); is.interior = 0;
        bool ok = prim != HIT_MISS && prim_intersect(S, prim, ld3(P.o[i]), ld3(P.d[i]), is);
        id[i] = ok ? (int32_t)prim : -1;
        t[i] = ok ? is.t : 0.f;
        nrm[3 * i] = ok ? is.n.x : 0.f; nrm[3 * i + 1] = ok ? is.n.y : 0.f; nrm[3 * i + 2] = ok ? is.n.z : 0.f;
        interior[i] = ok ? is.interior : 0;
    }
}
__global__ void k_primitive_batch(DevScene S, uint32_t prim, long n, const float* o, const float* d, int32_t* hit, float* t,
                                  float* nrm, int32_t* interior) {
    for (long i = blockIdx.x * (long)blockDim.x + threadIdx.x; i < n; i += (long)gridDim.x * blockDim.x) {
        vec3 ro = mk3(o[3 * i], o[3 * i + 1], o[3 * i + 2]), rd = mk3(d[3 * i], d[3 * i + 1], d[3 * i + 2]);
        Isect is;
        bool ok = prim_intersect(S, prim, ro, rd, is);
        hit[i] = ok;
        t[i] = ok ? is.t : 0.f;
        nrm[3 * i] = ok ? is.n.x : 0.f; nrm[3 * i + 1] = ok ? is.n.y : 0.f; nrm[3 * i + 2] = ok ? is.n.z : 0.f;
        interior[i] = ok ? is.interior : 0;
    }
}
__global__ void k_camera_batch(DevScene S, long n, const float* xy, float* o, float* d) {
    for (long i = blockIdx.x * (long)blockDim.x + threadIdx.x; i < n; i += (long)gridDim.x * blockDim.x) {
        vec3 ro, rd;
        camera_ray(S, xy[2 * i], xy[2 * i + 1], ro, rd);
        o[3 * i] = ro.x; o[3 * i + 1] = ro.y; o[3 * i + 2] = ro.z;
        d[3 * i] = rd.x; d[3 * i + 1] = rd.y; d[3 * i + 2] = rd.z;
    }
}
__global__ void k_pdf_batch(DevScene S, long n, const float* x, const float* nr, const float* d, float* pdf) {
    for (long i = blockIdx.x * (long)blockDim.x + threadIdx.x; i < n; i += (long)gridDim.x * blockDim.x)
        pdf[i] = mix_pdf(S, mk3(x[3 * i], x[3 * i + 1], x[3 * i + 2]), mk3(nr[3 * i], nr[3 * i + 1], nr[3 * i + 2]),
                         mk3(d[3 * i], d[3 * i + 1], d[3 * i + 2]));
}
__global__ void k_sample_batch(DevScene S, long n, const float* x, const float* nr, uint32_t seed, uint32_t sample,
                               uint32_t bounce, float* dir) {
    for (long i = blockIdx.x * (long)blockDim.x + threadIdx.x; i < n; i += (long)gridDim.x * blockDim.x) {
        Rng g{seed, (uint32_t)i, sample, bounce};
        vec3 r = mix_sample(S, g, mk3(x[3 * i], x[3 * i + 1], x[3 * i + 2]), mk3(nr[3 * i], nr[3 * i + 1], nr[3 * i + 2]));
        dir[3 * i] = r.x; dir[3 * i + 1] = r.y; dir[3 * i + 2] = r.z;
    }
}

// ------------------------------------------------------------------------------- launchers
static int grid_for(uint64_t n, int block, int sms, int per_sm) {
    uint64_t want = (n + block - 1) / block;
    uint64_t cap = (uint64_t)sms * per_sm;
    if (want < 1) want = 1;
    return (int)(want < cap ? want : cap);
}

void launch_generate(const LaunchCtx& c, const DevScene& S, PathSoA P, HitSoA H, uint32_t* q, uint32_t* tq, uint32_t* tq_count,
                     uint64_t first_path, uint32_t count, uint32_t seed, uint32_t sample_begin) {
    k_generate<<<grid_for(count, 256, c.sms, 8), 256, 0, c.stream>>>(S, P, H, q, tq, tq_count, first_path, count, seed, sample_begin);
}
void launch_generate_list(const LaunchCtx& c, const DevScene& S, PathSoA P, HitSoA H, uint32_t* q, uint32_t* tq, uint32_t* tq_count,
                          uint64_t first_path, uint32_t count, uint32_t seed, const uint32_t* plist, uint32_t npix, uint32_t sample_first) {
    k_generate_list<<<grid_for(count, 256, c.sms, 8), 256, 0, c.stream>>>(S, P, H, q, tq, tq_count, first_path, count, seed, plist,
                                                                          npix, sample_first);
}
void launch_adaptive_tiles(const LaunchCtx& c, const float4* A, const float4* B, uint32_t width, uint32_t height,
                           const uint32_t* tiles_in, uint32_t ntiles, uint32_t n, float inv_a, float inv_b, float tau, int mode,
                           uint32_t* tile_n, uint32_t* tiles_out, uint32_t* pixels_out, uint32_t* counts_out, uint32_t shard,
                           uint32_t nshards) {
    if (ntiles == 0) return;
    k_adaptive_tiles<<<grid_for((uint64_t)ntiles * 32, 128, c.sms, 16), 128, 0, c.stream>>>(A, B, width, height, tiles_in, ntiles, n, inv_a,
                                                                                          inv_b, tau, mode, tile_n, tiles_out,
                                                                                          pixels_out, counts_out, shard, nshards);
}
void launch_resolve_adaptive(const LaunchCtx& c, const float4* A, const float4* B, const uint32_t* tile_n, uint32_t width, uint32_t npix,
                             uint8_t* out, float* halves, uint32_t* spp) {
    k_resolve_adaptive<<<grid_for(npix, 256, c.sms, 8), 256, 0, c.stream>>>(A, B, tile_n, width, npix, out, halves, spp);
}
void launch_resolve_adaptive_peers(const LaunchCtx& c, const PeerHalves& P, uint32_t width, uint32_t npix, uint8_t* out, float* halves,
                                   uint32_t* spp) {
    k_resolve_adaptive_peers<<<grid_for(npix, 256, c.sms, 8), 256, 0, c.stream>>>(P, width, npix, out, halves, spp);
}
void launch_denoise_prep(const LaunchCtx& c, const float* halves, const uint32_t* spp, uint32_t npix, float* u, float4* D, float4* V,
                         uint8_t* rgb) {
    k_denoise_prep<<<grid_for(npix, 256, c.sms, 8), 256, 0, c.stream>>>(halves, spp, npix, u, D, V, rgb);
}
void launch_denoise_prep_peers(const LaunchCtx& c, const PeerHalves& P, uint32_t width, uint32_t row0, uint32_t nrows, float* u,
                               float4* D, float4* V, uint8_t* rgb, uint32_t rgb_first, uint32_t rgb_count) {
    const uint32_t npix = width * nrows;
    k_denoise_prep_peers<<<grid_for(npix, 256, c.sms, 8), 256, 0, c.stream>>>(P, width, row0, npix, u, D, V, rgb, rgb_first, rgb_count);
}
cudaError_t launch_denoise_nlm(const LaunchCtx& c, const float* u, const float4* D, const float4* V, uint32_t width, uint32_t height,
                               uint32_t tile_row0, uint32_t tile_rows, uint32_t buf_row0, float k2, float* mean, uint8_t* rgb) {
    const size_t bytes = kDenoiseSmemFloats * sizeof(float);
    cudaError_t e = cudaFuncSetAttribute(k_denoise_nlm, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
    if (e != cudaSuccess) return e;
    const dim3 grid((width + kDnTW - 1) / kDnTW, tile_rows);
    k_denoise_nlm<<<grid, kDnThreads, bytes, c.stream>>>(u, D, V, width, height, tile_row0, buf_row0, k2, mean, rgb);
    return cudaGetLastError();
}
void launch_pre(const LaunchCtx& c, const DevScene& S, PathSoA P, HitSoA H, const uint32_t* qcount, uint32_t max_count,
                uint32_t* tq, uint32_t* tq_count) {
    k_pre<<<grid_for(max_count, 256, c.sms, 8), 256, 0, c.stream>>>(S, P, H, qcount, tq, tq_count);
}
// blocks of 128 threads one SM holds of a persistent kernel, cached per device
template <class K>
static int resident_blocks(K kernel, int slot) {
    static int cache[4][64];
    int dev = 0;
    cudaGetDevice(&dev);
    if (dev < 0 || dev >= 64) dev = 0;
    if (cache[slot][dev] == 0) {
        int n = 0;
        cudaError_t e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&n, kernel, 128, 0);
        cache[slot][dev] = (e == cudaSuccess && n > 0) ? n : 4;
    }
    return cache[slot][dev];
}
void launch_traverse(const LaunchCtx& c, const DevScene& S, PathSoA P, HitSoA H, uint32_t max_count, const uint32_t* tq,
                     const uint32_t* tq_count, uint32_t* cursor, bool count_visits, unsigned long long* stats) {
    // persistent: exactly one resident wave of 128-thread blocks
    const int per_sm = count_visits ? resident_blocks(k_traverse<true>, 1) : resident_blocks(k_traverse<false>, 0);
    int grid = grid_for((uint64_t)max_count, 128, c.sms, per_sm);
    if (count_visits) k_traverse<true><<<grid, 128, 0, c.stream>>>(S, P, H, tq, tq_count, cursor, stats);
    else k_traverse<false><<<grid, 128, 0, c.stream>>>(S, P, H, tq, tq_count, cursor, stats);
}
void launch_extend_reftree(const LaunchCtx& c, const DevScene& S, PathSoA P, HitSoA H, const uint32_t* q, uint32_t cap) {
    k_extend_reftree<<<grid_for(cap, 128, c.sms, 16), 128, 0, c.stream>>>(S, P, H, q, cap);
}
void launch_shade(const LaunchCtx& c, const DevScene& S, PathSoA P, HitSoA H, PathSoA N, HitSoA HN, const uint32_t* qin,
                  uint32_t* qout, uint32_t* tq, uint32_t* tq_count, uint32_t max_count, float4* accum4, uint32_t bounce,
                  uint32_t seed) {
    const int grid = grid_for(max_count, RTC_SHADE_THREADS, c.sms, 2048 / RTC_SHADE_THREADS);
#define RTC_SHADE(HW3, FEAT) k_shade<HW3, FEAT><<<grid, RTC_SHADE_THREADS, 0, c.stream>>>(S, P, H, N, HN, qin, qout, tq, tq_count, accum4, bounce, seed, max_count)
    // the smallest instantiation that covers the scene's features (DevScene::features)
#ifdef RTC_SHADE_NO_SPECIALISATION
    const uint32_t feat = FE_ALL;
#else
    const uint32_t feat = S.features;
#endif
    if (S.dialect == DIALECT_HW3) RTC_SHADE(true, FE_ALL);
    else if (feat == 0) RTC_SHADE(false, 0);
    else if (feat == FE_SPECULAR) RTC_SHADE(false, FE_SPECULAR);
    else RTC_SHADE(false, FE_ALL);
#undef RTC_SHADE
}
void launch_expand_lca(const LaunchCtx& c, uint32_t* lca, const uint4* rmeta, uint32_t n, uint32_t levels) {
    for (uint32_t l = 1; l < levels; ++l)
        k_expand_lca_level<<<grid_for(n, 256, c.sms, 8), 256, 0, c.stream>>>(lca + (size_t)(l - 1) * n, lca + (size_t)l * n, rmeta, n, 1u << (l - 1));
}
void launch_expand_boxes(const LaunchCtx& c, const float4* sparse, uint32_t n, float4* ubox) {
    k_expand_boxes<<<grid_for(n, 256, c.sms, 8), 256, 0, c.stream>>>(sparse, n, ubox);
}
void launch_expand_palette(const LaunchCtx& c, const float4* palette, const uint16_t* index, uint32_t n, float4* out0, float4* out1) {
    k_expand_palette<<<grid_for(n, 256, c.sms, 8), 256, 0, c.stream>>>(palette, index, n, out0, out1);
}
void launch_fill_identity_rotations(const LaunchCtx& c, float4* rot, uint32_t n) {
    k_fill_identity_rotations<<<grid_for(n, 256, c.sms, 8), 256, 0, c.stream>>>(rot, n);
}
void launch_tally(const LaunchCtx& c, const uint32_t* q, const uint32_t* tqc, uint32_t ray_depth, unsigned long long* stats) {
    k_tally<<<1, 1, 0, c.stream>>>(q, tqc, ray_depth, stats);
}
void launch_fold(const LaunchCtx& c, const float4* accum4, float* accum, uint32_t npix) {
    k_fold<<<grid_for(npix, 256, c.sms, 8), 256, 0, c.stream>>>(accum4, accum, npix);
}
void launch_resolve(const LaunchCtx& c, const float* accum, float inv_samples, uint32_t nvalues, uint8_t* out) {
    k_resolve<<<grid_for(nvalues, 256, c.sms, 8), 256, 0, c.stream>>>(accum, inv_samples, nvalues, out);
}
void launch_resolve_peers(const LaunchCtx& c, const PeerAccums& A, float inv_samples, uint32_t nvalues, uint8_t* out, float* sum) {
    k_resolve_peers<<<grid_for(nvalues, 256, c.sms, 8), 256, 0, c.stream>>>(A, inv_samples, nvalues, out, sum);
}
void launch_tonemap(const LaunchCtx& c, const float* rgb, uint32_t nvalues, uint8_t* out) {
    k_tonemap<<<grid_for(nvalues, 256, c.sms, 8), 256, 0, c.stream>>>(rgb, nvalues, out);
}
void launch_pack_rays(const LaunchCtx& c, long n, const float* o, const float* d, PathSoA P, uint32_t* q) {
    k_pack_rays<<<grid_for((uint64_t)n, 256, c.sms, 8), 256, 0, c.stream>>>(n, o, d, P, q);
}
void launch_unpack_hits(const LaunchCtx& c, const DevScene& S, long n, PathSoA P, HitSoA H, int32_t* id, float* t, float* nrm,
                        int32_t* interior) {
    k_unpack_hits<<<grid_for((uint64_t)n, 256, c.sms, 8), 256, 0, c.stream>>>(S, n, P, H, id, t, nrm, interior);
}
void launch_primitive_batch(const LaunchCtx& c, const DevScene& S, uint32_t prim, long n, const float* o, const float* d,
                            int32_t* hit, float* t, float* nrm, int32_t* interior) {
    k_primitive_batch<<<grid_for((uint64_t)n, 128, c.sms, 16), 128, 0, c.stream>>>(S, prim, n, o, d, hit, t, nrm, interior);
}
void launch_camera_batch(const LaunchCtx& c, const DevScene& S, long n, const float* xy, float* o, float* d) {
    k_camera_batch<<<grid_for((uint64_t)n, 128, c.sms, 16), 128, 0, c.stream>>>(S, n, xy, o, d);
}
void launch_pdf_batch(const LaunchCtx& c, const DevScene& S, long n, const float* x, const float* nr, const float* d, float* pdf) {
    k_pdf_batch<<<grid_for((uint64_t)n, 128, c.sms, 16), 128, 0, c.stream>>>(S, n, x, nr, d, pdf);
}
void launch_sample_batch(const LaunchCtx& c, const DevScene& S, long n, const float* x, const float* nr, uint32_t seed,
                         uint32_t sample, uint32_t bounce, float* dir) {
    k_sample_batch<<<grid_for((uint64_t)n, 128, c.sms, 16), 128, 0, c.stream>>>(S, n, x, nr, seed, sample, bounce, dir);
}

}  // namespace rtc
