// c_api.cu -- the C-ABI of include/rtc_b200.h: scene handle, HBM residency, the wavefront
// render loop, and host-buffer convenience wrappers.  No CPU fallback anywhere: a compute call
// on a scene without a device fails with RTC_ERR_NO_DEVICE.
#include <cuda_runtime.h>

#include <algorithm>
#include <array>
#include <cfloat>
#include <cmath>
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <fstream>
#include <functional>
#include <map>
#include <memory>
#include <sstream>
#include <stdexcept>
#include <string>
#include <thread>
#include <vector>

#include "device_scene.h"
#include "rt_kernels.h"
#include "rtc_b200.h"
#include "scene_host.h"

using namespace rtc;

namespace {
thread_local std::string g_error;
int fail(int code, const std::string& msg) {
    g_error = msg;
    return code;
}
#define CU(call)                                                                                   \
    do {                                                                                           \
        cudaError_t e_ = (call);                                                                   \
        if (e_ != cudaSuccess)                                                                     \
            return fail(RTC_ERR_CUDA, std::string(#call) + ": " + cudaGetErrorString(e_));         \
    } while (0)

// Owners of the CUDA resources of a scene.  Each frees what it holds when it is destroyed, with the device that made it
// current (~rtc_scene sees to that); one that holds nothing makes no CUDA call, so that a scene without a device never
// touches the runtime (even cudaFree(nullptr) creates a context).
// A buffer of `count` T that only ever grows (ensure(0) frees it): device memory, or pinned host memory.
template <class T, bool pinned = false>
struct Buf {
    T* p = nullptr;
    size_t n = 0;
    Buf() = default;
    Buf(Buf&& o) noexcept : p(o.p), n(o.n) { o.p = nullptr; o.n = 0; }   // move-only
    ~Buf() { drop(); }
    cudaError_t ensure(size_t count) {
        if (count <= n && p) return cudaSuccess;
        drop();
        if (count == 0) return cudaSuccess;
        cudaError_t e = pinned ? cudaMallocHost((void**)&p, count * sizeof(T)) : cudaMalloc((void**)&p, count * sizeof(T));
        if (e == cudaSuccess) n = count;
        return e;
    }
private:
    void drop() {
        if (p) pinned ? cudaFreeHost(p) : cudaFree(p);
        p = nullptr;
        n = 0;
    }
};
template <class T> using DevBuf = Buf<T>;
template <class T> using PinnedBuf = Buf<T, true>;
// a stream or an event, created by the first ensure()
template <class H, cudaError_t (*create)(H*), cudaError_t (*destroy)(H)>
struct Handle {
    H h = nullptr;
    Handle() = default;
    Handle(Handle&& o) noexcept : h(o.h) { o.h = nullptr; }   // move-only
    ~Handle() { if (h) destroy(h); }
    cudaError_t ensure() { return h ? cudaSuccess : create(&h); }
    operator H() const { return h; }
};
cudaError_t new_stream(cudaStream_t* st) { return cudaStreamCreateWithFlags(st, cudaStreamNonBlocking); }
cudaError_t new_event(cudaEvent_t* e) { return cudaEventCreateWithFlags(e, cudaEventDisableTiming); }
cudaError_t new_timed_event(cudaEvent_t* e) { return cudaEventCreate(e); }
using Stream = Handle<cudaStream_t, new_stream, cudaStreamDestroy>;
using Event = Handle<cudaEvent_t, new_event, cudaEventDestroy>;
using TimedEvent = Handle<cudaEvent_t, new_timed_event, cudaEventDestroy>;   // per-kernel timing (rtc_set_profiling)

constexpr uint64_t kDefaultBatchPaths = 1ull << 24;
constexpr int kMaxDepthSlots = 64;
constexpr int kStatWords = 16;
constexpr int kMaxWhittedDepth = 32;   // course_device.cuh kWhittedStack = kMaxWhittedDepth + 2
}  // namespace

struct rtc_scene {
    // the host scene is shared by the per-device replicas of a multi-device render (rtc_render_u8_multi)
    std::shared_ptr<HostScene> host_ptr;
    HostScene& host;
    rtc_scene() : host_ptr(std::make_shared<HostScene>()), host(*host_ptr) {}
    explicit rtc_scene(const std::shared_ptr<HostScene>& h) : host_ptr(h), host(*h) {}
    int device = -1;
    int sms = 0;
    int traversal = RTC_TRAVERSAL_INDEX;
    uint64_t batch_paths = kDefaultBatchPaths;
    uint64_t device_bytes = 0;
    // scene arrays in HBM: one pinned host mirror, TWO device arenas.  A scene upload is a single H2D copy;
    // rtc_scene_upload_async fills the arena that is not in use on a copy stream of its own, so that the upload of
    // frame i + 1 runs under the kernels of frame i, and the next render switches over.
    DevBuf<unsigned char> arena_dev[2];
    PinnedBuf<unsigned char> arena_host;
    size_t arena_bytes = 0;
    size_t part_off[24] = {0};            // offsets of the scene arrays inside an arena (index = ArenaPart)
    // Only the head of an arena travels over the host link; its tail -- levels >= 1 of the LCA range-minimum table,
    // the exact boxes of the few leaves that need them, the identity rotations of a scene without rotated
    // primitives: 11 of 35 MB for the 100k dragon -- is a pure function of the head and is rebuilt on the device
    // after every upload (expand_arena), on the copy stream, under the kernels of the previous frame.
    size_t upload_bytes = 0;              // size of the head = bytes per H2D copy (and of the pinned mirror)
    size_t sparse_boxes = 0;              // entries of the part ubox_sparse: (slot, min, max) of the leaves with an explicit box
    bool rot_generated = false;           // xf_rot is all identity and lives in the tail
    // xf_pos / (mat0, mat1) travel as a palette of distinct rows + a 16-bit index per primitive and are expanded on the device
    size_t xf_palette_rows = 0, mat_palette_rows = 0;
    std::vector<unsigned char> arena_full; // the whole arena as the host would have uploaded it (tests: rtc_scene_arena_check)
    int arena_cur = 0;                    // the arena the next render reads
    DevScene slices{};                    // pointers into arena_dev[arena_cur] (scalars filled by dev())
    Stream copy_stream;
    // kernels that read the scene take it with arena_begin and end with arena_end, which wait for / record these
    Event arena_ready[2];                 // upload into arena i complete
    Event arena_idle[2];                  // last kernel that read arena i complete
    bool arena_pending = false;           // an async upload has to be waited for by the next reader
    // frames in flight (rtc_frame_begin / rtc_frame_end): per slot a stream, buffers and a pinned image
    struct Frame {
        Stream stream;
        Event done;
        DevBuf<float> accum;
        DevBuf<uint8_t> rgb;
        PinnedBuf<uint8_t> host;
        bool busy = false;
    };
    Frame frames[2];
    Event resolved;                       // rtc_resolve_to_host_async: the image may leave the device
    // float4 pixel sums of the renders in flight (k_shade deposits, k_fold reads): two, used alternately
    DevBuf<float4> accum4[2];
    Event accum4_idle[2];
    int accum4_next = 0;
    // probe entry points (rtc_intersect, ...): staging buffers that only ever grow
    struct Probe {
        DevBuf<float> fin[3];
        DevBuf<float> fout[2];
        DevBuf<int32_t> iout[2];
        DevBuf<float4> ray[2];
        DevBuf<uint32_t> hit, tq, q;
    } probe;
    // per-device replicas for rtc_render_u8_multi (this scene's own device is not among them)
    std::vector<std::unique_ptr<rtc_scene>> replicas;
    Stream multi_stream;
    Event multi_done;
    // wavefront state: kMaxLanes independent sets, each with its own stream, so that batches
    // overlap (the tail of one persistent k_traverse launch runs next to the other lane's kernels)
    struct Lane {
        Stream stream;
        Event done;
        DevBuf<float4> path[2][3];           // two ping-pong sets of (origin | sample, direction | closest plane, throughput | pixel)
        DevBuf<uint32_t> hit_id[2];
        DevBuf<uint32_t> trav_queue;         // ray indices handed to k_traverse
        DevBuf<uint32_t> queue;              // 4 x kMaxDepthSlots words: path counts (front, back per bounce), traverse counts, cursors
    };
    static constexpr int kMaxLanes = 4;
    Lane lanes[kMaxLanes];
    int nlanes = 2;                      // env RTC_STREAMS (1..4)
    unsigned next_lane = 0;              // small renders take the lanes in turn
    // renders up to this many paths are ONE batch on the next lane in turn (env RTC_SMALL_RENDER; measured on B200 with
    // two renders in flight: 16 spp of the headline frame 1619 -> 1805 Mpaths/s, 32 spp 1817 -> 1907)
    uint64_t small_render_paths = 9000000;
    Event fork;
    DevBuf<unsigned long long> stats;    // 16 words: rtc_render_counters (8) + rtc_traverse_lanes (8)
    DevBuf<float> accum;                 // internal accumulation buffer for the convenience calls
    DevBuf<uint8_t> rgb;
    // rtc_render_adaptive: the even- and odd-sample sums per pixel, the active tile and pixel lists of the current and the
    // next pass, the samples every tile took, the list lengths (tiles, pixels) of both passes and their pinned host copy
    struct Adaptive {
        DevBuf<float4> half[2];
        DevBuf<uint32_t> tiles[2], pixels[2], tile_n, counts, spp;
        DevBuf<float> halves;
        PinnedBuf<uint32_t> counts_host;
    } adaptive;
    // rtc_denoise / rtc_render_denoised: the linear mean u (3 floats per pixel), D and V (k_denoise_prep) and the filtered
    // mean (k_denoise_nlm)
    struct Denoise {
        DevBuf<float> u, mean;
        DevBuf<float4> d, v;
    } denoise;
    uint64_t launches = 0;
    // optional per-kernel timing (CUDA events on the launching stream)
    bool profiling = false;
    bool count_visits = false;
    struct Span { cudaEvent_t a, b; int kind; };
    std::vector<Span> spans;
    std::vector<TimedEvent> event_pool;    // span i holds events 2 i and 2 i + 1
    double prof_ms[4] = {0, 0, 0, 0};      // generate, traverse (or reference-tree extend), shade, pre
    uint64_t prof_launches[4] = {0, 0, 0, 0};

    void span_begin(int kind, cudaStream_t st) {
        if (!profiling) return;
        while (event_pool.size() < 2 * spans.size() + 2) {
            event_pool.emplace_back();
            event_pool.back().ensure();
        }
        Span sp{event_pool[2 * spans.size()], event_pool[2 * spans.size() + 1], kind};
        cudaEventRecord(sp.a, st);
        spans.push_back(sp);
    }
    void span_end(cudaStream_t st) {
        if (!profiling) return;
        cudaEventRecord(spans.back().b, st);
    }
    void collect_spans() {
        for (Span& sp : spans) {
            float ms = 0.f;
            if (cudaEventSynchronize(sp.b) == cudaSuccess && cudaEventElapsedTime(&ms, sp.a, sp.b) == cudaSuccess) {
                prof_ms[sp.kind] += ms;
                prof_launches[sp.kind] += 1;
            }
        }
        spans.clear();
    }

    DevScene dev() const {
        DevScene S;
        std::memset(&S, 0, sizeof S);
        S.geo0 = slices.geo0; S.geo1 = slices.geo1; S.geo2 = slices.geo2; S.xf_pos = slices.xf_pos; S.xf_rot = slices.xf_rot;
        S.mat0 = slices.mat0; S.mat1 = slices.mat1; S.inodes = slices.inodes; S.rnodes = slices.rnodes; S.rmeta = slices.rmeta;
        S.lca = slices.lca; S.lights = slices.lights; S.planes = slices.planes; S.ubox = slices.ubox;
        S.plights = slices.plights;
        fill_dev_scalars(host, S);
        return S;
    }
    // the replicas free themselves on their own devices, then the members are destroyed with this scene's device current
    ~rtc_scene() {
        replicas.clear();
        if (device < 0) return;
        cudaSetDevice(device);
        collect_spans();
    }
};

namespace {

// RTC_TIMING=1: phase times of scene creation on stderr (the host build prints its own phases, bvh_build.cpp)
struct Lap {
    bool on = std::getenv("RTC_TIMING") != nullptr;
    std::chrono::steady_clock::time_point t0 = std::chrono::steady_clock::now();
    void operator()(const char* what) {
        if (!on) return;
        const auto t1 = std::chrono::steady_clock::now();
        std::fprintf(stderr, "[rtc timing] %-28s %8.1f ms\n", what, std::chrono::duration<double, std::milli>(t1 - t0).count());
        t0 = t1;
    }
};

// Lays the flat scene arrays out in one arena (256-byte aligned slices): first everything that has to be uploaded, then
// what the device derives from it.
enum ArenaPart { A_GEO0, A_GEO1, A_GEO2, A_XF_POS, A_MAT0, A_MAT1, A_INODES, A_RNODES, A_RMETA, A_LIGHTS, A_PLANES, A_PLIGHTS,
                 A_UBOX_SPARSE, A_XF_PAL, A_XF_IDX, A_MAT_PAL, A_MAT_IDX, A_XF_ROT, A_LCA, A_UBOX, A_COUNT };
static_assert(A_COUNT <= 24, "rtc_scene::part_off");
// distinct rows of a float4 table with `k` float4 per row, and the row index of every entry; empty result = more than 65536
// distinct rows (the table then travels as it is)
bool build_palette(const f4* rows0, const f4* rows1, size_t n, std::vector<f4>& palette, std::vector<uint16_t>& index) {
    struct Key { uint32_t w[8]; bool operator<(const Key& o) const { return std::memcmp(w, o.w, sizeof w) < 0; } };
    std::map<Key, uint32_t> seen;
    palette.clear();
    index.assign(n, 0);
    for (size_t i = 0; i < n; ++i) {
        Key k;
        std::memset(&k, 0, sizeof k);
        std::memcpy(k.w, &rows0[i], 16);
        if (rows1) std::memcpy(k.w + 4, &rows1[i], 16);
        auto it = seen.find(k);
        if (it == seen.end()) {
            if (seen.size() >= 65536) { palette.clear(); index.clear(); return false; }
            it = seen.emplace(k, (uint32_t)seen.size()).first;
            palette.push_back(rows0[i]);
            if (rows1) palette.push_back(rows1[i]);
        }
        index[i] = (uint16_t)it->second;
    }
    return true;
}
void point_slices(rtc_scene* s, int which) {
    unsigned char* base = s->arena_dev[which].p;
    const size_t* off = s->part_off;
    DevScene& D = s->slices;
    D.geo0 = (const float4*)(base + off[A_GEO0]);     D.geo1 = (const float4*)(base + off[A_GEO1]);
    D.geo2 = (const float4*)(base + off[A_GEO2]);     D.xf_pos = (const float4*)(base + off[A_XF_POS]);
    D.xf_rot = (const float4*)(base + off[A_XF_ROT]); D.mat0 = (const float4*)(base + off[A_MAT0]);
    D.mat1 = (const float4*)(base + off[A_MAT1]);     D.inodes = (const float4*)(base + off[A_INODES]);
    D.rnodes = (const float4*)(base + off[A_RNODES]); D.rmeta = (const uint4*)(base + off[A_RMETA]);
    D.lca = (const uint32_t*)(base + off[A_LCA]);     D.lights = (const int32_t*)(base + off[A_LIGHTS]);
    D.planes = (const float4*)(base + off[A_PLANES]);
    D.ubox = (const float4*)(base + off[A_UBOX]);
    D.plights = (const float4*)(base + off[A_PLIGHTS]);
    s->arena_cur = which;
}
int prepare_arena(rtc_scene* s) {
    if (s->device < 0) return fail(RTC_ERR_NO_DEVICE, "scene has no CUDA device");
    CU(cudaSetDevice(s->device));
    if (s->arena_host.p) return RTC_OK;
    Lap lap;
    const FlatScene& F = s->host.flat;
    // The device reads ubox only for leaves whose exact box cannot be read off a single untransformed triangle
    // (rt_device.cuh leaf_test): the arena keeps those, as (slot, min, max) = 3 float4 each, and zeros elsewhere.
    std::vector<f4> dev_ubox(F.ubox.size(), f4{0.f, 0.f, 0.f, 0.f});
    for (const RefNode& nd : s->host.nodes) {
        if (nd.left != UINT32_MAX || nd.count == 0) continue;
        const Primitive& p0 = s->host.prims[nd.first];
        const bool ident = p0.rot.x == 0.f && p0.rot.y == 0.f && p0.rot.z == 0.f && p0.rot.w == 1.f && p0.pos.x == 0.f &&
                           p0.pos.y == 0.f && p0.pos.z == 0.f;
        if (nd.count == 1 && p0.type == PT_TRIANGLE && ident) continue;   // IREF_FAST (bvh_build.cpp)
        dev_ubox[2 * (size_t)nd.first] = F.ubox[2 * (size_t)nd.first];
        dev_ubox[2 * (size_t)nd.first + 1] = F.ubox[2 * (size_t)nd.first + 1];
    }
    std::vector<f4> sparse;
    for (size_t i = 0; 2 * i + 1 < dev_ubox.size(); ++i) {
        const f4 &mn = dev_ubox[2 * i], &mx = dev_ubox[2 * i + 1];
        const bool zero = mn.x == 0.f && mn.y == 0.f && mn.z == 0.f && mn.w == 0.f && mx.x == 0.f && mx.y == 0.f && mx.z == 0.f && mx.w == 0.f
                          && !std::signbit(mn.x) && !std::signbit(mn.y) && !std::signbit(mn.z) && !std::signbit(mx.x) && !std::signbit(mx.y) && !std::signbit(mx.z);
        if (zero) continue;
        f4 slot{0.f, 0.f, 0.f, 0.f};
        const uint32_t idx = (uint32_t)i;
        std::memcpy(&slot.x, &idx, 4);
        sparse.push_back(slot); sparse.push_back(mn); sparse.push_back(mx);
    }
    s->sparse_boxes = sparse.size() / 3;
    s->rot_generated = !(F.features & FE_ROTATION);   // every rotation is (0, 0, 0, 1)
    for (const f4& q : F.xf_rot)
        if (!(q.x == 0.f && q.y == 0.f && q.z == 0.f && q.w == 1.f) || std::signbit(q.x) || std::signbit(q.y) || std::signbit(q.z)) s->rot_generated = false;
    std::vector<f4> xf_pal, mat_pal;
    std::vector<uint16_t> xf_idx, mat_idx;
    const bool xf_packed = F.xf_pos.size() >= 1024 && build_palette(F.xf_pos.data(), nullptr, F.xf_pos.size(), xf_pal, xf_idx) &&
                           xf_pal.size() * 8 < F.xf_pos.size();
    const bool mat_packed = F.mat0.size() >= 1024 && build_palette(F.mat0.data(), F.mat1.data(), F.mat0.size(), mat_pal, mat_idx) &&
                            mat_pal.size() * 8 < F.mat0.size();
    lap("arena: sparse boxes, palettes");
    s->xf_palette_rows = xf_packed ? xf_pal.size() : 0;
    s->mat_palette_rows = mat_packed ? mat_pal.size() / 2 : 0;
    struct Part { const void* src; size_t bytes; bool head; };
    Part parts[A_COUNT];
    parts[A_GEO0] = {F.geo0.data(), F.geo0.size() * sizeof(f4), true};       parts[A_GEO1] = {F.geo1.data(), F.geo1.size() * sizeof(f4), true};
    parts[A_GEO2] = {F.geo2.data(), F.geo2.size() * sizeof(f4), true};       parts[A_XF_POS] = {F.xf_pos.data(), F.xf_pos.size() * sizeof(f4), !xf_packed};
    parts[A_MAT0] = {F.mat0.data(), F.mat0.size() * sizeof(f4), !mat_packed}; parts[A_MAT1] = {F.mat1.data(), F.mat1.size() * sizeof(f4), !mat_packed};
    parts[A_INODES] = {F.inodes.data(), F.inodes.size() * sizeof(f4), true}; parts[A_RNODES] = {F.rnodes.data(), F.rnodes.size() * sizeof(f4), true};
    parts[A_RMETA] = {F.rmeta.data(), F.rmeta.size() * sizeof(u4), true};    parts[A_LIGHTS] = {F.lights.data(), F.lights.size() * sizeof(int32_t), true};
    parts[A_PLANES] = {F.planes.data(), F.planes.size() * sizeof(f4), true}; parts[A_PLIGHTS] = {F.plights.data(), F.plights.size() * sizeof(f4), true};
    parts[A_UBOX_SPARSE] = {sparse.data(), sparse.size() * sizeof(f4), true};
    parts[A_XF_PAL] = {xf_pal.data(), xf_packed ? xf_pal.size() * sizeof(f4) : 0, true};
    parts[A_XF_IDX] = {xf_idx.data(), xf_packed ? xf_idx.size() * sizeof(uint16_t) : 0, true};
    parts[A_MAT_PAL] = {mat_pal.data(), mat_packed ? mat_pal.size() * sizeof(f4) : 0, true};
    parts[A_MAT_IDX] = {mat_idx.data(), mat_packed ? mat_idx.size() * sizeof(uint16_t) : 0, true};
    parts[A_XF_ROT] = {F.xf_rot.data(), F.xf_rot.size() * sizeof(f4), !s->rot_generated};
    parts[A_LCA] = {F.lca.data(), F.lca.size() * sizeof(uint32_t), false};   // its level 0 travels as a second, small copy
    parts[A_UBOX] = {dev_ubox.data(), dev_ubox.size() * sizeof(f4), false};
    size_t total = 0, head = 0;
    for (int pass = 0; pass < 2; ++pass) {   // the parts that travel first, then the ones the device derives from them
        for (int i = 0; i < A_COUNT; ++i) {
            if (parts[i].head != (pass == 0)) continue;
            s->part_off[i] = total;
            total += (parts[i].bytes + 255) & ~(size_t)255;
        }
        if (pass == 0) head = total;
    }
    if (total == 0) total = 256;
    s->arena_full.assign(total, 0);
    for (int i = 0; i < A_COUNT; ++i)
        if (parts[i].bytes) std::memcpy(s->arena_full.data() + s->part_off[i], parts[i].src, parts[i].bytes);
    s->upload_bytes = head;
    s->arena_bytes = total;
    lap("arena: host image");
    CU(s->arena_dev[0].ensure(total));
    CU(cudaMemset(s->arena_dev[0].p, 0, total));   // the padding between the device-built parts is never written again
    // pinned mirror of what travels: the head, and level 0 of the LCA table right behind it
    const size_t level0 = F.lca_levels ? (((size_t)s->host.nbvh * sizeof(uint32_t) + 255) & ~(size_t)255) : 0;
    CU(s->arena_host.ensure(head + level0 + 256));
    std::memcpy(s->arena_host.p, s->arena_full.data(), head);
    if (level0) std::memcpy(s->arena_host.p + head, s->arena_full.data() + s->part_off[A_LCA], (size_t)s->host.nbvh * sizeof(uint32_t));
    s->device_bytes = head + (F.lca_levels ? (size_t)s->host.nbvh * sizeof(uint32_t) : 0);
    point_slices(s, 0);
    for (int a = 0; a < 2; ++a) {
        CU(s->arena_ready[a].ensure());
        CU(s->arena_idle[a].ensure());
        CU(s->accum4_idle[a].ensure());
    }
    CU(s->copy_stream.ensure());
    CU(s->stats.ensure(kStatWords));
    CU(cudaMemset(s->stats.p, 0, kStatWords * sizeof(unsigned long long)));
    lap("arena: cudaMalloc, pinned mirror");
    return RTC_OK;
}
// H2D copies of the head (+ LCA level 0) into arena `target`, then the device-side rebuild of the tail; all on `st`
int issue_upload(rtc_scene* s, int target, cudaStream_t st) {
    unsigned char* dev = s->arena_dev[target].p;
    const FlatScene& F = s->host.flat;
    if (s->upload_bytes) CU(cudaMemcpyAsync(dev, s->arena_host.p, s->upload_bytes, cudaMemcpyHostToDevice, st));
    const size_t level0 = F.lca_levels ? (size_t)s->host.nbvh * sizeof(uint32_t) : 0;
    if (level0) CU(cudaMemcpyAsync(dev + s->part_off[A_LCA], s->arena_host.p + s->upload_bytes, level0, cudaMemcpyHostToDevice, st));
    LaunchCtx c{st, s->sms};
    if (F.lca_levels > 1)
        launch_expand_lca(c, (uint32_t*)(dev + s->part_off[A_LCA]), (const uint4*)(dev + s->part_off[A_RMETA]), s->host.nbvh, F.lca_levels);
    if (!F.ubox.empty()) {
        CU(cudaMemsetAsync(dev + s->part_off[A_UBOX], 0, F.ubox.size() * sizeof(f4), st));
        if (s->sparse_boxes)
            launch_expand_boxes(c, (const float4*)(dev + s->part_off[A_UBOX_SPARSE]), (uint32_t)s->sparse_boxes, (float4*)(dev + s->part_off[A_UBOX]));
    }
    if (s->rot_generated && !F.xf_rot.empty())
        launch_fill_identity_rotations(c, (float4*)(dev + s->part_off[A_XF_ROT]), (uint32_t)F.xf_rot.size());
    if (s->xf_palette_rows)
        launch_expand_palette(c, (const float4*)(dev + s->part_off[A_XF_PAL]), (const uint16_t*)(dev + s->part_off[A_XF_IDX]),
                              (uint32_t)F.xf_pos.size(), (float4*)(dev + s->part_off[A_XF_POS]), nullptr);
    if (s->mat_palette_rows)
        launch_expand_palette(c, (const float4*)(dev + s->part_off[A_MAT_PAL]), (const uint16_t*)(dev + s->part_off[A_MAT_IDX]),
                              (uint32_t)F.mat0.size(), (float4*)(dev + s->part_off[A_MAT0]), (float4*)(dev + s->part_off[A_MAT1]));
    CU(cudaGetLastError());
    return RTC_OK;
}
// synchronous upload into the arena in use, complete on return
int upload_scene(rtc_scene* s, uint64_t* h2d) {
    int rc = prepare_arena(s);
    if (rc) return rc;
    Lap lap;
    CU(cudaDeviceSynchronize());   // nothing may still be reading the arena
    if ((rc = issue_upload(s, s->arena_cur, s->copy_stream))) return rc;
    CU(cudaStreamSynchronize(s->copy_stream));
    lap("upload + device-built tail");
    s->arena_pending = false;
    if (h2d) *h2d = s->device_bytes;
    return RTC_OK;
}
// asynchronous upload into the OTHER arena on the copy stream; the next render waits for it and reads that arena
int upload_scene_async(rtc_scene* s, uint64_t* h2d) {
    int rc = prepare_arena(s);
    if (rc) return rc;
    const int target = 1 - s->arena_cur;
    if (!s->arena_dev[target].p) {
        CU(s->arena_dev[target].ensure(s->arena_bytes));
        CU(cudaMemsetAsync(s->arena_dev[target].p, 0, s->arena_bytes, s->copy_stream));
    }
    CU(cudaStreamWaitEvent(s->copy_stream, s->arena_idle[target], 0));   // the renders that read it are done
    if ((rc = issue_upload(s, target, s->copy_stream))) return rc;
    CU(cudaEventRecord(s->arena_ready[target], s->copy_stream));
    point_slices(s, target);
    s->arena_pending = true;
    if (h2d) *h2d = s->device_bytes;
    return RTC_OK;
}

int finish_scene(rtc_scene* s, int device) {
    if (const char* v = std::getenv("RTC_STREAMS")) {
        int n = std::atoi(v);
        s->nlanes = n < 1 ? 1 : (n > rtc_scene::kMaxLanes ? rtc_scene::kMaxLanes : n);
    }
    if (const char* v = std::getenv("RTC_SMALL_RENDER")) s->small_render_paths = std::strtoull(v, nullptr, 10);
    s->device = device;
    if (device >= 0) {
        int count = 0;
        if (cudaGetDeviceCount(&count) != cudaSuccess || device >= count)
            return fail(RTC_ERR_NO_DEVICE, "CUDA device " + std::to_string(device) + " is not available");
        cudaDeviceProp prop;
        cudaGetDeviceProperties(&prop, device);
        s->sms = prop.multiProcessorCount;
        return upload_scene(s, nullptr);
    }
    return RTC_OK;
}

// the host build of `text` in `s`, its limits checked, then resident on `device` (none when < 0)
int build_scene(rtc_scene* s, const std::string& text, int device, int dialect) {
    Lap lap;
    try {
        s->host.dialect = dialect;
        s->host.parse(text);
        lap("scene text -> primitives");
        s->host.init();
        lap("host build (sum of the above)");
    } catch (const std::exception& e) {
        return fail(RTC_ERR_UNSUPPORTED, e.what());
    }
    if (s->host.ray_depth + 2 > (unsigned)kMaxDepthSlots) return fail(RTC_ERR_UNSUPPORTED, "RAY_DEPTH above 62 is not supported");
    if (dialect == DIALECT_HW2 && s->host.ray_depth > (unsigned)kMaxWhittedDepth)
        return fail(RTC_ERR_UNSUPPORTED, "hw2 dialect: RAY_DEPTH above 32 is not supported");
    if (s->host.flat.ref_depth + 1 >= 96) return fail(RTC_ERR_UNSUPPORTED, "reference BVH deeper than 95 levels is not supported");
    return finish_scene(s, device);
}
rtc_scene* make_scene(const std::string& text, int device, int dialect = DIALECT_HW5) {
    if (dialect < DIALECT_HW1 || dialect > DIALECT_HW5) {
        fail(RTC_ERR_ARG, "dialect must be 1..5");
        return nullptr;
    }
    rtc_scene* s = new rtc_scene();
    if (build_scene(s, text, device, dialect) == RTC_OK) return s;
    delete s;
    return nullptr;
}

int need_device(const rtc_scene* s) {
    if (!s) return fail(RTC_ERR_ARG, "null scene");
    if (s->device < 0) return fail(RTC_ERR_NO_DEVICE, "scene was created without a CUDA device; there is no CPU path");
    cudaError_t e = cudaSetDevice(s->device);
    if (e != cudaSuccess) return fail(RTC_ERR_CUDA, std::string("cudaSetDevice: ") + cudaGetErrorString(e));
    return RTC_OK;
}

// Every entry point whose kernels read the scene brackets them with these two, on the stream of its launches.
// arena_begin: the scene for kernels on `st`, after an asynchronous upload into the arena in use has landed.
int arena_begin(rtc_scene* s, cudaStream_t st, DevScene* S) {
    if (s->arena_pending) CU(cudaStreamWaitEvent(st, s->arena_ready[s->arena_cur], 0));
    *S = s->dev();
    return RTC_OK;
}
// arena_end: after the last launch; the next upload into this arena waits for it
int arena_end(rtc_scene* s, cudaStream_t st) {
    CU(cudaEventRecord(s->arena_idle[s->arena_cur], st));
    return RTC_OK;
}

// the samples of one frame: SAMPLES, or the one deterministic frame of hw1 / hw2, which have no SAMPLES
int frame_samples(const rtc_scene* s, uint32_t* samples) {
    *samples = s->host.dialect <= DIALECT_HW2 ? 1u : s->host.samples;
    if (*samples == 0) return fail(RTC_ERR_ARG, "scene has SAMPLES 0");
    return RTC_OK;
}
// one frame of `samples` samples on `st`: zero `accum`, add the samples, resolve them into `rgb`
int render_frame(rtc_scene* s, uint32_t seed, uint32_t samples, float* accum, uint8_t* rgb, cudaStream_t st) {
    const size_t nvalues = 3 * (size_t)s->host.cam.width * s->host.cam.height;
    CU(cudaMemsetAsync(accum, 0, nvalues * sizeof(float), st));
    int rc = rtc_render_accumulate(s, seed, 0, samples, accum, st);
    return rc ? rc : rtc_render_resolve(s, accum, samples, rgb, st);
}
int write_ppm(const char* path, unsigned width, unsigned height, const std::vector<uint8_t>& img) {
    std::ofstream out(path, std::ios::binary);
    if (!out) return fail(RTC_ERR_IO, std::string("cannot open output file ") + path);
    out << "P6\n" << width << " " << height << "\n" << 255 << "\n";  // src/scene.cpp:206-208
    out.write(reinterpret_cast<const char*>(img.data()), (std::streamsize)img.size());
    if (!out) return fail(RTC_ERR_IO, std::string("write failed: ") + path);
    return RTC_OK;
}

// temporary device copies of host arrays for the probe entry points
struct Staged {
    std::vector<void*> ptrs;
    ~Staged() { for (void* p : ptrs) cudaFree(p); }
    template <class T>
    T* in(const T* host, size_t n) {
        T* d = nullptr;
        if (cudaMalloc(&d, (n ? n : 1) * sizeof(T)) != cudaSuccess) return nullptr;
        ptrs.push_back(d);
        if (n && cudaMemcpy(d, host, n * sizeof(T), cudaMemcpyHostToDevice) != cudaSuccess) return nullptr;
        return d;
    }
    template <class T>
    T* out(size_t n) {
        T* d = nullptr;
        if (cudaMalloc(&d, (n ? n : 1) * sizeof(T)) != cudaSuccess) return nullptr;
        ptrs.push_back(d);
        return d;
    }
};
#define NEED(ptr) if (!(ptr)) return fail(RTC_ERR_CUDA, "device staging allocation/copy failed")

// the lane streams are non-blocking and joined only into the stream a render was given: whoever reads the
// counters through another stream waits for the lanes themselves
cudaError_t sync_lanes(rtc_scene* s) {
    for (auto& l : s->lanes)
        if (l.stream) {
            cudaError_t e = cudaStreamSynchronize(l.stream);
            if (e != cudaSuccess) return e;
        }
    return cudaSuccess;
}

int ensure_wavefront(rtc_scene* s, uint64_t cap, int nlanes) {
    for (int i = 0; i < nlanes; ++i) {
        rtc_scene::Lane& l = s->lanes[i];
        CU(l.stream.ensure());
        CU(l.done.ensure());
        for (auto& set : l.path) for (auto& b : set) CU(b.ensure(cap));
        for (auto& b : l.hit_id) CU(b.ensure(cap));
        CU(l.trav_queue.ensure(cap * kTraverseQueueWords));
        CU(l.queue.ensure(4 * kMaxDepthSlots));
    }
    return RTC_OK;
}

// Which (pixel, sample) path p of a render is: pixel p % npix of the frame and sample sample_first + p / npix when
// plist is null (rtc_render_accumulate), else pixel plist[p % npix] and sample sample_first + 2 (p / npix) (an adaptive
// pass renders the even or the odd samples of its pixel list)
struct PathMap {
    const uint32_t* plist;
    uint32_t npix;
    uint32_t sample_first;
};
// fork: the lane streams of the next render_paths calls start after everything already queued on the caller's stream
int fork_lanes(rtc_scene* s, cudaStream_t user) {
    CU(s->fork.ensure());
    CU(cudaEventRecord(s->fork, user));
    return RTC_OK;
}
// join: the caller's stream continues when the lanes in `used` (bit i = lane i) are done
int join_lanes(rtc_scene* s, unsigned used, cudaStream_t user) {
    for (int i = 0; i < rtc_scene::kMaxLanes; ++i) {
        if (!(used >> i & 1u)) continue;
        CU(cudaEventRecord(s->lanes[i].done, s->lanes[i].stream));
        CU(cudaStreamWaitEvent(user, s->lanes[i].done, 0));
    }
    return RTC_OK;
}
// The wavefront batches of `total` paths laid out by `map`: every hit deposits into `target` (float4 per pixel of the
// frame).  The lanes wait for the last fork_lanes; the lanes that carry work are added to *used.
int render_paths(rtc_scene* s, const DevScene& S, uint32_t seed, const PathMap& map, uint64_t total, float4* target, unsigned* used) {
    int rc;
    const uint32_t depth = s->host.ray_depth;
    // batch size: the configured one, but small enough that every lane gets a batch (overlap matters
    // more than batch size: profiles/r01_experiments.md), rounded up to whole warps
    uint64_t cap = total < s->batch_paths ? total : s->batch_paths;
    // A small render (the share of one GPU of eight: 4 Mi paths) is ONE batch on the next lane in turn instead of one
    // batch per lane: its launches are twice as large (a persistent k_traverse launch ends with its longest ray, ~30 us
    // whatever its size), and the overlap comes from the caller's next render, which takes the other lane.
    const bool whole = !s->profiling && s->nlanes > 1 && total <= s->small_render_paths;
    if (!s->profiling && s->nlanes > 1 && !whole) {
        uint64_t per_lane = ((total + s->nlanes - 1) / s->nlanes + 31) & ~(uint64_t)31;
        if (per_lane < cap) cap = per_lane;
    }
    const uint64_t nbatches = (total + cap - 1) / cap;
    // per-kernel event timing needs the kernels back to back on one stream
    const int nlanes = s->profiling ? 1 : whole ? s->nlanes : (int)(nbatches < (uint64_t)s->nlanes ? nbatches : (uint64_t)s->nlanes);
    const int lane_first = whole ? (int)(s->next_lane++ % (unsigned)s->nlanes) : 0;
    if ((rc = ensure_wavefront(s, cap, nlanes))) return rc;
    for (int i = 0; i < nlanes; ++i)
        if (!whole || i == lane_first) {   // the other lanes belong to the caller's other renders
            CU(cudaStreamWaitEvent(s->lanes[i].stream, s->fork, 0));
            *used |= 1u << i;
        }
    uint64_t batch = 0;
    for (uint64_t first = 0; first < total; first += cap, ++batch) {
        rtc_scene::Lane& L = s->lanes[(lane_first + batch) % nlanes];
        cudaStream_t st = L.stream;
        LaunchCtx c{st, s->sms};
        uint32_t* tqc = L.queue.p + 2 * kMaxDepthSlots;    // rays queued for k_traverse, per bounce
        uint32_t* cursor = L.queue.p + 3 * kMaxDepthSlots; // k_traverse work cursors, per bounce
        uint32_t count = (uint32_t)((total - first) < cap ? (total - first) : cap);
        CU(cudaMemsetAsync(L.queue.p, 0, 4 * kMaxDepthSlots * sizeof(uint32_t), st));
        PathSoA cur{L.path[0][0].p, L.path[0][1].p, L.path[0][2].p};
        PathSoA nxt{L.path[1][0].p, L.path[1][1].p, L.path[1][2].p};
        HitSoA hcur{L.hit_id[0].p}, hnxt{L.hit_id[1].p};
        s->span_begin(0, st);
        if (map.plist) launch_generate_list(c, S, cur, hcur, L.queue.p, L.trav_queue.p, tqc, first, count, seed, map.plist, map.npix, map.sample_first);
        else launch_generate(c, S, cur, hcur, L.queue.p, L.trav_queue.p, tqc, first, count, seed, map.sample_first);
        s->span_end(st);
        s->launches++;
        for (uint32_t b = 1; b <= depth; ++b) {
            s->span_begin(1, st);
            if (s->traversal == RTC_TRAVERSAL_REFTREE) launch_extend_reftree(c, S, cur, hcur, L.queue.p + 2 * (b - 1), count);
            else launch_traverse(c, S, cur, hcur, count, L.trav_queue.p, tqc + (b - 1), cursor + (b - 1), s->count_visits, s->stats.p);
            s->span_end(st);
            s->span_begin(2, st);
            launch_shade(c, S, cur, hcur, nxt, hnxt, L.queue.p + 2 * (b - 1), L.queue.p + 2 * b, L.trav_queue.p, tqc + b, count,
                         target, b, seed);
            s->span_end(st);
            s->launches += 2;
            PathSoA tmp = cur; cur = nxt; nxt = tmp;
            HitSoA htmp = hcur; hcur = hnxt; hnxt = htmp;
        }
        launch_tally(c, L.queue.p, tqc, depth, s->stats.p);
        s->launches++;
    }
    return RTC_OK;
}

}  // namespace

extern "C" {

const char* rtc_last_error(void) { return g_error.c_str(); }
int rtc_version(void) { return 100; }
int rtc_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
    return n;
}

rtc_scene* rtc_scene_parse(const char* text, long len, int device) {
    if (!text || len < 0) { fail(RTC_ERR_ARG, "null scene text"); return nullptr; }
    return make_scene(std::string(text, (size_t)len), device);
}
rtc_scene* rtc_scene_parse_dialect(const char* text, long len, int device, int dialect) {
    if (!text || len < 0) { fail(RTC_ERR_ARG, "null scene text"); return nullptr; }
    return make_scene(std::string(text, (size_t)len), device, dialect);
}
rtc_scene* rtc_scene_load_dialect(const char* path, int device, int dialect) {
    if (!path) { fail(RTC_ERR_ARG, "null path"); return nullptr; }
    std::ifstream in(path, std::ios::binary);
    if (!in) { fail(RTC_ERR_IO, std::string("cannot open scene file ") + path); return nullptr; }
    Lap lap;
    std::ostringstream ss;
    ss << in.rdbuf();
    lap("read scene file");
    return make_scene(ss.str(), device, dialect);
}
rtc_scene* rtc_scene_load(const char* path, int device) { return rtc_scene_load_dialect(path, device, DIALECT_HW5); }
int rtc_scene_dialect(const rtc_scene* s) { return s ? s->host.dialect : 0; }
void rtc_scene_free(rtc_scene* s) {
    delete s;
}
int rtc_scene_upload(rtc_scene* s, uint64_t* h2d_bytes) {
    int rc = need_device(s);
    if (rc) return rc;
    return upload_scene(s, h2d_bytes);
}
int rtc_scene_arena_check(rtc_scene* s, uint64_t* mismatching_bytes) {
    int rc = need_device(s);
    if (rc) return rc;
    if (!mismatching_bytes) return fail(RTC_ERR_ARG, "null argument");
    CU(cudaDeviceSynchronize());
    std::vector<unsigned char> got(s->arena_bytes);
    CU(cudaMemcpy(got.data(), s->arena_dev[s->arena_cur].p, s->arena_bytes, cudaMemcpyDeviceToHost));
    uint64_t bad = 0;
    for (size_t i = 0; i < s->arena_bytes; ++i) bad += got[i] != s->arena_full[i];
    *mismatching_bytes = bad;
    return RTC_OK;
}
int rtc_scene_info(const rtc_scene* s, uint32_t out[8]) {
    if (!s || !out) return fail(RTC_ERR_ARG, "null argument");
    out[0] = s->host.cam.width; out[1] = s->host.cam.height; out[2] = s->host.ray_depth; out[3] = s->host.samples;
    out[4] = (uint32_t)s->host.prims.size(); out[5] = s->host.nbvh; out[6] = (uint32_t)s->host.nodes.size();
    out[7] = (uint32_t)s->host.lights.size();
    return RTC_OK;
}
int rtc_scene_stats(const rtc_scene* s, uint64_t out[8]) {
    if (!s || !out) return fail(RTC_ERR_ARG, "null argument");
    const FlatScene& F = s->host.flat;
    out[0] = F.inodes.size() / kIndexNodeF4; out[1] = F.index_depth; out[2] = F.ref_depth; out[3] = F.units;
    out[4] = s->device_bytes; out[5] = F.lca_levels; out[6] = kIndexNodeF4 * sizeof(f4); out[7] = F.features;
    return RTC_OK;
}
int rtc_scene_override(rtc_scene* s, int width, int height, int samples, int ray_depth) {
    if (!s) return fail(RTC_ERR_ARG, "null scene");
    if (ray_depth >= 0 && ray_depth + 2 > kMaxDepthSlots) return fail(RTC_ERR_UNSUPPORTED, "RAY_DEPTH above 62 is not supported");
    // the Whitted kernel keeps its recursion in a per-thread stack of kWhittedStack entries (course_device.cuh)
    if (ray_depth > kMaxWhittedDepth && s->host.dialect == DIALECT_HW2)
        return fail(RTC_ERR_UNSUPPORTED, "hw2 dialect: RAY_DEPTH above 32 is not supported");
    if (width >= 0) s->host.cam.width = (unsigned)width;
    if (height >= 0) s->host.cam.height = (unsigned)height;
    if (samples >= 0) s->host.samples = (unsigned)samples;
    if (ray_depth >= 0) s->host.ray_depth = (unsigned)ray_depth;
    return RTC_OK;
}
int rtc_scene_prim_order(const rtc_scene* s, int32_t* out) {
    if (!s || !out) return fail(RTC_ERR_ARG, "null argument");
    for (size_t i = 0; i < s->host.prims.size(); ++i) out[i] = s->host.prims[i].orig;
    return RTC_OK;
}
int rtc_scene_prims(const rtc_scene* s, int32_t* tm, float* d) {
    if (!s || !tm || !d) return fail(RTC_ERR_ARG, "null argument");
    for (size_t i = 0; i < s->host.prims.size(); ++i) {
        const Primitive& p = s->host.prims[i];
        tm[2 * i] = p.type; tm[2 * i + 1] = p.material;
        float* o = d + 26 * i;
        const float v[26] = {p.col.x, p.col.y, p.col.z, p.emission.x, p.emission.y, p.emission.z, p.pos.x, p.pos.y, p.pos.z,
                             p.rot.x, p.rot.y, p.rot.z, p.rot.w, p.ior, p.d0.x, p.d0.y, p.d0.z, p.d1.x, p.d1.y, p.d1.z,
                             p.d2.x, p.d2.y, p.d2.z, 0.f, 0.f, 0.f};
        std::memcpy(o, v, sizeof v);
    }
    return RTC_OK;
}
int rtc_scene_nodes(const rtc_scene* s, float* aabb, uint32_t* links) {
    if (!s || !aabb || !links) return fail(RTC_ERR_ARG, "null argument");
    for (size_t i = 0; i < s->host.nodes.size(); ++i) {
        const RefNode& n = s->host.nodes[i];
        const float b[6] = {n.box.mn.x, n.box.mn.y, n.box.mn.z, n.box.mx.x, n.box.mx.y, n.box.mx.z};
        std::memcpy(aabb + 6 * i, b, sizeof b);
        links[4 * i] = n.left; links[4 * i + 1] = n.right; links[4 * i + 2] = n.first; links[4 * i + 3] = n.count;
    }
    return RTC_OK;
}
uint32_t rtc_scene_root(const rtc_scene* s) { return s ? s->host.root : 0; }
void rtc_set_traversal(rtc_scene* s, int mode) { if (s) s->traversal = mode == RTC_TRAVERSAL_REFTREE ? 1 : 0; }
int rtc_set_batch_paths(rtc_scene* s, uint64_t paths) {
    if (!s) return fail(RTC_ERR_ARG, "null scene");
    s->batch_paths = paths ? paths : kDefaultBatchPaths;
    if (s->batch_paths > (1ull << 28)) s->batch_paths = 1ull << 28;
    return RTC_OK;
}

// ------------------------------------------------------------------ probes (host buffers)
// Scene::RayIntersection for a batch of rays whose arrays are ALREADY on the scene's device (3 floats per origin /
// direction / normal): the kernels of the render path on pooled scratch buffers, asynchronous on `stream`.
int rtc_intersect_dev(rtc_scene* s, long n, const float* o_dev, const float* d_dev, int32_t* id_dev, float* t_dev,
                      float* normal_dev, int32_t* interior_dev, int mode, void* stream) {
    int rc = need_device(s);
    if (rc) return rc;
    if (n < 0 || !o_dev || !d_dev || !id_dev || !t_dev || !normal_dev || !interior_dev) return fail(RTC_ERR_ARG, "bad argument");
    if (n == 0) return RTC_OK;
    if ((uint64_t)n > (1ull << 28)) return fail(RTC_ERR_ARG, "too many rays in one call (limit 2^28)");
    rtc_scene::Probe& pb = s->probe;
    CU(pb.ray[0].ensure((size_t)n)); CU(pb.ray[1].ensure((size_t)n));
    CU(pb.hit.ensure((size_t)n)); CU(pb.tq.ensure((size_t)n * kTraverseQueueWords)); CU(pb.q.ensure(4));   // q: rays (front, back = 0), traverse count, cursor
    cudaStream_t st = (cudaStream_t)stream;
    PathSoA P{pb.ray[0].p, pb.ray[1].p, nullptr};
    HitSoA H{pb.hit.p};
    uint32_t* q = pb.q.p;
    CU(cudaMemsetAsync(q, 0, 4 * sizeof(uint32_t), st));
    DevScene S;
    if ((rc = arena_begin(s, st, &S))) return rc;
    LaunchCtx c{st, s->sms};
    // the same kernels as the render path: rays into the float4 queue layout, extend, read back
    launch_pack_rays(c, n, o_dev, d_dev, P, q);
    if (mode == RTC_TRAVERSAL_REFTREE) launch_extend_reftree(c, S, P, H, q, (uint32_t)n);
    else {
        launch_pre(c, S, P, H, q, (uint32_t)n, pb.tq.p, q + 2);
        launch_traverse(c, S, P, H, (uint32_t)n, pb.tq.p, q + 2, q + 3, false, s->stats.p);
    }
    launch_unpack_hits(c, S, n, P, H, id_dev, t_dev, normal_dev, interior_dev);
    if ((rc = arena_end(s, st))) return rc;
    CU(cudaGetLastError());
    return RTC_OK;
}
// host-buffer form: two copies in, one kernel chain, four copies out, on buffers that are allocated once and grow
int rtc_intersect(const rtc_scene* cs, long n, const float* o, const float* d, int32_t* id, float* t, float* normal,
                  int32_t* interior, int mode) {
    rtc_scene* s = const_cast<rtc_scene*>(cs);
    int rc = need_device(s);
    if (rc) return rc;
    if (n < 0 || !o || !d || !id || !t || !normal || !interior) return fail(RTC_ERR_ARG, "bad argument");
    if (n == 0) return RTC_OK;
    if ((uint64_t)n > (1ull << 28)) return fail(RTC_ERR_ARG, "too many rays in one call (limit 2^28)");
    rtc_scene::Probe& pb = s->probe;
    const size_t N = (size_t)n;
    CU(pb.fin[0].ensure(3 * N)); CU(pb.fin[1].ensure(3 * N));
    CU(pb.fout[0].ensure(N)); CU(pb.fout[1].ensure(3 * N));
    CU(pb.iout[0].ensure(N)); CU(pb.iout[1].ensure(N));
    CU(cudaMemcpyAsync(pb.fin[0].p, o, 3 * N * sizeof(float), cudaMemcpyHostToDevice, nullptr));
    CU(cudaMemcpyAsync(pb.fin[1].p, d, 3 * N * sizeof(float), cudaMemcpyHostToDevice, nullptr));
    if ((rc = rtc_intersect_dev(s, n, pb.fin[0].p, pb.fin[1].p, pb.iout[0].p, pb.fout[0].p, pb.fout[1].p, pb.iout[1].p, mode, nullptr)))
        return rc;
    CU(cudaMemcpyAsync(id, pb.iout[0].p, N * 4, cudaMemcpyDeviceToHost, nullptr));
    CU(cudaMemcpyAsync(t, pb.fout[0].p, N * 4, cudaMemcpyDeviceToHost, nullptr));
    CU(cudaMemcpyAsync(normal, pb.fout[1].p, N * 12, cudaMemcpyDeviceToHost, nullptr));
    CU(cudaMemcpyAsync(interior, pb.iout[1].p, N * 4, cudaMemcpyDeviceToHost, nullptr));
    CU(cudaStreamSynchronize(nullptr));
    return RTC_OK;
}
int rtc_primitive_intersect(const rtc_scene* cs, int prim, long n, const float* o, const float* d, int32_t* hit, float* t,
                            float* normal, int32_t* interior) {
    rtc_scene* s = const_cast<rtc_scene*>(cs);   // arena_end records on the scene's event
    int rc = need_device(s);
    if (rc) return rc;
    if (n < 0 || prim < 0 || prim >= (int)s->host.prims.size() || !o || !d || !hit || !t || !normal || !interior)
        return fail(RTC_ERR_ARG, "bad argument");
    if (n == 0) return RTC_OK;
    Staged st;
    float* od = st.in(o, 3 * (size_t)n); NEED(od);
    float* dd = st.in(d, 3 * (size_t)n); NEED(dd);
    int32_t* hd = st.out<int32_t>((size_t)n); NEED(hd);
    float* td = st.out<float>((size_t)n); NEED(td);
    float* nd = st.out<float>(3 * (size_t)n); NEED(nd);
    int32_t* ind = st.out<int32_t>((size_t)n); NEED(ind);
    DevScene S;
    if ((rc = arena_begin(s, nullptr, &S))) return rc;
    launch_primitive_batch(LaunchCtx{nullptr, s->sms}, S, (uint32_t)prim, n, od, dd, hd, td, nd, ind);
    if ((rc = arena_end(s, nullptr))) return rc;
    CU(cudaGetLastError());
    CU(cudaMemcpy(hit, hd, (size_t)n * 4, cudaMemcpyDeviceToHost));
    CU(cudaMemcpy(t, td, (size_t)n * 4, cudaMemcpyDeviceToHost));
    CU(cudaMemcpy(normal, nd, (size_t)n * 12, cudaMemcpyDeviceToHost));
    CU(cudaMemcpy(interior, ind, (size_t)n * 4, cudaMemcpyDeviceToHost));
    return RTC_OK;
}
int rtc_camera_rays(const rtc_scene* cs, long n, const float* xy, float* o, float* d) {
    rtc_scene* s = const_cast<rtc_scene*>(cs);   // arena_end records on the scene's event
    int rc = need_device(s);
    if (rc) return rc;
    if (n < 0 || !xy || !o || !d) return fail(RTC_ERR_ARG, "bad argument");
    if (n == 0) return RTC_OK;
    Staged st;
    float* xd = st.in(xy, 2 * (size_t)n); NEED(xd);
    float* od = st.out<float>(3 * (size_t)n); NEED(od);
    float* dd = st.out<float>(3 * (size_t)n); NEED(dd);
    DevScene S;
    if ((rc = arena_begin(s, nullptr, &S))) return rc;
    launch_camera_batch(LaunchCtx{nullptr, s->sms}, S, n, xd, od, dd);
    if ((rc = arena_end(s, nullptr))) return rc;
    CU(cudaGetLastError());
    CU(cudaMemcpy(o, od, (size_t)n * 12, cudaMemcpyDeviceToHost));
    CU(cudaMemcpy(d, dd, (size_t)n * 12, cudaMemcpyDeviceToHost));
    return RTC_OK;
}
int rtc_mix_pdf(const rtc_scene* cs, long n, const float* x, const float* nrm, const float* d, float* pdf) {
    rtc_scene* s = const_cast<rtc_scene*>(cs);   // arena_end records on the scene's event
    int rc = need_device(s);
    if (rc) return rc;
    if (n < 0 || !x || !nrm || !d || !pdf) return fail(RTC_ERR_ARG, "bad argument");
    if (n == 0) return RTC_OK;
    Staged st;
    float* xd = st.in(x, 3 * (size_t)n); NEED(xd);
    float* nd = st.in(nrm, 3 * (size_t)n); NEED(nd);
    float* dd = st.in(d, 3 * (size_t)n); NEED(dd);
    float* pd = st.out<float>((size_t)n); NEED(pd);
    DevScene S;
    if ((rc = arena_begin(s, nullptr, &S))) return rc;
    launch_pdf_batch(LaunchCtx{nullptr, s->sms}, S, n, xd, nd, dd, pd);
    if ((rc = arena_end(s, nullptr))) return rc;
    CU(cudaGetLastError());
    CU(cudaMemcpy(pdf, pd, (size_t)n * 4, cudaMemcpyDeviceToHost));
    return RTC_OK;
}
int rtc_mix_sample(const rtc_scene* cs, long n, const float* x, const float* nrm, uint32_t seed, uint32_t sample,
                   uint32_t bounce, float* dir) {
    rtc_scene* s = const_cast<rtc_scene*>(cs);   // arena_end records on the scene's event
    int rc = need_device(s);
    if (rc) return rc;
    if (n < 0 || !x || !nrm || !dir) return fail(RTC_ERR_ARG, "bad argument");
    if (n == 0) return RTC_OK;
    Staged st;
    float* xd = st.in(x, 3 * (size_t)n); NEED(xd);
    float* nd = st.in(nrm, 3 * (size_t)n); NEED(nd);
    float* dd = st.out<float>(3 * (size_t)n); NEED(dd);
    DevScene S;
    if ((rc = arena_begin(s, nullptr, &S))) return rc;
    launch_sample_batch(LaunchCtx{nullptr, s->sms}, S, n, xd, nd, seed, sample, bounce, dd);
    if ((rc = arena_end(s, nullptr))) return rc;
    CU(cudaGetLastError());
    CU(cudaMemcpy(dir, dd, (size_t)n * 12, cudaMemcpyDeviceToHost));
    return RTC_OK;
}
int rtc_tonemap_u8(const rtc_scene* s, long npix, const float* rgb, uint8_t* out) {
    int rc = need_device(s);
    if (rc) return rc;
    if (npix < 0 || !rgb || !out) return fail(RTC_ERR_ARG, "bad argument");
    if (npix == 0) return RTC_OK;
    Staged st;
    float* rd = st.in(rgb, 3 * (size_t)npix); NEED(rd);
    uint8_t* od = st.out<uint8_t>(3 * (size_t)npix); NEED(od);
    LaunchCtx c{nullptr, s->sms};
    launch_tonemap(c, rd, (uint32_t)(3 * npix), od);
    CU(cudaGetLastError());
    CU(cudaMemcpy(out, od, 3 * (size_t)npix, cudaMemcpyDeviceToHost));
    return RTC_OK;
}

// ------------------------------------------------------------------ render
int rtc_render_accumulate(rtc_scene* s, uint32_t seed, uint32_t sample_begin, uint32_t sample_count, float* accum_dev,
                          void* stream) {
    int rc = need_device(s);
    if (rc) return rc;
    const uint64_t npix = (uint64_t)s->host.cam.width * s->host.cam.height;
    const uint64_t total = npix * sample_count;
    if (total == 0) return RTC_OK;   // an empty frame (no DIMENSIONS) or an empty sample range: nothing to add
    if (!accum_dev) return fail(RTC_ERR_ARG, "null accumulation buffer");
    cudaStream_t user = (cudaStream_t)stream;
    DevScene S;
    if (s->host.dialect <= DIALECT_HW2) {
        // hw1 / hw2: ONE deterministic frame = sample 0.  A range that holds sample 0 adds the colour once, any
        // other range adds nothing, so that sample ranges split over several devices still sum to one frame.
        if (sample_begin > 0) return RTC_OK;
        if ((rc = arena_begin(s, user, &S))) return rc;
        LaunchCtx c{user, s->sms};
        if (s->host.dialect == DIALECT_HW1) launch_raycast_hw1(c, S, accum_dev);
        else launch_whitted_hw2(c, S, accum_dev);
        s->launches++;
        if ((rc = arena_end(s, user))) return rc;
        CU(cudaGetLastError());
        return RTC_OK;
    }
    // the float4 pixel sums of this render: two buffers used alternately, so that two renders may be in flight on
    // two streams; a third waits for the first to have been folded
    const int a4 = s->accum4_next;
    s->accum4_next ^= 1;
    DevBuf<float4>& accum4 = s->accum4[a4];
    CU(accum4.ensure(npix));
    CU(cudaStreamWaitEvent(user, s->accum4_idle[a4], 0));
    CU(cudaMemsetAsync(accum4.p, 0, npix * sizeof(float4), user));
    if ((rc = arena_begin(s, user, &S))) return rc;
    if ((rc = fork_lanes(s, user))) return rc;
    unsigned used = 0;
    if ((rc = render_paths(s, S, seed, PathMap{nullptr, (uint32_t)npix, sample_begin}, total, accum4.p, &used))) return rc;
    if ((rc = join_lanes(s, used, user))) return rc;
    launch_fold(LaunchCtx{user, s->sms}, accum4.p, accum_dev, (uint32_t)npix);
    s->launches++;
    CU(cudaEventRecord(s->accum4_idle[a4], user));
    if ((rc = arena_end(s, user))) return rc;
    CU(cudaGetLastError());
    return RTC_OK;
}
int rtc_render_counters(rtc_scene* s, void* stream, uint64_t out[8]) {
    int rc = need_device(s);
    if (rc) return rc;
    if (!out) return fail(RTC_ERR_ARG, "null argument");
    CU(cudaStreamSynchronize((cudaStream_t)stream));
    CU(sync_lanes(s));
    unsigned long long h[8];
    CU(cudaMemcpy(h, s->stats.p, sizeof h, cudaMemcpyDeviceToHost));
    for (int i = 0; i < 8; ++i) out[i] = h[i];
    out[2] = s->launches;
    return RTC_OK;
}
int rtc_traverse_lanes(rtc_scene* s, void* stream, uint64_t out[8]) {
    int rc = need_device(s);
    if (rc) return rc;
    if (!out) return fail(RTC_ERR_ARG, "null argument");
    CU(cudaStreamSynchronize((cudaStream_t)stream));
    CU(sync_lanes(s));
    unsigned long long h[8];
    CU(cudaMemcpy(h, s->stats.p + 8, sizeof h, cudaMemcpyDeviceToHost));
    for (int i = 0; i < 8; ++i) out[i] = h[i];
    return RTC_OK;
}
int rtc_render_reset_counters(rtc_scene* s) {
    int rc = need_device(s);
    if (rc) return rc;
    CU(cudaMemset(s->stats.p, 0, kStatWords * sizeof(unsigned long long)));
    s->launches = 0;
    return RTC_OK;
}
int rtc_render_resolve(rtc_scene* s, const float* accum_dev, uint32_t total_samples, uint8_t* rgb_dev, void* stream) {
    int rc = need_device(s);
    if (rc) return rc;
    if (!accum_dev || !rgb_dev || total_samples == 0) return fail(RTC_ERR_ARG, "bad argument");
    LaunchCtx c{(cudaStream_t)stream, s->sms};
    uint32_t nvalues = 3u * s->host.cam.width * s->host.cam.height;
    if (s->host.dialect == DIALECT_HW1) launch_resolve_flat(c, accum_dev, 1.f / (float)total_samples, nvalues, rgb_dev);
    else launch_resolve(c, accum_dev, 1.f / (float)total_samples, nvalues, rgb_dev);  // 1.f / samples * sum, src/scene.cpp:201
    s->launches++;
    CU(cudaGetLastError());
    return RTC_OK;
}
int rtc_render_sum(rtc_scene* s, uint32_t seed, uint32_t sample_begin, uint32_t sample_count, float* sum_host) {
    int rc = need_device(s);
    if (rc) return rc;
    if (!sum_host) return fail(RTC_ERR_ARG, "null argument");
    size_t nvalues = 3 * (size_t)s->host.cam.width * s->host.cam.height;
    if (nvalues == 0) return RTC_OK;
    CU(s->accum.ensure(nvalues));
    CU(cudaMemset(s->accum.p, 0, nvalues * sizeof(float)));
    if ((rc = rtc_render_accumulate(s, seed, sample_begin, sample_count, s->accum.p, nullptr))) return rc;
    CU(cudaMemcpy(sum_host, s->accum.p, nvalues * sizeof(float), cudaMemcpyDeviceToHost));
    return RTC_OK;
}
int rtc_render_u8(rtc_scene* s, uint32_t seed, uint8_t* rgb_host) {
    int rc = need_device(s);
    if (rc) return rc;
    if (!rgb_host) return fail(RTC_ERR_ARG, "null argument");
    uint32_t samples;
    if ((rc = frame_samples(s, &samples))) return rc;
    size_t nvalues = 3 * (size_t)s->host.cam.width * s->host.cam.height;
    if (nvalues == 0) return RTC_OK;   // no DIMENSIONS: the reference writes a PPM header and no pixels
    CU(s->accum.ensure(nvalues));
    CU(s->rgb.ensure(nvalues));
    if ((rc = render_frame(s, seed, samples, s->accum.p, s->rgb.p, nullptr))) return rc;
    CU(cudaMemcpy(rgb_host, s->rgb.p, nvalues, cudaMemcpyDeviceToHost));
    return RTC_OK;
}
int rtc_render_ppm(rtc_scene* s, uint32_t seed, const char* out_path) {
    if (!s || !out_path) return fail(RTC_ERR_ARG, "null argument");
    std::vector<uint8_t> img(3 * (size_t)s->host.cam.width * s->host.cam.height);
    int rc = rtc_render_u8(s, seed, img.data());
    return rc ? rc : write_ppm(out_path, s->host.cam.width, s->host.cam.height, img);
}

// ------------------------------------------------------------------ adaptive sampling
// Passes over the still-active 8x8 tiles: every active tile renders samples [n, target) -- the even ones into one
// half-sum buffer, the odd ones into the other, one render_paths call each, so that small passes run on two lanes at
// once -- then k_adaptive_tiles measures the tiles' error from the two halves and lists the tiles (and their pixels) that
// go on to target = min(2 target, max).  The length of the next pixel list is the one read back per pass.
static_assert(kAdaptiveTile == RTC_ADAPTIVE_TILE, "rt_kernels.h and rtc_b200.h disagree on the tile size");
namespace {
uint32_t adaptive_tiles(uint32_t width, uint32_t height) {
    return ((width + kAdaptiveTile - 1) / kAdaptiveTile) * ((height + kAdaptiveTile - 1) / kAdaptiveTile);
}
// The pass loop of an adaptive render of the tiles shard, shard + nshards, ... of the frame on context `c` (its device
// current), on stream `user`: it leaves the half sums of those tiles' pixels in c->adaptive.half and their sample counts
// in c->adaptive.tile_n, and adds its passes, paths and tiles stopped to st[0], st[1] and st[3].  A shard without a tile
// does nothing.
int adaptive_passes(rtc_scene* c, cudaStream_t user, uint32_t shard, uint32_t nshards, uint32_t seed, float tolerance,
                    uint32_t min_samples, uint32_t smax, uint64_t st[4]) {
    const uint32_t width = c->host.cam.width, height = c->host.cam.height;
    const uint32_t npix = width * height, ntiles = adaptive_tiles(width, height);
    if (shard >= ntiles) return RTC_OK;
    const uint32_t shard_tiles = (ntiles - shard + nshards - 1) / nshards;
    // the pixels of the shard's tiles: whole tiles, less what the partial tiles of the last column and row lack (a loop
    // over the edge tiles, not over all of them: this runs on the host before every render)
    constexpr uint32_t T = kAdaptiveTile;
    const uint32_t tiles_x = (width + T - 1) / T, tiles_y = ntiles / tiles_x;
    const uint32_t wl = width - (tiles_x - 1) * T, hl = height - (tiles_y - 1) * T;   // size of the last column / row
    uint32_t shard_pix = T * T * shard_tiles;
    if (wl < T)
        for (uint32_t ty = 0; ty < tiles_y; ++ty)
            if ((ty * tiles_x + tiles_x - 1) % nshards == shard) shard_pix -= (T - wl) * T;
    if (hl < T)
        for (uint32_t tx = 0; tx < tiles_x; ++tx)
            if (((tiles_y - 1) * tiles_x + tx) % nshards == shard) shard_pix -= (T - hl) * (tx + 1 < tiles_x ? T : wl);
    int rc;
    rtc_scene::Adaptive& ad = c->adaptive;
    for (auto& b : ad.half) CU(b.ensure(npix));
    for (auto& b : ad.tiles) CU(b.ensure(ntiles));
    for (auto& b : ad.pixels) CU(b.ensure(npix));
    CU(ad.tile_n.ensure(ntiles));
    CU(ad.counts.ensure(4));
    CU(ad.counts_host.ensure(2));
    LaunchCtx lc{user, c->sms};
    for (auto& b : ad.half) CU(cudaMemsetAsync(b.p, 0, npix * sizeof(float4), user));
    CU(cudaMemsetAsync(ad.counts.p, 0, 4 * sizeof(uint32_t), user));
    DevScene S;
    if ((rc = arena_begin(c, user, &S))) return rc;
    // every tile of the shard is active with n = 0; lists of pass 0 in set 0
    launch_adaptive_tiles(lc, nullptr, nullptr, width, height, nullptr, shard_tiles, 0, 0.f, 0.f, tolerance, ADAPTIVE_FIRST, ad.tile_n.p,
                          ad.tiles[0].p, ad.pixels[0].p, ad.counts.p, shard, nshards);
    c->launches++;
    uint32_t active_tiles = shard_tiles, active_pix = shard_pix, n = 0, target = min_samples < smax ? min_samples : smax;
    int cur = 0;
    for (;;) {
        ++st[0];
        if ((rc = fork_lanes(c, user))) return rc;
        unsigned used = 0;
        for (uint32_t h = 0; h < 2; ++h) {   // h = 0: the even samples of [n, target) into half 0, h = 1: the odd ones
            const uint32_t first = n + ((n ^ h) & 1u);
            if (first >= target) continue;
            const uint64_t total = (uint64_t)((target - first + 1) / 2) * active_pix;
            if ((rc = render_paths(c, S, seed, PathMap{ad.pixels[cur].p, active_pix, first}, total, ad.half[h].p, &used))) return rc;
            st[1] += total;
        }
        if ((rc = join_lanes(c, used, user))) return rc;
        n = target;
        const bool last = n == smax;
        const int nxt = cur ^ 1;
        if (!last) CU(cudaMemsetAsync(ad.counts.p + 2 * nxt, 0, 2 * sizeof(uint32_t), user));
        launch_adaptive_tiles(lc, ad.half[0].p, ad.half[1].p, width, height, ad.tiles[cur].p, active_tiles, n, 1.f / (float)((n + 1) / 2),
                              1.f / (float)(n / 2), tolerance, last ? ADAPTIVE_LAST : ADAPTIVE_DECIDE, ad.tile_n.p, ad.tiles[nxt].p,
                              ad.pixels[nxt].p, ad.counts.p + 2 * nxt, 0, 1);
        c->launches++;
        if (last) break;
        CU(cudaMemcpyAsync(ad.counts_host.p, ad.counts.p + 2 * nxt, 2 * sizeof(uint32_t), cudaMemcpyDeviceToHost, user));
        CU(cudaStreamSynchronize(user));
        st[3] += active_tiles - ad.counts_host.p[0];
        active_tiles = ad.counts_host.p[0];
        active_pix = ad.counts_host.p[1];
        if (active_tiles == 0) break;
        cur = nxt;
        target = (uint64_t)2 * target < smax ? 2 * target : smax;
    }
    return arena_end(c, user);
}
}  // namespace
int rtc_render_adaptive(rtc_scene* s, uint32_t seed, float tolerance, uint32_t min_samples, uint32_t max_samples,
                        uint8_t* rgb_host, float* halves_host, uint32_t* spp_host, uint64_t stats[4]) {
    if (!s) return fail(RTC_ERR_ARG, "null scene");
    if (!std::isfinite(tolerance) || tolerance < 0.f) return fail(RTC_ERR_ARG, "tolerance must be finite and >= 0");
    if (min_samples < 2) return fail(RTC_ERR_ARG, "min_samples must be at least 2");
    int rc = need_device(s);
    if (rc) return rc;
    const uint32_t width = s->host.cam.width, height = s->host.cam.height;
    const uint32_t npix = width * height;
    const uint32_t ntiles = adaptive_tiles(width, height);
    uint64_t st[4] = {0, 0, 0, 0};   // passes, paths, tiles, tiles stopped below the maximum
    if (stats) std::memcpy(stats, st, sizeof st);
    if (npix == 0) return RTC_OK;
    const size_t nvalues = 3 * (size_t)npix;
    CU(s->rgb.ensure(nvalues));
    if (s->host.dialect <= DIALECT_HW2) {
        // hw1 / hw2: the one deterministic frame, resolved as rtc_render_u8 does; it is the "even" half, spp = 1
        CU(s->accum.ensure(nvalues));
        if ((rc = render_frame(s, seed, 1, s->accum.p, s->rgb.p, nullptr))) return rc;
        if (rgb_host) CU(cudaMemcpy(rgb_host, s->rgb.p, nvalues, cudaMemcpyDeviceToHost));
        if (halves_host) {
            std::vector<float> frame(nvalues);
            CU(cudaMemcpy(frame.data(), s->accum.p, nvalues * sizeof(float), cudaMemcpyDeviceToHost));
            for (size_t i = 0; i < npix; ++i)
                for (int c = 0; c < 3; ++c) { halves_host[6 * i + c] = frame[3 * i + c]; halves_host[6 * i + 3 + c] = 0.f; }
        }
        if (spp_host) for (size_t i = 0; i < npix; ++i) spp_host[i] = 1;
        const uint64_t one[4] = {1, npix, ntiles, 0};
        if (stats) std::memcpy(stats, one, sizeof one);
        return RTC_OK;
    }
    const uint32_t smax = max_samples ? max_samples : s->host.samples;
    if (smax == 0) return fail(RTC_ERR_ARG, "scene has SAMPLES 0");
    cudaStream_t user = nullptr;
    st[2] = ntiles;
    if ((rc = adaptive_passes(s, user, 0, 1, seed, tolerance, min_samples, smax, st))) return rc;
    rtc_scene::Adaptive& ad = s->adaptive;
    CU(ad.halves.ensure(halves_host ? 6 * (size_t)npix : 0));
    CU(ad.spp.ensure(spp_host ? npix : 0));
    launch_resolve_adaptive(LaunchCtx{user, s->sms}, ad.half[0].p, ad.half[1].p, ad.tile_n.p, width, npix, s->rgb.p,
                            halves_host ? ad.halves.p : nullptr, spp_host ? ad.spp.p : nullptr);
    s->launches++;
    CU(cudaGetLastError());
    if (rgb_host) CU(cudaMemcpy(rgb_host, s->rgb.p, nvalues, cudaMemcpyDeviceToHost));
    if (halves_host) CU(cudaMemcpy(halves_host, ad.halves.p, 6 * (size_t)npix * sizeof(float), cudaMemcpyDeviceToHost));
    if (spp_host) CU(cudaMemcpy(spp_host, ad.spp.p, (size_t)npix * sizeof(uint32_t), cudaMemcpyDeviceToHost));
    CU(cudaStreamSynchronize(user));
    if (stats) std::memcpy(stats, st, sizeof st);
    return RTC_OK;
}

// ------------------------------------------------------------------ denoising
namespace {
int check_strength(float strength) {
    if (!std::isfinite(strength) || strength < 0.f) return fail(RTC_ERR_ARG, "strength must be finite and >= 0");
    return RTC_OK;
}
// The filter on the half sums and sample counts in halves_dev / spp_dev (the layout of k_resolve_adaptive's optional
// outputs, every spp >= 2), on the default stream: k_denoise_prep, then k_denoise_nlm unless strength is 0 (then the
// image is that of the mean u, as rtc_render_adaptive resolves it).  Copies the image and the mean to the host.
int denoise(rtc_scene* s, const float* halves_dev, const uint32_t* spp_dev, float strength, uint8_t* rgb_host, float* mean_host) {
    const uint32_t width = s->host.cam.width, height = s->host.cam.height, npix = width * height;
    rtc_scene::Denoise& dn = s->denoise;
    CU(dn.u.ensure(3 * (size_t)npix));
    CU(dn.d.ensure(npix));
    CU(dn.v.ensure(npix));
    CU(s->rgb.ensure(3 * (size_t)npix));
    const LaunchCtx lc{nullptr, s->sms};
    const bool filter = strength > 0.f;
    launch_denoise_prep(lc, halves_dev, spp_dev, npix, dn.u.p, dn.d.p, dn.v.p, filter ? nullptr : s->rgb.p);
    s->launches++;
    CU(cudaGetLastError());
    if (filter) {
        CU(dn.mean.ensure(3 * (size_t)npix));
        // k^2 saturates instead of overflowing: the weights are then all 1 where the patches' variance is non-zero
        CU(launch_denoise_nlm(lc, dn.u.p, dn.d.p, dn.v.p, width, height, 0, (height + kDenoiseTileH - 1) / kDenoiseTileH, 0,
                              std::fmin(strength * strength, FLT_MAX), dn.mean.p, s->rgb.p));
        s->launches++;
    }
    if (rgb_host) CU(cudaMemcpy(rgb_host, s->rgb.p, 3 * (size_t)npix, cudaMemcpyDeviceToHost));
    if (mean_host) CU(cudaMemcpy(mean_host, filter ? dn.mean.p : dn.u.p, 3 * (size_t)npix * sizeof(float), cudaMemcpyDeviceToHost));
    CU(cudaStreamSynchronize(nullptr));
    return RTC_OK;
}
}  // namespace
int rtc_denoise(rtc_scene* s, const float* halves_host, const uint32_t* spp_host, float strength, uint8_t* rgb_host, float* mean_host) {
    if (!s) return fail(RTC_ERR_ARG, "null scene");
    if (!halves_host || !spp_host) return fail(RTC_ERR_ARG, "null halves or spp");
    int rc = check_strength(strength);
    if (rc) return rc;
    if (s->host.dialect <= DIALECT_HW2) return fail(RTC_ERR_ARG, "hw1 / hw2 scenes have no noise to filter");
    const size_t npix = (size_t)s->host.cam.width * s->host.cam.height;
    for (size_t i = 0; i < npix; ++i)
        if (spp_host[i] < 2) return fail(RTC_ERR_ARG, "every pixel needs at least 2 samples (pixel " + std::to_string(i) + ")");
    if ((rc = need_device(s))) return rc;
    if (npix == 0) return RTC_OK;
    rtc_scene::Adaptive& ad = s->adaptive;
    CU(ad.halves.ensure(6 * npix));
    CU(ad.spp.ensure(npix));
    CU(cudaMemcpy(ad.halves.p, halves_host, 6 * npix * sizeof(float), cudaMemcpyHostToDevice));
    CU(cudaMemcpy(ad.spp.p, spp_host, npix * sizeof(uint32_t), cudaMemcpyHostToDevice));
    return denoise(s, ad.halves.p, ad.spp.p, strength, rgb_host, mean_host);
}
int rtc_render_denoised(rtc_scene* s, uint32_t seed, float tolerance, uint32_t min_samples, uint32_t max_samples, float strength,
                        uint8_t* rgb_host, float* mean_host, uint64_t stats[4]) {
    if (!s) return fail(RTC_ERR_ARG, "null scene");
    int rc = check_strength(strength);
    if (rc) return rc;
    const uint32_t width = s->host.cam.width, height = s->host.cam.height, npix = width * height;
    if (s->host.dialect <= DIALECT_HW2) {
        // the one deterministic frame, unfiltered: rtc_render_adaptive's, whose mean is the frame it leaves in s->accum
        if ((rc = rtc_render_adaptive(s, seed, tolerance, min_samples, max_samples, rgb_host, nullptr, nullptr, stats))) return rc;
        if (mean_host && npix) CU(cudaMemcpy(mean_host, s->accum.p, 3 * (size_t)npix * sizeof(float), cudaMemcpyDeviceToHost));
        return RTC_OK;
    }
    if (!std::isfinite(tolerance) || tolerance < 0.f) return fail(RTC_ERR_ARG, "tolerance must be finite and >= 0");
    if (min_samples < 2) return fail(RTC_ERR_ARG, "min_samples must be at least 2");
    const uint32_t smax = max_samples ? max_samples : s->host.samples;
    if (smax < 2) return fail(RTC_ERR_ARG, "the maximum sample count must be at least 2");
    if ((rc = need_device(s))) return rc;
    uint64_t st[4] = {0, 0, 0, 0};   // passes, paths, tiles, tiles stopped below the maximum
    if (stats) std::memcpy(stats, st, sizeof st);
    if (npix == 0) return RTC_OK;
    st[2] = adaptive_tiles(width, height);
    if ((rc = adaptive_passes(s, nullptr, 0, 1, seed, tolerance, min_samples, smax, st))) return rc;
    rtc_scene::Adaptive& ad = s->adaptive;
    CU(s->rgb.ensure(3 * (size_t)npix));
    CU(ad.halves.ensure(6 * (size_t)npix));
    CU(ad.spp.ensure(npix));
    launch_resolve_adaptive(LaunchCtx{nullptr, s->sms}, ad.half[0].p, ad.half[1].p, ad.tile_n.p, width, npix, s->rgb.p, ad.halves.p,
                            ad.spp.p);
    s->launches++;
    CU(cudaGetLastError());
    if ((rc = denoise(s, ad.halves.p, ad.spp.p, strength, rgb_host, mean_host))) return rc;
    if (stats) std::memcpy(stats, st, sizeof st);
    return RTC_OK;
}

int rtc_scene_upload_async(rtc_scene* s, uint64_t* h2d_bytes) {
    int rc = need_device(s);
    if (rc) return rc;
    return upload_scene_async(s, h2d_bytes);
}

// ------------------------------------------------------------------ frames in flight
// One frame = what run.sh does with a scene that is already parsed: flattened scene host -> HBM, render, resolve,
// 8-bit image HBM -> host.  rtc_frame_begin queues all of it (no host synchronisation: the upload on the copy stream
// into the arena that is not being read, the kernels on the slot's stream, the image into a pinned buffer),
// rtc_frame_end waits for the slot and hands the image over.  Two slots: frame i + 1 is queued before frame i is collected.
int rtc_frame_begin(rtc_scene* s, uint32_t seed, int slot, uint64_t* h2d_bytes) {
    int rc = need_device(s);
    if (rc) return rc;
    if (slot < 0 || slot > 1) return fail(RTC_ERR_ARG, "frame slot must be 0 or 1");
    rtc_scene::Frame& f = s->frames[slot];
    if (f.busy) return fail(RTC_ERR_ARG, "frame slot is in flight: call rtc_frame_end first");
    uint32_t samples;
    if ((rc = frame_samples(s, &samples))) return rc;
    const size_t nvalues = 3 * (size_t)s->host.cam.width * s->host.cam.height;
    CU(f.stream.ensure());
    CU(f.done.ensure());
    CU(f.accum.ensure(nvalues));
    CU(f.rgb.ensure(nvalues));
    CU(f.host.ensure(nvalues));
    if ((rc = upload_scene_async(s, h2d_bytes))) return rc;
    if (nvalues) {
        if ((rc = render_frame(s, seed, samples, f.accum.p, f.rgb.p, f.stream))) return rc;
        CU(cudaMemcpyAsync(f.host.p, f.rgb.p, nvalues, cudaMemcpyDeviceToHost, f.stream));
    }
    CU(cudaEventRecord(f.done, f.stream));
    f.busy = true;
    return RTC_OK;
}
int rtc_frame_end(rtc_scene* s, int slot, uint8_t* rgb_host) {
    int rc = need_device(s);
    if (rc) return rc;
    if (slot < 0 || slot > 1) return fail(RTC_ERR_ARG, "frame slot must be 0 or 1");
    rtc_scene::Frame& f = s->frames[slot];
    if (!f.busy) return fail(RTC_ERR_ARG, "frame slot is not in flight");
    CU(cudaEventSynchronize(f.done));
    f.busy = false;
    const size_t nvalues = 3 * (size_t)s->host.cam.width * s->host.cam.height;
    if (rgb_host && nvalues) std::memcpy(rgb_host, f.host.p, nvalues);
    return RTC_OK;
}
// resolve a device accumulation buffer and start the 8-bit image on its way to a pinned host buffer (slot 0's);
// rtc_host_image_wait collects the last one.  Used by multi-process renders after their reduce.
int rtc_resolve_to_host_async(rtc_scene* s, const float* accum_dev, uint32_t total_samples, void* stream) {
    int rc = need_device(s);
    if (rc) return rc;
    rtc_scene::Frame& f = s->frames[0];
    const size_t nvalues = 3 * (size_t)s->host.cam.width * s->host.cam.height;
    if (!accum_dev || nvalues == 0) return fail(RTC_ERR_ARG, "bad argument");
    CU(f.stream.ensure());
    CU(f.done.ensure());
    CU(f.rgb.ensure(nvalues));
    CU(f.host.ensure(nvalues));
    cudaStream_t user = (cudaStream_t)stream;
    // the previous image must have left the device buffer before it is resolved into again
    CU(cudaStreamWaitEvent(user, f.done, 0));
    if ((rc = rtc_render_resolve(s, accum_dev, total_samples, f.rgb.p, user))) return rc;
    CU(s->resolved.ensure());
    CU(cudaEventRecord(s->resolved, user));
    CU(cudaStreamWaitEvent(f.stream, s->resolved, 0));
    CU(cudaMemcpyAsync(f.host.p, f.rgb.p, nvalues, cudaMemcpyDeviceToHost, f.stream));
    CU(cudaEventRecord(f.done, f.stream));
    return RTC_OK;
}
int rtc_host_image_wait(rtc_scene* s, uint8_t* rgb_host) {
    int rc = need_device(s);
    if (rc) return rc;
    rtc_scene::Frame& f = s->frames[0];
    if (!f.done) return fail(RTC_ERR_ARG, "no image in flight");
    CU(cudaEventSynchronize(f.done));
    const size_t nvalues = 3 * (size_t)s->host.cam.width * s->host.cam.height;
    if (rgb_host && nvalues) std::memcpy(rgb_host, f.host.p, nvalues);
    return RTC_OK;
}

// ------------------------------------------------------------------ one call, several devices
// Scene::Render uses the whole machine (src/scene.cpp:212 omp_set_num_threads(hardware_concurrency)); so does this:
// the samples are split over `ndev` devices of this process (disjoint Philox streams, rtc_render_accumulate), every
// device renders into its own buffer, and the first device sums them over NVLink peer access and resolves
// (k_resolve_peers).  A device may be listed more than once (its share is then rendered twice as often).
namespace {
rtc_scene* replica_on(rtc_scene* s, int device, int ordinal) {
    // the ordinal-th use of `device` in the list: the scene itself serves the first use of its own device
    int seen = 0;
    if (device == s->device) { if (ordinal == 0) return s; seen = 1; }
    for (const auto& r : s->replicas)
        if (r->device == device) { if (seen == ordinal) return r.get(); ++seen; }
    auto r = std::make_unique<rtc_scene>(s->host_ptr);
    r->traversal = s->traversal;
    r->batch_paths = s->batch_paths;
    if (finish_scene(r.get(), device) != RTC_OK) return nullptr;
    s->replicas.push_back(std::move(r));
    return s->replicas.back().get();
}
// issue(i) for i in [0, n): i >= 1 on host threads of their own, i = 0 on the caller's; the first failure in list order
// is returned, with its message
int fan_out(int n, const std::function<int(int)>& issue) {
    std::vector<int> rcs((size_t)n, RTC_OK);
    std::vector<std::string> errs((size_t)n);
    std::vector<std::thread> workers;
    for (int i = 1; i < n; ++i)
        workers.emplace_back([&, i] { rcs[i] = issue(i); if (rcs[i]) errs[i] = g_error; });   // g_error is per thread
    rcs[0] = issue(0);
    for (std::thread& w : workers) w.join();
    for (int i = 0; i < n; ++i)
        if (rcs[i]) return i == 0 ? rcs[0] : fail(rcs[i], errs[i]);
    return RTC_OK;
}
// Whether device `head` (current) reads the memory of device `dev` in place: the same device, or peer access, which
// this enables.  When it cannot, the caller copies what it needs over with stage_peer.
int peer_mapped(int head, int dev, bool* mapped) {
    *mapped = head == dev;
    if (*mapped) return RTC_OK;
    int can = 0;
    CU(cudaDeviceCanAccessPeer(&can, head, dev));
    if (can) {
        cudaError_t e = cudaDeviceEnablePeerAccess(dev, 0);
        if (e == cudaSuccess || e == cudaErrorPeerAccessAlreadyEnabled) { cudaGetLastError(); *mapped = true; }
        else cudaGetLastError();
    }
    return RTC_OK;
}
// a copy on device `head` (current) of `bytes` at `src` on device `dev`, queued on `st` and held by `staged`; null when
// it cannot be made (the message in rtc_last_error)
void* stage_peer(int head, int dev, const void* src, size_t bytes, cudaStream_t st, std::vector<DevBuf<unsigned char>>& staged) {
    staged.emplace_back();
    cudaError_t e = staged.back().ensure(bytes);
    if (e == cudaSuccess) e = cudaMemcpyPeerAsync(staged.back().p, head, src, dev, bytes, st);
    if (e != cudaSuccess) { fail(RTC_ERR_CUDA, std::string("staging a peer copy: ") + cudaGetErrorString(e)); return nullptr; }
    return staged.back().p;
}
// the context of every entry of `devices`: this scene for the first use of its own device, replicas for the others
int device_contexts(rtc_scene* s, const int* devices, int ndev, std::vector<rtc_scene*>& ctx) {
    ctx.assign((size_t)ndev, nullptr);
    std::vector<int> uses(64, 0);
    for (int i = 0; i < ndev; ++i) {
        if (devices[i] < 0 || devices[i] >= 64) return fail(RTC_ERR_ARG, "bad device index");
        ctx[i] = replica_on(s, devices[i], uses[devices[i]]++);
        if (!ctx[i]) return RTC_ERR_CUDA;
    }
    return RTC_OK;
}
}  // namespace
int rtc_render_u8_multi(rtc_scene* s, const int* devices, int ndev, uint32_t seed, uint8_t* rgb_host, float* sum_host) {
    int rc = need_device(s);
    if (rc) return rc;
    if (!devices || ndev < 1 || ndev > kMaxPeers || !rgb_host) return fail(RTC_ERR_ARG, "bad argument");
    uint32_t samples;
    if ((rc = frame_samples(s, &samples))) return rc;
    const size_t nvalues = 3 * (size_t)s->host.cam.width * s->host.cam.height;
    if (nvalues == 0) return RTC_OK;
    // the first listed device reduces: make it this scene's device or a replica there
    std::vector<rtc_scene*> ctx;
    if ((rc = device_contexts(s, devices, ndev, ctx))) return rc;
    PeerAccums A;
    std::memset(&A, 0, sizeof A);
    A.n = ndev;
    rtc_scene* head = ctx[0];
    // every device renders its sample range into its own buffer on its own stream; the ~30 launches of a device's
    // share are issued by a host thread of its own (one thread issuing for 8 devices took 1.1 of a 3.9 ms frame)
    auto issue = [&](int i) -> int {
        rtc_scene* c = ctx[i];
        CU(cudaSetDevice(c->device));
        CU(c->multi_stream.ensure());
        CU(c->multi_done.ensure());
        CU(c->accum.ensure(nvalues));
        CU(cudaMemsetAsync(c->accum.p, 0, nvalues * sizeof(float), c->multi_stream));
        const uint32_t lo = (uint32_t)((uint64_t)i * samples / ndev), hi = (uint32_t)((uint64_t)(i + 1) * samples / ndev);
        int r = rtc_render_accumulate(c, seed, lo, hi - lo, c->accum.p, c->multi_stream);
        if (r) return r;
        CU(cudaEventRecord(c->multi_done, c->multi_stream));
        return RTC_OK;
    };
    if ((rc = fan_out(ndev, issue))) return rc;
    for (int i = 0; i < ndev; ++i) A.p[i] = ctx[i]->accum.p;
    // the head device reads the others' buffers in place (peer access), or copies them over when it cannot
    CU(cudaSetDevice(head->device));
    std::vector<DevBuf<unsigned char>> staged;
    for (int i = 1; i < ndev; ++i) {
        rtc_scene* c = ctx[i];
        CU(cudaStreamWaitEvent(head->multi_stream, c->multi_done, 0));
        bool mapped;
        if ((rc = peer_mapped(head->device, c->device, &mapped))) return rc;
        if (mapped) continue;
        void* p = stage_peer(head->device, c->device, A.p[i], nvalues * sizeof(float), head->multi_stream, staged);
        if (!p) return RTC_ERR_CUDA;
        A.p[i] = (const float*)p;
    }
    CU(head->rgb.ensure(nvalues));
    float* sum_dev = nullptr;
    if (sum_host) { CU(head->frames[1].accum.ensure(nvalues)); sum_dev = head->frames[1].accum.p; }
    LaunchCtx lc{head->multi_stream, head->sms};
    if (head->host.dialect == DIALECT_HW1) {
        // hw1 writes colours as they are: only the device that holds sample 0 has any
        launch_resolve_flat(lc, A.p[0], 1.f, (uint32_t)nvalues, head->rgb.p);
        if (sum_dev) CU(cudaMemcpyAsync(sum_dev, A.p[0], nvalues * sizeof(float), cudaMemcpyDeviceToDevice, head->multi_stream));
    } else launch_resolve_peers(lc, A, 1.f / (float)samples, (uint32_t)nvalues, head->rgb.p, sum_dev);
    head->launches++;
    CU(cudaGetLastError());
    CU(cudaMemcpyAsync(rgb_host, head->rgb.p, nvalues, cudaMemcpyDeviceToHost, head->multi_stream));
    if (sum_host) CU(cudaMemcpyAsync(sum_host, sum_dev, nvalues * sizeof(float), cudaMemcpyDeviceToHost, head->multi_stream));
    CU(cudaStreamSynchronize(head->multi_stream));
    staged.clear();   // while the head device is current
    CU(cudaSetDevice(s->device));
    return RTC_OK;
}
int rtc_render_ppm_multi(rtc_scene* s, const int* devices, int ndev, uint32_t seed, const char* out_path) {
    if (!s || !out_path) return fail(RTC_ERR_ARG, "null argument");
    std::vector<uint8_t> img(3 * (size_t)s->host.cam.width * s->host.cam.height);
    int rc = rtc_render_u8_multi(s, devices, ndev, seed, img.data(), nullptr);
    return rc ? rc : write_ppm(out_path, s->host.cam.width, s->host.cam.height, img);
}

// Adaptive sampling on several devices: tile t of the frame belongs to devices[t % ndev], and every device runs the
// pass loop of rtc_render_adaptive on its own tiles, on its own stream and host thread.  A tile's decisions read only its
// own half sums, so the devices do not talk to each other until devices[0] resolves every pixel from its owner's
// half sums and tile counts (k_resolve_adaptive_peers).
namespace {
int check_adaptive_multi_args(float tolerance, uint32_t min_samples, const int* devices, int ndev) {
    if (!std::isfinite(tolerance) || tolerance < 0.f) return fail(RTC_ERR_ARG, "tolerance must be finite and >= 0");
    if (min_samples < 2) return fail(RTC_ERR_ARG, "min_samples must be at least 2");
    if (!devices || ndev < 1 || ndev > kMaxPeers) return fail(RTC_ERR_ARG, "devices must list 1 to 16 entries");
    for (int i = 0; i < ndev; ++i)
        if (devices[i] < 0 || devices[i] >= 64) return fail(RTC_ERR_ARG, "bad device index");
    return RTC_OK;
}
// The passes of every entry of `ctx`: entry i runs adaptive_passes on the tiles i, i + n, ... on its multi_stream and a
// host thread of its own, and records its multi_done.  st: passes (the most of any entry), paths, tiles, tiles stopped.
int adaptive_passes_multi(const std::vector<rtc_scene*>& ctx, uint32_t seed, float tolerance, uint32_t min_samples, uint32_t smax,
                          uint32_t ntiles, uint64_t st[4]) {
    const int ndev = (int)ctx.size();
    std::vector<std::array<uint64_t, 4>> dev_st((size_t)ndev, std::array<uint64_t, 4>{0, 0, 0, 0});
    auto issue = [&](int i) -> int {
        rtc_scene* c = ctx[i];
        CU(cudaSetDevice(c->device));
        CU(c->multi_stream.ensure());
        CU(c->multi_done.ensure());
        int r = adaptive_passes(c, c->multi_stream, (uint32_t)i, (uint32_t)ndev, seed, tolerance, min_samples, smax, dev_st[i].data());
        if (r) return r;
        CU(cudaEventRecord(c->multi_done, c->multi_stream));
        return RTC_OK;
    };
    int rc = fan_out(ndev, issue);
    if (rc) return rc;
    st[2] = ntiles;
    for (const auto& d : dev_st) {
        st[0] = std::max(st[0], d[0]);
        st[1] += d[1];
        st[3] += d[3];
    }
    return RTC_OK;
}
// The owners' half sums of the image rows [row0, row0 + nrows) and their whole tile counts, for entry `c` (its device
// current) after adaptive_passes_multi: c's multi_stream waits for every other owner, and reads its buffers in place
// (peer access) or copies those rows over (held by `staged`).
int owner_halves(rtc_scene* c, const std::vector<rtc_scene*>& ctx, uint32_t width, uint32_t row0, uint32_t nrows, uint32_t ntiles,
                 std::vector<DevBuf<unsigned char>>& staged, PeerHalves* P) {
    std::memset(P, 0, sizeof *P);
    P->n = (int)ctx.size();
    const int owners = ctx.size() < ntiles ? (int)ctx.size() : (int)ntiles;   // the others have no tile
    const size_t first = (size_t)row0 * width, npix = (size_t)nrows * width;
    for (int i = 0; i < owners; ++i) {
        rtc_scene* o = ctx[i];
        P->a[i] = o->adaptive.half[0].p + first;
        P->b[i] = o->adaptive.half[1].p + first;
        P->tile_n[i] = o->adaptive.tile_n.p;
        if (o == c) continue;
        CU(cudaStreamWaitEvent(c->multi_stream, o->multi_done, 0));
        bool mapped;
        int rc = peer_mapped(c->device, o->device, &mapped);
        if (rc) return rc;
        if (mapped) continue;
        void* a = stage_peer(c->device, o->device, P->a[i], npix * sizeof(float4), c->multi_stream, staged);
        void* b = a ? stage_peer(c->device, o->device, P->b[i], npix * sizeof(float4), c->multi_stream, staged) : nullptr;
        void* n = b ? stage_peer(c->device, o->device, P->tile_n[i], ntiles * sizeof(uint32_t), c->multi_stream, staged) : nullptr;
        if (!n) return RTC_ERR_CUDA;
        P->a[i] = (const float4*)a;
        P->b[i] = (const float4*)b;
        P->tile_n[i] = (const uint32_t*)n;
    }
    return RTC_OK;
}
}  // namespace
int rtc_render_adaptive_multi(rtc_scene* s, const int* devices, int ndev, uint32_t seed, float tolerance, uint32_t min_samples,
                              uint32_t max_samples, uint8_t* rgb_host, float* halves_host, uint32_t* spp_host, uint64_t stats[4]) {
    if (!s) return fail(RTC_ERR_ARG, "null scene");
    int rc = check_adaptive_multi_args(tolerance, min_samples, devices, ndev);
    if (rc) return rc;
    rc = need_device(s);
    if (rc) return rc;
    const uint32_t width = s->host.cam.width, height = s->host.cam.height;
    const uint32_t npix = width * height, ntiles = adaptive_tiles(width, height);
    uint64_t st[4] = {0, 0, 0, 0};   // passes (the most of any device), paths, tiles, tiles stopped below the maximum
    if (stats) std::memcpy(stats, st, sizeof st);
    if (npix == 0) return RTC_OK;
    const size_t nvalues = 3 * (size_t)npix;
    if (s->host.dialect <= DIALECT_HW2) {
        // one deterministic frame, not split: rtc_render_adaptive on the first listed device
        rtc_scene* head = replica_on(s, devices[0], 0);
        if (!head) return RTC_ERR_CUDA;
        if ((rc = rtc_render_adaptive(head, seed, tolerance, min_samples, max_samples, rgb_host, halves_host, spp_host, stats)))
            return rc;
        CU(cudaSetDevice(s->device));
        return RTC_OK;
    }
    const uint32_t smax = max_samples ? max_samples : s->host.samples;
    if (smax == 0) return fail(RTC_ERR_ARG, "scene has SAMPLES 0");
    std::vector<rtc_scene*> ctx;
    if ((rc = device_contexts(s, devices, ndev, ctx))) return rc;
    rtc_scene* head = ctx[0];
    if ((rc = adaptive_passes_multi(ctx, seed, tolerance, min_samples, smax, ntiles, st))) return rc;
    // the head device reads the owners' half sums and tile counts in place (peer access), or copies them over
    CU(cudaSetDevice(head->device));
    PeerHalves P;
    std::vector<DevBuf<unsigned char>> staged;
    if ((rc = owner_halves(head, ctx, width, 0, height, ntiles, staged, &P))) return rc;
    rtc_scene::Adaptive& ad = head->adaptive;
    CU(head->rgb.ensure(nvalues));
    CU(ad.halves.ensure(halves_host ? 6 * (size_t)npix : 0));
    CU(ad.spp.ensure(spp_host ? npix : 0));
    launch_resolve_adaptive_peers(LaunchCtx{head->multi_stream, head->sms}, P, width, npix, head->rgb.p,
                                  halves_host ? ad.halves.p : nullptr, spp_host ? ad.spp.p : nullptr);
    head->launches++;
    CU(cudaGetLastError());
    if (rgb_host) CU(cudaMemcpyAsync(rgb_host, head->rgb.p, nvalues, cudaMemcpyDeviceToHost, head->multi_stream));
    if (halves_host)
        CU(cudaMemcpyAsync(halves_host, ad.halves.p, 6 * (size_t)npix * sizeof(float), cudaMemcpyDeviceToHost, head->multi_stream));
    if (spp_host) CU(cudaMemcpyAsync(spp_host, ad.spp.p, (size_t)npix * sizeof(uint32_t), cudaMemcpyDeviceToHost, head->multi_stream));
    CU(cudaStreamSynchronize(head->multi_stream));
    staged.clear();   // while the head device is current
    CU(cudaSetDevice(s->device));
    if (stats) std::memcpy(stats, st, sizeof st);
    return RTC_OK;
}

// Denoising on several devices: rtc_render_adaptive_multi's passes, then entry i filters the image rows of the tile rows
// [i T / n, (i + 1) T / n) of k_denoise_nlm's grid (T = ceil(H / kDenoiseTileH)), so that the bands together are the
// one-device grid block for block.  It reads the rows it filters and kDenoiseApron more on either side from the tiles'
// owners where they lie, on its own stream and host thread, and copies its rows of the image and the mean to the host.
int rtc_render_denoised_multi(rtc_scene* s, const int* devices, int ndev, uint32_t seed, float tolerance, uint32_t min_samples,
                              uint32_t max_samples, float strength, uint8_t* rgb_host, float* mean_host, float* halves_host,
                              uint32_t* spp_host, uint64_t stats[4]) {
    if (!s) return fail(RTC_ERR_ARG, "null scene");
    int rc = check_strength(strength);
    if (rc) return rc;
    if ((rc = check_adaptive_multi_args(tolerance, min_samples, devices, ndev))) return rc;
    const bool deterministic = s->host.dialect <= DIALECT_HW2;
    const uint32_t smax = max_samples ? max_samples : s->host.samples;
    if (!deterministic && smax < 2) return fail(RTC_ERR_ARG, "the maximum sample count must be at least 2");
    if ((rc = need_device(s))) return rc;
    const uint32_t width = s->host.cam.width, height = s->host.cam.height;
    const uint32_t npix = width * height, ntiles = adaptive_tiles(width, height);
    uint64_t st[4] = {0, 0, 0, 0};
    if (stats) std::memcpy(stats, st, sizeof st);
    if (npix == 0) return RTC_OK;
    if (deterministic) {
        // rtc_render_denoised's unfiltered frame on the first listed device, with rtc_render_adaptive's halves and spp
        rtc_scene* head = replica_on(s, devices[0], 0);
        if (!head) return RTC_ERR_CUDA;
        if ((rc = rtc_render_adaptive(head, seed, tolerance, min_samples, max_samples, rgb_host, halves_host, spp_host, stats))) return rc;
        if (mean_host) CU(cudaMemcpy(mean_host, head->accum.p, 3 * (size_t)npix * sizeof(float), cudaMemcpyDeviceToHost));
        CU(cudaSetDevice(s->device));
        return RTC_OK;
    }
    std::vector<rtc_scene*> ctx;
    if ((rc = device_contexts(s, devices, ndev, ctx))) return rc;
    if ((rc = adaptive_passes_multi(ctx, seed, tolerance, min_samples, smax, ntiles, st))) return rc;
    const bool filter = strength > 0.f;
    const float k2 = std::fmin(strength * strength, FLT_MAX);   // as in denoise()
    const uint32_t tile_rows = (height + kDenoiseTileH - 1) / kDenoiseTileH;
    auto band = [&](int i) -> int {
        rtc_scene* c = ctx[i];
        CU(cudaSetDevice(c->device));
        const cudaStream_t st_i = c->multi_stream;
        const LaunchCtx lc{st_i, c->sms};
        std::vector<DevBuf<unsigned char>> staged;   // freed on return, with c's device current
        PeerHalves P;
        int r;
        if (i == 0 && (halves_host || spp_host)) {
            // the whole half sums and spp, as rtc_render_adaptive_multi gathers them
            rtc_scene::Adaptive& ad = c->adaptive;
            CU(c->rgb.ensure(3 * (size_t)npix));
            CU(ad.halves.ensure(halves_host ? 6 * (size_t)npix : 0));
            CU(ad.spp.ensure(spp_host ? npix : 0));
            if ((r = owner_halves(c, ctx, width, 0, height, ntiles, staged, &P))) return r;
            launch_resolve_adaptive_peers(lc, P, width, npix, c->rgb.p, halves_host ? ad.halves.p : nullptr, spp_host ? ad.spp.p : nullptr);
            c->launches++;
            CU(cudaGetLastError());
            if (halves_host) CU(cudaMemcpyAsync(halves_host, ad.halves.p, 6 * (size_t)npix * sizeof(float), cudaMemcpyDeviceToHost, st_i));
            if (spp_host) CU(cudaMemcpyAsync(spp_host, ad.spp.p, (size_t)npix * sizeof(uint32_t), cudaMemcpyDeviceToHost, st_i));
        }
        const uint32_t t0 = (uint32_t)((uint64_t)i * tile_rows / ndev), t1 = (uint32_t)((uint64_t)(i + 1) * tile_rows / ndev);
        if (t0 < t1) {
            const uint32_t y0 = t0 * kDenoiseTileH, y1 = std::min(height, t1 * kDenoiseTileH);
            const uint32_t apron = kDenoiseApron;
            const uint32_t r0 = y0 > apron ? y0 - apron : 0, r1 = std::min(height, y1 + apron);
            const size_t prep_pix = (size_t)(r1 - r0) * width, out_pix = (size_t)(y1 - y0) * width, out_first = (size_t)(y0 - r0) * width;
            rtc_scene::Denoise& dn = c->denoise;
            CU(dn.u.ensure(3 * prep_pix));
            CU(dn.d.ensure(prep_pix));
            CU(dn.v.ensure(prep_pix));
            CU(dn.mean.ensure(3 * out_pix));
            CU(c->rgb.ensure(3 * out_pix));
            if ((r = owner_halves(c, ctx, width, r0, r1 - r0, ntiles, staged, &P))) return r;
            launch_denoise_prep_peers(lc, P, width, r0, r1 - r0, dn.u.p, dn.d.p, dn.v.p, filter ? nullptr : c->rgb.p, (uint32_t)out_first,
                                      (uint32_t)out_pix);
            c->launches++;
            CU(cudaGetLastError());
            if (filter) {
                CU(launch_denoise_nlm(lc, dn.u.p, dn.d.p, dn.v.p, width, height, t0, t1 - t0, r0, k2, dn.mean.p, c->rgb.p));
                c->launches++;
            }
            if (rgb_host) CU(cudaMemcpyAsync(rgb_host + 3 * (size_t)y0 * width, c->rgb.p, 3 * out_pix, cudaMemcpyDeviceToHost, st_i));
            if (mean_host)
                CU(cudaMemcpyAsync(mean_host + 3 * (size_t)y0 * width, filter ? dn.mean.p : dn.u.p + 3 * out_first,
                                   3 * out_pix * sizeof(float), cudaMemcpyDeviceToHost, st_i));
        }
        CU(cudaStreamSynchronize(st_i));
        return RTC_OK;
    };
    if ((rc = fan_out(ndev, band))) return rc;
    CU(cudaSetDevice(s->device));
    if (stats) std::memcpy(stats, st, sizeof st);
    return RTC_OK;
}

int rtc_set_profiling(rtc_scene* s, int kernel_events, int count_visits) {
    if (!s) return fail(RTC_ERR_ARG, "null scene");
    s->profiling = kernel_events != 0;
    s->count_visits = count_visits != 0;
    return RTC_OK;
}
int rtc_render_profile(rtc_scene* s, void* stream, double ms[4], uint64_t launches[4], int reset) {
    int rc = need_device(s);
    if (rc) return rc;
    if (!ms || !launches) return fail(RTC_ERR_ARG, "null argument");
    CU(cudaStreamSynchronize((cudaStream_t)stream));
    CU(sync_lanes(s));
    s->collect_spans();
    for (int i = 0; i < 4; ++i) { ms[i] = s->prof_ms[i]; launches[i] = s->prof_launches[i]; }
    if (reset) for (int i = 0; i < 4; ++i) { s->prof_ms[i] = 0; s->prof_launches[i] = 0; }
    return RTC_OK;
}

void rtc_philox4x32_10(const uint32_t ctr[4], const uint32_t key[2], uint32_t out[4]) {
    uint32_t c0 = ctr[0], c1 = ctr[1], c2 = ctr[2], c3 = ctr[3], k0 = key[0], k1 = key[1];
    for (int r = 0; r < 10; ++r) {
        uint64_t p0 = (uint64_t)0xD2511F53u * c0, p1 = (uint64_t)0xCD9E8D57u * c2;
        uint32_t n0 = (uint32_t)(p1 >> 32) ^ c1 ^ k0, n1 = (uint32_t)p1, n2 = (uint32_t)(p0 >> 32) ^ c3 ^ k1, n3 = (uint32_t)p0;
        c0 = n0; c1 = n1; c2 = n2; c3 = n3;
        k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
    }
    out[0] = c0; out[1] = c1; out[2] = c2; out[3] = c3;
}

}  // extern "C"
