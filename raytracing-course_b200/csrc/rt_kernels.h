// rt_kernels.h -- host-callable launchers of the kernels in rt_kernels.cu.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "device_scene.h"

namespace rtc {

// Words per traverse-queue entry: an entry is the ray itself -- (origin, bits(slot | entered root children)) (direction,
// closest-plane distance) -- written by the kernel that makes the ray while it is still in registers, so that a refill
// of k_traverse is ONE coalesced round trip instead of two dependent ones (the queue word, then the scattered path
// state: measured 10.58 -> 10.25 ms, profiles/r02_experiments.md).
constexpr uint32_t kTraverseQueueWords = 8;

struct LaunchCtx {
    cudaStream_t stream;
    int sms;  // multiprocessor count of the device (grid sizing)
};

// camera rays of one wavefront batch + their pre_step (planes, index root, traverse queue)
void launch_generate(const LaunchCtx& c, const DevScene& S, PathSoA P, HitSoA H, uint32_t* q, uint32_t* tq, uint32_t* tq_count,
                     uint64_t first_path, uint32_t count, uint32_t seed, uint32_t sample_begin);
// the same over a pixel list: path p = pixel plist[p % npix], sample sample_first + 2 (p / npix)
void launch_generate_list(const LaunchCtx& c, const DevScene& S, PathSoA P, HitSoA H, uint32_t* q, uint32_t* tq, uint32_t* tq_count,
                          uint64_t first_path, uint32_t count, uint32_t seed, const uint32_t* plist, uint32_t npix, uint32_t sample_first);
// adaptive sampling (rtc_render_adaptive): square tiles of kAdaptiveTile pixels a side (= RTC_ADAPTIVE_TILE), one warp each
constexpr uint32_t kAdaptiveTile = 8;
static_assert(kAdaptiveTile * kAdaptiveTile == 64, "k_adaptive_tiles: one warp per tile, two pixels per lane");
enum { ADAPTIVE_FIRST = 0, ADAPTIVE_DECIDE = 1, ADAPTIVE_LAST = 2 };
// per active tile: record n, decide (mode), append the kept tiles and their pixels to the next lists; ADAPTIVE_FIRST
// visits the ntiles tiles shard, shard + nshards, shard + 2 nshards, ... of the frame
void launch_adaptive_tiles(const LaunchCtx& c, const float4* A, const float4* B, uint32_t width, uint32_t height,
                           const uint32_t* tiles_in, uint32_t ntiles, uint32_t n, float inv_a, float inv_b, float tau, int mode,
                           uint32_t* tile_n, uint32_t* tiles_out, uint32_t* pixels_out, uint32_t* counts_out, uint32_t shard,
                           uint32_t nshards);
// u8 image (and optionally the half sums, 6 floats per pixel, and the samples per pixel) from the even / odd sums
void launch_resolve_adaptive(const LaunchCtx& c, const float4* A, const float4* B, const uint32_t* tile_n, uint32_t width, uint32_t npix,
                             uint8_t* out, float* halves, uint32_t* spp);
// denoising (rtc_denoise, rtc_render_denoised; DESIGN.md "Denoising"): the fixed constants of the non-local-means rule
// -- search window (2R+1)^2, patch (2F+1)^2, box (2S+1)^2 that smooths the variance estimate, variance cancellation
// alpha, epsilon -- and the output tile of one block
constexpr int kDenoiseRadius = 7, kDenoisePatch = 3, kDenoiseVarRadius = 1;
constexpr float kDenoiseAlpha = 1.f, kDenoiseEps = 1e-8f;
constexpr int kDenoiseTileW = 32, kDenoiseTileH = 16;
// the rows of u, D and V beyond its tile that a filter block reads: the window and the patch, then the box around V
constexpr int kDenoiseApron = kDenoiseRadius + kDenoisePatch + kDenoiseVarRadius;
// per pixel from the half sums (6 floats) and spp (>= 2): the linear mean u (3 floats), D = display(u) and the variance
// estimate V (float4, w unused); rgb (optional) = the 8-bit image of u
void launch_denoise_prep(const LaunchCtx& c, const float* halves, const uint32_t* spp, uint32_t npix, float* u, float4* D, float4* V,
                         uint8_t* rgb);
// the filter with k2 = strength^2 on the tile rows [tile_row0, tile_row0 + tile_rows) of kDenoiseTileH pixels: mean (3
// floats per pixel) and its 8-bit image, from the first row of the band on; u, D and V hold the image rows [buf_row0,
// min(height, band end + kDenoiseApron)).  The whole frame: (0, ceil(height / kDenoiseTileH), 0).
cudaError_t launch_denoise_nlm(const LaunchCtx& c, const float* u, const float4* D, const float4* V, uint32_t width, uint32_t height,
                               uint32_t tile_row0, uint32_t tile_rows, uint32_t buf_row0, float k2, float* mean, uint8_t* rgb);
// Scene::RayIntersection for the rays of queue P (fills H): launch_pre then launch_traverse
// (index BVH), or launch_extend_reftree alone (the reference-tree twin).
void launch_pre(const LaunchCtx& c, const DevScene& S, PathSoA P, HitSoA H, const uint32_t* qcount, uint32_t max_count,
                uint32_t* tq, uint32_t* tq_count);
void launch_traverse(const LaunchCtx& c, const DevScene& S, PathSoA P, HitSoA H, uint32_t max_count, const uint32_t* tq,
                     const uint32_t* tq_count, uint32_t* cursor, bool count_visits, unsigned long long* stats);
void launch_extend_reftree(const LaunchCtx& c, const DevScene& S, PathSoA P, HitSoA H, const uint32_t* q, uint32_t cap);
// shading of queue P with hits H; survivors go to queue N with their pre_step results in HN / tq
void launch_shade(const LaunchCtx& c, const DevScene& S, PathSoA P, HitSoA H, PathSoA N, HitSoA HN, const uint32_t* qin,
                  uint32_t* qout, uint32_t* tq, uint32_t* tq_count, uint32_t max_count, float4* accum4, uint32_t bounce,
                  uint32_t seed);
// accum += accum4 (xyz): the library's float4 pixel sums into the caller's buffer at the end of a frame
void launch_fold(const LaunchCtx& c, const float4* accum4, float* accum, uint32_t npix);
// the tail of a scene arena, rebuilt on the device after every upload of its head (c_api.cu issue_upload)
void launch_expand_lca(const LaunchCtx& c, uint32_t* lca, const uint4* rmeta, uint32_t n, uint32_t levels);
void launch_expand_boxes(const LaunchCtx& c, const float4* sparse, uint32_t n, float4* ubox);
void launch_fill_identity_rotations(const LaunchCtx& c, float4* rot, uint32_t n);
void launch_expand_palette(const LaunchCtx& c, const float4* palette, const uint16_t* index, uint32_t n, float4* out0, float4* out1);
void launch_tally(const LaunchCtx& c, const uint32_t* q, const uint32_t* tqc, uint32_t ray_depth, unsigned long long* stats);
void launch_resolve(const LaunchCtx& c, const float* accum, float inv_samples, uint32_t nvalues, uint8_t* out);
void launch_tonemap(const LaunchCtx& c, const float* rgb, uint32_t nvalues, uint8_t* out);
// per-device accumulation buffers of one multi-device frame (device pointers valid on the device that launches:
// its own memory or peer-mapped memory), summed in order and resolved to 8 bits
constexpr int kMaxPeers = 16;
struct PeerAccums {
    const float* p[kMaxPeers];
    int n;
};
void launch_resolve_peers(const LaunchCtx& c, const PeerAccums& A, float inv_samples, uint32_t nvalues, uint8_t* out, float* sum);
// per-device half sums and tile counts of one multi-device adaptive render (tile t belongs to device t % n; pointers
// valid on the device that launches), resolved as launch_resolve_adaptive does
struct PeerHalves {
    const float4* a[kMaxPeers];
    const float4* b[kMaxPeers];
    const uint32_t* tile_n[kMaxPeers];
    int n;
};
void launch_resolve_adaptive_peers(const LaunchCtx& c, const PeerHalves& P, uint32_t width, uint32_t npix, uint8_t* out, float* halves,
                                   uint32_t* spp);
// launch_denoise_prep for the image rows [row0, row0 + nrows) of such a render (P.a / P.b point at row row0, P.tile_n at
// the whole tile counts); u, D and V are band-local, rgb (optional) gets the pixels [rgb_first, rgb_first + rgb_count)
// of the band
void launch_denoise_prep_peers(const LaunchCtx& c, const PeerHalves& P, uint32_t width, uint32_t row0, uint32_t nrows, float* u,
                               float4* D, float4* V, uint8_t* rgb, uint32_t rgb_first, uint32_t rgb_count);
void launch_pack_rays(const LaunchCtx& c, long n, const float* o, const float* d, PathSoA P, uint32_t* q);
void launch_unpack_hits(const LaunchCtx& c, const DevScene& S, long n, PathSoA P, HitSoA H, int32_t* id, float* t, float* nrm,
                        int32_t* interior);
void launch_primitive_batch(const LaunchCtx& c, const DevScene& S, uint32_t prim, long n, const float* o, const float* d,
                            int32_t* hit, float* t, float* nrm, int32_t* interior);
void launch_camera_batch(const LaunchCtx& c, const DevScene& S, long n, const float* xy, float* o, float* d);
void launch_pdf_batch(const LaunchCtx& c, const DevScene& S, long n, const float* x, const float* nr, const float* d, float* pdf);
void launch_sample_batch(const LaunchCtx& c, const DevScene& S, long n, const float* x, const float* nr, uint32_t seed,
                         uint32_t sample, uint32_t bounce, float* dir);

// course_kernels.cu: the deterministic dialects, one launch per frame, colour ADDED into accum (3 floats per pixel)
void launch_raycast_hw1(const LaunchCtx& c, const DevScene& S, float* accum);
void launch_whitted_hw2(const LaunchCtx& c, const DevScene& S, float* accum);
void launch_resolve_flat(const LaunchCtx& c, const float* accum, float inv_samples, uint32_t nvalues, uint8_t* out);

}  // namespace rtc
