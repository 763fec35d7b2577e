/*
 * rtc_b200.h -- C-ABI of the B200-native hw5 path tracer hot path (librtc_b200.so).
 *
 * Drop-in boundary for FeggieBoss/raytracing-course hw5: every entry point below replaces one
 * reference interface (cited as file:line under /root/reference/hw5).  Plain pointers and
 * sizes only; no C++/torch types cross this boundary.  All functions return 0 (RTC_OK) or a
 * negative rtc_status; rtc_last_error() gives the message for the calling thread.  There is
 * NO CPU fallback: without a CUDA device every compute entry point fails with
 * RTC_ERR_NO_DEVICE.
 *
 * Buffers named *_host are host pointers, *_dev are device pointers on the scene's device.
 * `stream` is a cudaStream_t passed as void* (NULL = the legacy default stream).
 */
#ifndef RTC_B200_H
#define RTC_B200_H
#include <stdint.h>
#ifdef __cplusplus
extern "C" {
#endif

typedef struct rtc_scene rtc_scene;

typedef enum {
    RTC_OK = 0,
    RTC_ERR_IO = -1,          /* cannot open / read / write a file */
    RTC_ERR_NO_DEVICE = -2,   /* no CUDA device, or device index out of range */
    RTC_ERR_CUDA = -3,        /* a CUDA runtime call failed (message in rtc_last_error) */
    RTC_ERR_ARG = -4,         /* bad argument */
    RTC_ERR_UNSUPPORTED = -5  /* scene exceeds a documented limit (DESIGN.md "Limits") */
} rtc_status;

/* traversal selection for rtc_intersect* and rtc_set_traversal */
#define RTC_TRAVERSAL_INDEX   0  /* index BVH + reference-recursion emulation (default, fast) */
#define RTC_TRAVERSAL_REFTREE 1  /* walks the reference's own BVH node by node (slow, exact twin) */

const char* rtc_last_error(void);
int rtc_version(void);
int rtc_device_count(void);

/* ---- Scene::Load + Scene::InitScene  (src/sceneload.cpp:112-176, src/scene.cpp:7-40,
 *      src/main.cpp:9-15).  Parses the hw5 text format on the host, reproduces the reference's
 *      primitive order and SAH BVH (src/bvh.cpp:99-179), builds the index BVH, and uploads the
 *      flattened SoA scene to `device` (HBM) once.  device < 0: host-only scene (parse/build
 *      only; compute calls fail with RTC_ERR_NO_DEVICE). */
rtc_scene* rtc_scene_load(const char* path, int device);
rtc_scene* rtc_scene_parse(const char* text, long len, int device);
void rtc_scene_free(rtc_scene* s);
/* ---- the earlier snapshots of the same renderer (hw1..hw4 src/scene.cpp Scene::Load / Scene::Render, each
 *      behind its own `run.sh <scene> <out.ppm>`): `dialect` 1..5 selects the vocabulary of the scene
 *      reader and the variant of Scene::RayTrace (1 ray casting, 2 Whitted with point / directional lights,
 *      3 path tracing with uniform-hemisphere sampling, 4 cosine + light mix without triangles, 5 = the two
 *      calls above).  hw1 and hw2 have no samples: the render calls produce the one deterministic frame. */
#define RTC_DIALECT_HW1 1
#define RTC_DIALECT_HW2 2
#define RTC_DIALECT_HW3 3
#define RTC_DIALECT_HW4 4
#define RTC_DIALECT_HW5 5
rtc_scene* rtc_scene_load_dialect(const char* path, int device, int dialect);
rtc_scene* rtc_scene_parse_dialect(const char* text, long len, int device, int dialect);
int rtc_scene_dialect(const rtc_scene* s);
/* re-upload the already built host scene to its device (bench e2e: the per-step H2D copy).
 * returns the number of bytes copied through *h2d_bytes. */
int rtc_scene_upload(rtc_scene* s, uint64_t* h2d_bytes);

/* out: width,height,ray_depth,samples,nprims,nbvh(non-plane prims),nnodes(reference BVH),nlights */
int rtc_scene_info(const rtc_scene* s, uint32_t out[8]);
/* Only the head of the flattened scene travels to the device (rtc_scene_upload*); its tail -- the upper levels of the
 * LCA table, the per-slot exact leaf boxes, identity rotations -- is rebuilt there.  Compares the arena in HBM, byte for
 * byte, with the one the host would have uploaded in full (tests). */
int rtc_scene_arena_check(rtc_scene* s, uint64_t* mismatching_bytes);
/* out: index-BVH nodes, index-BVH depth, reference-BVH depth, units(reference leaves),
 *      device bytes of the scene, LCA table levels, bytes per index node, scene feature bits */
int rtc_scene_stats(const rtc_scene* s, uint64_t out[8]);
/* DIMENSIONS / SAMPLES / RAY_DEPTH overrides (value < 0 keeps the file's) */
int rtc_scene_override(rtc_scene* s, int width, int height, int samples, int ray_depth);
/* final primitive order after std::partition + the BVH sorts (scene.cpp:17, bvh.cpp:129,168):
 * original file index of every slot; and the per-primitive record type,material + 26 floats
 * (col3 emission3 pos3 rot4(xyzw) ior d0(3) d1(3) d2(3) pad3) */
int rtc_scene_prim_order(const rtc_scene* s, int32_t* out_orig_index_host);
int rtc_scene_prims(const rtc_scene* s, int32_t* type_material_host, float* data_host);
/* reference BVH (BVH_t::nodes, bvh.h:30-36) in vector order: aabb_min3 aabb_max3 per node and
 * left,right,first_primitive_id,primitive_count */
int rtc_scene_nodes(const rtc_scene* s, float* aabb_host, uint32_t* links_host);
uint32_t rtc_scene_root(const rtc_scene* s);
void rtc_set_traversal(rtc_scene* s, int mode);

/* ---- Scene::RayIntersection (src/scene.cpp:46-77) = planes + BVH_t::Intersect
 *      (src/bvh.cpp:181-225) + Primitive::Intersect (src/primitives.cpp:14-174), n rays.
 *      o,d: 3 floats per ray.  id = -1 on a miss (t, normal, interior then 0). */
int rtc_intersect(const rtc_scene* s, long n, const float* o_host, const float* d_host,
                  int32_t* id_host, float* t_host, float* normal_host, int32_t* interior_host, int mode);
/* the same with every array already on the scene's device (3 floats per origin / direction / normal), asynchronous
 * on `stream`, on scratch buffers the scene keeps: the form to use at rate (tens of millions of rays per call) */
int rtc_intersect_dev(rtc_scene* s, long n, const float* o_dev, const float* d_dev, int32_t* id_dev, float* t_dev,
                      float* normal_dev, int32_t* interior_dev, int mode, void* stream);
/* ---- Primitive::Intersect (src/primitives.cpp:14-52) of one primitive (final-order id) */
int rtc_primitive_intersect(const rtc_scene* s, int prim, long n, const float* o_host, const float* d_host,
                            int32_t* hit_host, float* t_host, float* normal_host, int32_t* interior_host);
/* ---- Camera::GetToRay (src/scene.cpp:180-187): xy = 2 floats per ray */
int rtc_camera_rays(const rtc_scene* s, long n, const float* xy_host, float* o_host, float* d_host);
/* ---- Distribution::Pdf of Scene::mix_distrib (src/distributions.cpp:401-416, 289-372) */
int rtc_mix_pdf(const rtc_scene* s, long n, const float* x_host, const float* nrm_host, const float* d_host,
                float* pdf_host);
/* ---- Distribution::Sample of Scene::mix_distrib (src/distributions.cpp:385-399, 144-159,
 *      227-269, 318-338) with the Philox stream (seed, pixel = ray index, sample, bounce) */
int rtc_mix_sample(const rtc_scene* s, long n, const float* x_host, const float* nrm_host,
                   uint32_t seed, uint32_t sample, uint32_t bounce, float* dir_host);
/* ---- AcesTonemap + GammaCorrected + Color::toUInts (src/color.cpp:26-49) */
int rtc_tonemap_u8(const rtc_scene* s, long npix, const float* rgb_host, uint8_t* out_host);

/* ---- Scene::Render (src/scene.cpp:205-252) / Scene::Sample (:189-203) / Scene::RayTrace
 *      (:83-178), as a wavefront integrator.
 * rtc_render_accumulate adds, for every pixel, the radiance of samples
 * [sample_begin, sample_begin+sample_count) into accum_dev (3 floats per pixel, row-major,
 * device memory, NOT cleared here).  Samples use disjoint counter-based RNG streams, so N
 * ranks rendering disjoint sample ranges and summing their buffers (NCCL reduce) reproduce
 * the single-GPU image.  Asynchronous on `stream`; counters are valid after
 * rtc_render_counters (which synchronises the stream). */
int rtc_render_accumulate(rtc_scene* s, uint32_t seed, uint32_t sample_begin, uint32_t sample_count,
                          float* accum_dev, void* stream);
/* out: paths, rays (RayIntersection calls), launches (kernels launched), wavefront batches,
 *      index-BVH node visits and (slot 6) primitive tests (only with rtc_set_profiling
 *      count_visits), slot 5 fallback rays, 0 -- totals since
 * the scene was created or rtc_render_reset_counters. */
int rtc_render_counters(rtc_scene* s, void* stream, uint64_t out[8]);
int rtc_render_reset_counters(rtc_scene* s);
/* Warp-execution efficiency of k_traverse's per-warp scheduler (only with count_visits): out[0..3] = warp
 * iterations of kind VISIT / LEAF / FINISH / REFILL, out[4..7] = lanes that took part in them (of 32 each). */
int rtc_traverse_lanes(rtc_scene* s, void* stream, uint64_t out[8]);
/* mean = 1/total_samples * sum ; tonemap ; gamma ; u8 -> rgb_dev (3 bytes per pixel, device) */
int rtc_render_resolve(rtc_scene* s, const float* accum_dev, uint32_t total_samples, uint8_t* rgb_dev, void* stream);
/* whole Scene::Render with the scene's own SAMPLES: host u8 image (3*W*H bytes) */
int rtc_render_u8(rtc_scene* s, uint32_t seed, uint8_t* rgb_host);
/* linear per-pixel radiance SUM over a sample range, copied to the host (parity tests) */
int rtc_render_sum(rtc_scene* s, uint32_t seed, uint32_t sample_begin, uint32_t sample_count, float* sum_host);
/* run.sh <scene> <out.ppm> in one call: "P6\nW H\n255\n" + bytes (src/scene.cpp:206-208,243-251) */
int rtc_render_ppm(rtc_scene* s, uint32_t seed, const char* out_path);
/* ---- adaptive sampling: Scene::Render with a noise threshold instead of a fixed sample count per pixel (single
 *      device).  The frame is cut into RTC_ADAPTIVE_TILE x RTC_ADAPTIVE_TILE tiles (partial at the right and bottom
 *      edges).  Every tile starts with samples [0, n0), n0 = min(min_samples, max); a pass renders [n, target) for each
 *      still-active tile, the even samples into one half sum A and the odd ones into another, B.  A tile then stops when
 *      its error E < tolerance, else it goes on to target = min(2 target, max).  E = the mean over the tile's pixels of
 *      (|D(a_r) - D(b_r)| + |D(a_g) - D(b_g)| + |D(a_b) - D(b_b)|) / 3 with a = A / ceil(n/2), b = B / floor(n/2) and
 *      D = the display value before 8-bit rounding (ACES, gamma 1/2.2); a NaN error keeps the tile.  tolerance = 0
 *      renders max samples everywhere.  Samples use the streams of rtc_render_accumulate: a pixel that took n samples
 *      holds the sums of its samples [0, n).  max_samples = 0: the scene's SAMPLES.  tolerance must be finite and >= 0,
 *      min_samples >= 2 (else RTC_ERR_ARG).  hw1 / hw2 render their one frame: spp = 1, A = the frame, B = 0.
 * stats: passes, paths rendered, tiles, tiles stopped below max_samples.  Every output may be NULL.
 * rgb_host: 3 bytes per pixel, to_u8(aces(1/spp * (A + B))).
 * halves_host: 6 floats per pixel (even-sample sum rgb, odd-sample sum rgb); spp_host: 1 per pixel. */
#define RTC_ADAPTIVE_TILE 8
int rtc_render_adaptive(rtc_scene* s, uint32_t seed, float tolerance, uint32_t min_samples, uint32_t max_samples,
                        uint8_t* rgb_host, float* halves_host, uint32_t* spp_host, uint64_t stats[4]);
/* ---- Scene::Render on several devices of this process (src/scene.cpp:205-252 uses every hardware thread of the
 *      machine, :212): the samples are split over devices[0..ndev) (a device may be listed more than once), each
 *      renders its range into its own buffer, and devices[0] sums them where they lie -- peer access over NVLink --
 *      and resolves to 8 bits in the same kernel.  sum_host (optional, 3 floats per pixel) receives the float sums.
 *      run.sh takes the list from RTC_DEVICES ("0,1,2,3" or "0-7"). */
int rtc_render_u8_multi(rtc_scene* s, const int* devices, int ndev, uint32_t seed, uint8_t* rgb_host, float* sum_host);
int rtc_render_ppm_multi(rtc_scene* s, const int* devices, int ndev, uint32_t seed, const char* out_path);
/* ---- rtc_render_adaptive on several devices of this process.  Tile t (row-major over the frame, the tiles of
 *      rtc_render_adaptive) belongs to devices[t % ndev]; each device runs the passes of rtc_render_adaptive on its own
 *      tiles, and devices[0] resolves every pixel from its owner's half sums over peer access.  A tile's decisions read
 *      only its own half sums and the samples are those of rtc_render_accumulate, so the result is rtc_render_adaptive's
 *      up to float summation order.  A device may be listed more than once; one listed beyond the tile count renders
 *      nothing.  hw1 / hw2 render their one frame on devices[0], as rtc_render_adaptive does.  Arguments and outputs are
 *      those of rtc_render_adaptive; devices must list 1 to 16 indices in 0..63 (else RTC_ERR_ARG, checked before any
 *      device is touched).
 * stats: passes (the most of any device), paths (summed over the devices), tiles (of the frame), tiles stopped below
 *      max_samples (summed over the devices). */
int rtc_render_adaptive_multi(rtc_scene* s, const int* devices, int ndev, uint32_t seed, float tolerance, uint32_t min_samples,
                              uint32_t max_samples, uint8_t* rgb_host, float* halves_host, uint32_t* spp_host, uint64_t stats[4]);
/* ---- denoising: non-local means on the even / odd half sums of a render (Rousselle, Knaus and Zwicker, "Adaptive
 *      Rendering with Non-Local Means Filtering", 2012; DESIGN.md "Denoising").  Per pixel with n >= 2 samples: the mean
 *      u = 1/n (A + B), D = display(u) (ACES, gamma 1/2.2, before 8-bit rounding) and, per channel, the variance estimate
 *      V = ((D(A / ceil(n/2)) - D(B / floor(n/2))) / 2)^2.  The filtered mean of p is the weighted mean of u_q over the
 *      15x15 window around p (q in the image, u_q finite), with w(p,q) = exp(-max(0, d2)), d2 = the mean over a 7x7 patch
 *      (coordinates clamped to the image) and the channels of ((D_p - D_q)^2 - (V_p + min(V_p, V_q))) /
 *      (1e-8 + strength^2 (V_p + V_q)).  A pixel whose mean is not finite keeps it.  strength must be finite and >= 0 (else
 *      RTC_ERR_ARG); 0 is the identity, and the filter does not run.  rgb_host: 3 bytes per pixel, to_u8(aces(filtered
 *      mean)); mean_host (may be NULL): the filtered mean, 3 floats per pixel.
 * rtc_denoise filters halves the caller has, in the layout rtc_render_adaptive and rtc_render_adaptive_multi return
 *      (6 floats and 1 spp per pixel of the scene's frame).  RTC_ERR_ARG, checked before any device call: a null halves or
 *      spp pointer, a bad strength, any spp < 2, a hw1 / hw2 scene (no noise to estimate). */
int rtc_denoise(rtc_scene* s, const float* halves_host, const uint32_t* spp_host, float strength, uint8_t* rgb_host, float* mean_host);
/* rtc_render_denoised runs rtc_render_adaptive's passes and filters the half sums where they lie.  Arguments and stats are
 *      rtc_render_adaptive's; min_samples >= the maximum (max_samples, or SAMPLES when it is 0) renders every pixel at
 *      the maximum in one pass.  A maximum below 2 is RTC_ERR_ARG.  hw1 / hw2 return their one frame unfiltered, and the
 *      frame as the mean. */
int rtc_render_denoised(rtc_scene* s, uint32_t seed, float tolerance, uint32_t min_samples, uint32_t max_samples, float strength,
                        uint8_t* rgb_host, float* mean_host, uint64_t stats[4]);
/* rtc_render_denoised on several devices of this process: the passes of rtc_render_adaptive_multi (tile t belongs to
 *      devices[t % ndev]), then the filter split into bands of rows.  With T = ceil(H / 16) tile rows of the filter,
 *      entry i filters the rows [16 floor(i T / ndev), min(H, 16 floor((i + 1) T / ndev))) -- none when ndev > T -- on
 *      its own device, reading those rows and 11 more on either side from the tiles' owners over peer access (or copies
 *      of those rows when a pair cannot map each other), and writes its rows of rgb_host and mean_host.  The result is
 *      rtc_denoise's on the same half sums, bit for bit.  halves_host / spp_host (optional, rtc_render_adaptive_multi's
 *      layout) are gathered on devices[0]; they are the half sums the filter read.  Arguments, errors and stats are the
 *      union of rtc_render_denoised's and rtc_render_adaptive_multi's, every check before any device call.  hw1 / hw2
 *      return rtc_render_denoised's unfiltered frame, rendered on devices[0]. */
int rtc_render_denoised_multi(rtc_scene* s, const int* devices, int ndev, uint32_t seed, float tolerance, uint32_t min_samples,
                              uint32_t max_samples, float strength, uint8_t* rgb_host, float* mean_host, float* halves_host,
                              uint32_t* spp_host, uint64_t stats[4]);
/* ---- frames in flight: what run.sh does with a parsed scene (flattened scene host -> HBM, render, resolve, 8-bit
 *      image HBM -> host), queued without host synchronisation.  rtc_frame_begin uploads into the arena that is not
 *      being read (rtc_scene_upload_async: on a copy stream, under the kernels of the frame before), renders with the
 *      scene's own SAMPLES on the slot's stream and starts the image on its way to a pinned buffer; rtc_frame_end
 *      waits for the slot and copies the image out.  slot = 0 or 1: two frames may be in flight. */
int rtc_scene_upload_async(rtc_scene* s, uint64_t* h2d_bytes);
int rtc_frame_begin(rtc_scene* s, uint32_t seed, int slot, uint64_t* h2d_bytes);
int rtc_frame_end(rtc_scene* s, int slot, uint8_t* rgb_host);
/* resolve a device accumulation buffer (after a reduce over ranks) and start its 8-bit image towards the host on a
 * stream of its own; rtc_host_image_wait waits for the last one and copies it out (rgb_host may be NULL) */
int rtc_resolve_to_host_async(rtc_scene* s, const float* accum_dev, uint32_t total_samples, void* stream);
int rtc_host_image_wait(rtc_scene* s, uint8_t* rgb_host);
/* Instrumentation (off by default).  kernel_events: bracket every wavefront kernel with CUDA
 * events on the launching stream; count_visits: use the extend-kernel variant that counts
 * index-BVH node visits and primitive tests (counters 4 and 6 of rtc_render_counters).
 * rtc_render_profile synchronises `stream` and returns total milliseconds and launch counts per
 * kernel class: 0 generate, 1 extend (Scene::RayIntersection), 2 shade, 3 other. */
int rtc_set_profiling(rtc_scene* s, int kernel_events, int count_visits);
int rtc_render_profile(rtc_scene* s, void* stream, double ms[4], uint64_t launches[4], int reset);
/* wavefront batch size in paths (0 = default); takes effect at the next render call */
int rtc_set_batch_paths(rtc_scene* s, uint64_t paths);

/* Philox4x32-10 block (the RNG of the render path), host-side, for known-answer tests */
void rtc_philox4x32_10(const uint32_t ctr[4], const uint32_t key[2], uint32_t out[4]);

#ifdef __cplusplus
}
#endif
#endif
