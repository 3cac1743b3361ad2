/*
 * include/drt_cuda.h -- the drop-in boundary: a plain C ABI over the sm_100a render path.
 *
 * The reference has no plugin or FFI layer; its seams are C functions inside one translation unit
 * (SURVEY.md 8b).  These entry points replace them one for one:
 *
 *   drt_cuda_render_*       <- render_image's sampling loop      src/daily_ray_trace.c:709-752
 *                              (sample_scene :571-618, cast_ray :432-479, film + Welford :720-743)
 *   drt_cuda_sample_paths   <- sample_scene per (x, y, sample)    src/daily_ray_trace.c:571 (the inner seam, :729)
 *   drt_cuda_film_to_rgb    <- spd_file_to_rgb_f64_pixels         src/daily_ray_trace.c:1-28
 *                              + spectrum_to_rgb_f64 src/spectrum.c:49-82 + rgb_f64_to_rgb_u8 src/win32_platform.c:136-147
 *   drt_cuda_film_merge     <- (new) combines films of disjoint sample ranges: multi-GPU sample sharding
 *   drt_cuda_upload_scene   <- load_scene's result (scene_data/camera_data, daily_ray_trace.h:146-170) + init_spd_tables
 *
 * Conventions: POD structs and raw pointers only (no C++/torch types); every call returns 0 or a negative
 * DRT_CUDA_E_* code and drt_cuda_last_error() describes the failure; a context is bound to one CUDA device and
 * may be driven by one host thread at a time.  There is no CPU fallback: without a CUDA device every call fails.
 *
 * Film layout (all planes f32, pixel-major, row-major from the film's bottom-left like the .spd files):
 *   sum[W*H*N]  sum of path contributions        filter[W*H]  sum of filter weights (= sample count, Q20)
 *   mean[W*H*N] Welford running mean             m2[W*H*N]    Welford sum of squared deviations (Q17)
 */
#ifndef DRT_CUDA_H
#define DRT_CUDA_H

#include <stddef.h>
#include <stdint.h>
#include "drt_scene.h"

#ifdef __cplusplus
extern "C" {
#endif

enum
{
    DRT_CUDA_OK = 0,
    DRT_CUDA_E_NO_DEVICE = -101,   /* no CUDA device / driver: the product path never falls back to the CPU */
    DRT_CUDA_E_CUDA = -102,        /* a CUDA runtime call failed (message holds cudaGetErrorString) */
    DRT_CUDA_E_ARG = -103,
    DRT_CUDA_E_UNSUPPORTED = -104, /* scene outside what the kernels handle (message says what) */
    DRT_CUDA_E_STATE = -105        /* call order: render before upload_scene, ... */
};

typedef struct drt_cuda_context drt_cuda_context;

/* arithmetic of the geometric part of a path (intersection, sampling, visibility) */
enum { DRT_GEOMETRY_F32 = 0, DRT_GEOMETRY_F64 = 1 };

typedef struct
{
    float *sum, *filter, *mean, *m2;   /* device pointers (render_device) or host pointers (render_host) */
} drt_film;

/* work counters of one render call: the R_c, R_s, B of the flops formula in SURVEY.md 8d */
typedef struct
{
    uint64_t paths, closest_rays, shadow_rays, shaded_bounces, rng_draws;
    uint64_t terminated_at_depth[8];
    uint64_t reached_depth_cap;
    uint64_t kernel_launches;          /* kernels of this library launched by the call */
} drt_cuda_stats;

const char *drt_cuda_last_error(void);
int  drt_cuda_device_count(void);

int  drt_cuda_create(int device, drt_cuda_context **out);
void drt_cuda_destroy(drt_cuda_context *ctx);

/* Copies scene, camera and tables to the device (f64 narrowed as the kernels need). */
int  drt_cuda_upload_scene(drt_cuda_context *ctx, const drt_scene *scene, const drt_camera *camera, const drt_tables *tables);

/* The checks upload_scene applies to a scene before anything reaches the device, as plain host arithmetic (no device needed):
 * counts, material indices of surfaces / base / escape, lobe counts and ids, sampler ids, surface types, 630 nm inside the
 * wavelength grid.  DRT_CUDA_E_ARG / DRT_CUDA_E_UNSUPPORTED with a message, or DRT_CUDA_OK. */
int  drt_cuda_validate_scene(const drt_scene *scene);

/* Bytes the last upload_scene copied host -> device. */
int  drt_cuda_scene_upload_bytes(const drt_cuda_context *ctx, size_t *bytes);

/* DRT_GEOMETRY_F32 (default) or DRT_GEOMETRY_F64; spectra and film are f32 in both. */
int  drt_cuda_set_geometry_precision(drt_cuda_context *ctx, int precision);

/* Bytes of one f32 film plane set for a W x H image with the uploaded scene's N wavelengths. */
int  drt_cuda_film_sizes(const drt_cuda_context *ctx, uint32_t width, uint32_t height, size_t *spectral_plane_bytes, size_t *filter_plane_bytes);

/* Renders samples [sample_begin, sample_end) of every pixel into caller-owned DEVICE planes on `stream`
 * (a cudaStream_t passed as void*, NULL = default stream).  accumulate=0 overwrites the planes; accumulate=1
 * continues films that already hold earlier samples of the same pixels.  Asynchronous w.r.t. the host. */
int  drt_cuda_render_device(drt_cuda_context *ctx, const drt_render_params *params, const drt_film *film_device,
                            int accumulate, void *stream);

/* Multi-GPU render fused with the scatter half of the film exchange.  The image's pixels are split into `count` slices of
 * `slice_pixels` (rank r owns pixels [r * slice_pixels, (r + 1) * slice_pixels)); staging_device[o] is the staging film in the
 * memory of rank o (local or a peer mapping from drt_cuda_film_ipc_open), sized for count * slice_pixels pixels.  This rank
 * (`rank`) renders its samples of EVERY pixel and writes each finished pixel straight into its owner's staging film at pixel
 * rank * slice_pixels + (p - owner * slice_pixels): peer stores over NVLink, issued as pixels finish, so the transfer hides
 * under the render.  Afterwards every owner holds all ranks' partial films of its slice locally (drt_cuda_film_merge_slices). */
int  drt_cuda_render_device_scatter(drt_cuda_context *ctx, const drt_render_params *params, const drt_film *staging_device, int count, int rank,
                                    uint64_t slice_pixels, void *stream);

/* The same through HOST buffers: renders into library-owned device planes, then copies the four planes to
 * `film_host` (pinned or pageable) and waits.  This is the end-to-end call the Linux main uses. */
int  drt_cuda_render_host(drt_cuda_context *ctx, const drt_render_params *params, const drt_film *film_host);

/* Adaptive sampling: every pixel takes samples from sample_begin on in batches of 32 and stops at the end of the first batch after which
 * its film (count n, including samples an accumulate=1 call loaded) satisfies
 *     n >= min_samples  and  err <= rel_error * Y,   Y = sum_l w_l mean_l,   err = sum_l w_l sqrt(M2_l / (n (n - 1)))
 * with w_l the luminance weights cmf_y * ref_white of the .bmp conversion (err bounds the standard error of Y from above: the sd of a
 * sum is at most the sum of the sds), or when the samples of [sample_begin, sample_end) run out.  Sample s of a pixel is the same path
 * as in a uniform render, so a pixel that stops after k samples holds the film of [sample_begin, sample_begin + k): k is a multiple of
 * 32, or the whole range.  The filter plane holds each pixel's count, so sum / filter stays the mean; M2 (and the variance image) is a
 * sum over a count that varies from pixel to pixel.  Pixels whose samples are all zero (also those the screen-space culling counts
 * instead of tracing) and pixels without variance stop at the first batch end at or past min_samples; pixels with Y = 0 but noise, and
 * pixels whose film holds a NaN, run to the end of the range.  drt_cuda_get_stats reports the paths actually taken.
 * rel_error: finite, > 0; min_samples: 32 ..  sample_end - sample_begin (so the range holds at least 32 samples); else DRT_CUDA_E_ARG.
 * f64 geometry (a diagnostic) has no adaptive kernel: DRT_CUDA_E_UNSUPPORTED.  The multi-GPU form shards by ROWS, not by samples (with
 * the samples of a pixel split over devices, no device would see the merged film the rule needs): a device renders every sample of the
 * pixels of its rows, so each pixel's rule sees its whole film, nothing is merged, and the shards together are the one-device film bit
 * for bit (a pixel's paths and their order within a batch do not depend on the device or warp that takes it). */
typedef struct
{
    float    rel_error;
    uint32_t min_samples;
} drt_adaptive;

int  drt_cuda_render_device_adaptive(drt_cuda_context *ctx, const drt_render_params *params, const drt_adaptive *adaptive,
                                     const drt_film *film_device, int accumulate, void *stream);
int  drt_cuda_render_host_adaptive(drt_cuda_context *ctx, const drt_render_params *params, const drt_adaptive *adaptive,
                                   const drt_film *film_host);

/* Adaptive sampling of the rows y = rank (mod count) of the frame into a full-frame device film (other rows untouched): pixels are
 * stored, and with accumulate = 1 loaded, at their global positions.  count: 1 .. 16, rank: 0 .. count - 1, else DRT_CUDA_E_ARG; the other
 * checks are those of drt_cuda_render_device_adaptive.  A rank without rows (rank >= height) launches nothing, and drt_cuda_get_stats
 * then reports zeros.  Multi-process callers: rank r of `count` calls this with (count, r), then drt_cuda_film_read_rows. */
int  drt_cuda_render_device_adaptive_rows(drt_cuda_context *ctx, const drt_render_params *params, const drt_adaptive *adaptive,
                                          const drt_film *film_device, int accumulate, int count, int rank, void *stream);
/* Stream-ordered copy of those rows of a full-frame device film into a WHOLE host film (pinned for the copy to run asynchronously): one
 * cudaMemcpy2DAsync per plane; the host film's other rows are untouched. */
int  drt_cuda_film_read_rows(drt_cuda_context *ctx, const drt_film *film_device, uint32_t width, uint32_t height,
                             int count, int rank, const drt_film *film_host, void *stream);
/* Adaptive sampling on several devices of ONE process: contexts[g] live on distinct devices and hold the same scene; device g renders
 * rows y = g (mod count) into its library-owned full-frame film and copies them to film_host over its own PCIe link, then the call
 * waits.  The devices render at once; the copies overlap each other and the slower renders when film_host is pinned
 * (drt_cuda_host_alloc), and run one after another when it is pageable.  No peer access, no exchange.  With count > height the surplus devices stay idle.  Each context's
 * drt_cuda_get_stats reports the paths its device took.  count = 1 gives the film of drt_cuda_render_host_adaptive. */
int  drt_cuda_render_host_multi_adaptive(drt_cuda_context **contexts, int count, const drt_render_params *params,
                                         const drt_adaptive *adaptive, const drt_film *film_host);

/* render_host on several devices of ONE process (what `drt_raytrace --gpus G` calls): contexts[g] live on distinct devices and hold
 * the same scene; the samples [sample_begin, sample_end) are split evenly over them.  With peer access every device renders its share
 * of every pixel with drt_cuda_render_device_scatter, announces it with device-side flags (drt_cuda_flags_signal / _wait, no host
 * synchronisation), merges its own pixel slice locally (drt_cuda_film_merge_slices_local) and copies that slice to `film_host` over its
 * own PCIe link, all devices at once; staging memory persists between calls on contexts[0].  Without peer access the partial films
 * are merged one after the other on contexts[0]'s device (slower, same result); with fewer samples than devices the surplus devices
 * stay idle.  count = 1 is render_host. */
int  drt_cuda_render_host_multi(drt_cuda_context **contexts, int count, const drt_render_params *params, const drt_film *film_host);

/* The same, plus the three 8-bit images of win32_main.c:150-152 (sum / filter, mean, M2 / per-pixel max; packed BGRA as drt_write_bmp
 * takes them) converted ON THE DEVICES from the merged film -- fused into the merge kernel when several devices take part -- and copied
 * to the three host buffers of width * height words: the Linux main writes the .bmp files from these instead of re-reading the .spd
 * files it just wrote (9.4 GB each at 4096 x 4096) and converting on the CPU.  f32 arithmetic: bytes may differ by 1 from the f64
 * conversion of drt_spd_to_rgb. */
int  drt_cuda_render_host_multi_images(drt_cuda_context **contexts, int count, const drt_render_params *params, const drt_film *film_host,
                                       uint32_t *bgra_sum_host, uint32_t *bgra_mean_host, uint32_t *bgra_var_host);

/* Which render kernel the uploaded scene and the geometry precision select, for logs and benchmark lines:
 * name = "drt::render_kernel<float,5,true,true>" style string (geometry type, wavelength slots per half-warp lane, all-plastic
 * specialisation, one-pixel-per-task shape), warps_per_cta and ctas_per_sm as launched for a film render with `params`. */
int  drt_cuda_render_kernel_info(drt_cuda_context *ctx, const drt_render_params *params, char *name, size_t name_len, int *warps_per_cta, int *ctas_per_sm);

/* The two exact cullings drt_cuda_upload_scene prepares, as plain host arithmetic (no device needed; used by the CPU-tier tests):
 * hit_rect = {x0, y0, x1, y1}: pixels outside [x0, x1) x [y0, y1) of a width x height image cannot see any surface (pinhole camera;
 * the whole image when no bound exists, e.g. a thin lens), so the kernel counts their camera paths instead of tracing them;
 * boundary[i] = 1 for a plane that has the whole scene in one closed half-space: shadow rays do not test it. */
int  drt_cuda_analyse_scene(const drt_scene *scene, const drt_camera *camera, uint32_t width, uint32_t height,
                            uint32_t hit_rect[4], int32_t *boundary /* [scene->num_surfaces] */);

/* What drt_cuda_upload_scene decides about a scene, as plain host arithmetic (no device needed; used by the CPU-tier tests):
 * *kernel_mode = 1 plastic-only, 2 classed, 0 general (csrc/drt_render.cuh; f64 geometry always runs the general kernel);
 * material_class[m] (may be NULL) = 0 plastic, 1 single-basis specular, 2 rough conductor, 3 general, for every material;
 * specular_constants[m][match][2] (may be NULL; match 0 none, 1 reflection, 2 refraction) = the constants (c0, c1) of the
 * bdsf() sum c0 + c1 X of a specular material, tabulated by walking its lobe list with the reference's stale-scratch rule (Q7). */
int  drt_cuda_plan_scene(const drt_scene *scene, const drt_camera *camera, int32_t *kernel_mode,
                         int32_t *material_class /* [scene->num_materials] */, float *specular_constants /* [scene->num_materials][3][2] */);

/* Counters of the most recent render_* / sample_paths call (waits for it to finish). */
int  drt_cuda_get_stats(drt_cuda_context *ctx, drt_cuda_stats *out);

/* Per-path spectral radiance, the sample_scene seam: for every pixel of the rectangle [x0,x1) x [y0,y1) and every
 * sample in [params->sample_begin, sample_end) writes N f32 values to host buffer out[((y-y0)*(x1-x0)+(x-x0))*spp + s][N]. */
int  drt_cuda_sample_paths(drt_cuda_context *ctx, const drt_render_params *params,
                           uint32_t x0, uint32_t y0, uint32_t x1, uint32_t y1, float *out_host);

/* Diagnostics: the raw path records (the scalar weights phase 1 hands to phase 2, layout in csrc/drt_device.cuh) of the
 * same rectangle/sample range.  With out_host == NULL only *words_per_path is returned. */
int  drt_cuda_debug_records(drt_cuda_context *ctx, const drt_render_params *params, uint32_t x0, uint32_t y0, uint32_t x1, uint32_t y1,
                            float *out_host, size_t out_capacity_words, uint32_t *words_per_path);

/* which = 0: sum/filter, 1: mean, 2: m2 divided by its per-pixel maximum (the three .bmp images of win32_main.c:150-152).
 * rgb_device: 3 f32 per pixel (linear RGB, may be NULL); bgra_device: packed u32 per pixel (may be NULL). */
int  drt_cuda_film_to_rgb(drt_cuda_context *ctx, const drt_film *film_device, uint32_t width, uint32_t height, int which,
                          float *rgb_device, uint32_t *bgra_device, void *stream);

/* dst <- dst (+) src for films over the same pixels and disjoint samples (Chan et al. merge of count/mean/M2,
 * plain addition of sum/filter).  All device pointers; src may live on a peer GPU that this device can address. */
int  drt_cuda_film_merge(drt_cuda_context *ctx, const drt_film *dst_device, const drt_film *src_device,
                         uint32_t width, uint32_t height, void *stream);

/* Non-local-means denoising of a finished film, guided by its own mean and M2 (Rousselle, Knaus and Zwicker, "Adaptive rendering with
 * non-local means filtering", SIGGRAPH Asia 2012).  Reads the mean, m2 and filter planes (sum is ignored and may be NULL) and writes the
 * filtered mean plane [W*H*N] to mean_out, which must not overlap the film's planes; the film is not written.
 *   usable pixel p:  count n_p = filter >= 2, every mean and m2 value finite, and |Y_p| and v_p at most FLT_MAX (finite as f32)
 *   guide:           Y_p = sum_l w_l mean_l(p),  v_p = (sum_l w_l sqrt(max(0, m2_l(p) / (n_p (n_p - 1)))))^2  (w_l = cmf_y * ref_white,
 *                    the adaptive rule's weights; a negative m2 counts as zero variance); Y_p = v_p = 0 for an unusable p (they only
 *                    enter the patches of other pixels)
 *   distance:        for q = p + d, d in [-r, r]^2, q inside the image and usable:
 *                    D(a, b) = ((Y_a - Y_b)^2 - (v_a + min(v_a, v_b))) / (1e-10 + k^2 (v_a + v_b))
 *                    d2(p, q) = mean over o in [-f, f]^2 of D(clamp(p + o), clamp(q + o))   (clamp replicates the border)
 *   output:          wt(p, q) = exp(-max(0, d2(p, q))), or 0 where d2(p, q) is NaN; wt(p, p) = 1;
 *                    out_l(p) = sum_q wt(p, q) mean_l(q) / sum_q wt(p, q) for a usable p; an unusable p is copied bit for bit.
 * r = search_radius 1..15 (default 7), f = patch_radius 0..4 (default 3), k = strength in [2^-63, 2^64) so that k^2 is a normal f32
 * (default 0.45), else DRT_CUDA_E_ARG;
 * also W, H > 0 and the planes present.  N and w come from the uploaded scene (DRT_CUDA_E_STATE without one).  f32 sums in a fixed order:
 * the result is deterministic. */
typedef struct
{
    uint32_t search_radius, patch_radius;
    float    strength;
} drt_denoise;

/* Stream-ordered: film_device and mean_out_device are device planes.  Calls on one context may run on different streams: each waits for
 * the previous call's filter before it overwrites the context's guide scratch. */
int  drt_cuda_film_denoise(drt_cuda_context *ctx, const drt_film *film_device, uint32_t width, uint32_t height, const drt_denoise *opt,
                           float *mean_out_device, void *stream);
/* The same on host planes: copies the film up into library-owned device planes, filters, copies the result down and waits. */
int  drt_cuda_film_denoise_host(drt_cuda_context *ctx, const drt_film *film_host, uint32_t width, uint32_t height, const drt_denoise *opt,
                                float *mean_out_host);

/* ---- multi-GPU: library-owned films that other processes / devices can map, and the fused merge epilogue ---- */

/* Allocates the four planes of a W x H film with cudaMalloc (zero-filled) so that they can be exported over CUDA IPC. */
int  drt_cuda_film_alloc(drt_cuda_context *ctx, uint32_t width, uint32_t height, drt_film *out_device);
int  drt_cuda_film_free(drt_cuda_context *ctx, drt_film *film_device);

/* CUDA IPC handles (64 bytes each, order sum, filter, mean, m2) of a film from drt_cuda_film_alloc, and the reverse:
 * mapping a peer process's film into this context's address space (NVLink peer access).  Single-process callers can
 * skip IPC and pass another device's pointers directly after cudaDeviceEnablePeerAccess. */
int  drt_cuda_film_ipc_export(drt_cuda_context *ctx, const drt_film *film_device, unsigned char handles[4][64]);
int  drt_cuda_film_ipc_open(drt_cuda_context *ctx, const unsigned char handles[4][64], drt_film *out_mapped);
int  drt_cuda_film_ipc_close(drt_cuda_context *ctx, drt_film *mapped);

/* Plain device buffers that can be shared the same way (e.g. the root's three BGRA images). */
int  drt_cuda_buffer_alloc(drt_cuda_context *ctx, size_t bytes, void **out_device);
int  drt_cuda_buffer_free(drt_cuda_context *ctx, void *device_ptr);
int  drt_cuda_buffer_ipc_export(drt_cuda_context *ctx, const void *device_ptr, unsigned char handle[64]);
int  drt_cuda_buffer_ipc_open(drt_cuda_context *ctx, const unsigned char handle[64], void **out_mapped);
int  drt_cuda_buffer_ipc_close(drt_cuda_context *ctx, void *mapped);

/* ONE kernel on this device: for pixels [pixel_begin, pixel_end) read the partial films of all `count` ranks (any mix
 * of local and peer pointers, disjoint sample sets), merge them exactly (Chan), write the merged planes to dst_device
 * (may be peer memory, e.g. the root's film) and, if bgra_* are non-NULL, the three 8-bit images
 * (sum/filter, mean, M2/max) for those pixels.  Callers make sure all ranks have finished rendering first. */
int  drt_cuda_film_merge_many(drt_cuda_context *ctx, const drt_film *dst_device, const drt_film *srcs_device, int count,
                              uint32_t width, uint32_t height, uint64_t pixel_begin, uint64_t pixel_end,
                              uint32_t *bgra_sum, uint32_t *bgra_mean, uint32_t *bgra_var, void *stream);

/* The merge half of the scattered exchange, ONE kernel per rank on LOCAL data: merges the `count` partial films of this rank's
 * slice [pixel_begin, pixel_end) held in staging_device (layout of drt_cuda_render_device_scatter) into a library-owned
 * local scratch film, writes the three images like drt_cuda_film_merge_many, then copies the merged planes to dst_device at
 * the global pixel positions (may be peer memory, e.g. the root's film) as four contiguous stream-ordered copies.
 * [pixel_begin, pixel_end) may be a part (a band) of the slice: staging stays indexed from the slice's first pixel.  A range that
 * crosses a slice boundary is DRT_CUDA_E_ARG. */
int  drt_cuda_film_merge_slices(drt_cuda_context *ctx, const drt_film *dst_device, const drt_film *staging_device, int count, uint64_t slice_pixels,
                                uint32_t width, uint32_t height, uint64_t pixel_begin, uint64_t pixel_end,
                                uint32_t *bgra_sum, uint32_t *bgra_mean, uint32_t *bgra_var, void *stream);

/* The merge half of the scattered exchange with a SHARDED result: like drt_cuda_film_merge_slices, but the merged planes of
 * [pixel_begin, pixel_end) stay on this device in the caller's slice film (indexed from pixel_begin; a drt_cuda_film_alloc of
 * ceil(slice_pixels / width) rows), and nothing but the three images (if given; usually the root's memory) leaves the device.
 * [pixel_begin, pixel_end) may also be a part (a band) of the slice: staging and slice film stay indexed from the slice's first pixel. */
int  drt_cuda_film_merge_slices_local(drt_cuda_context *ctx, const drt_film *slice_device, const drt_film *staging_device, int count, uint64_t slice_pixels,
                                      uint32_t width, uint32_t height, uint64_t pixel_begin, uint64_t pixel_end,
                                      uint32_t *bgra_sum, uint32_t *bgra_mean, uint32_t *bgra_var, void *stream);

/* Four stream-ordered device -> host copies of (a part of) a merged slice into a WHOLE host film (pinned for the copies to overlap) at
 * the pixels' global positions: every rank reads its own slice back over its own PCIe link.  slice_device is indexed from pixel
 * slice_begin (the first pixel of the owner's slice); [pixel_begin, pixel_end) is the part to copy. */
int  drt_cuda_film_read_slice(drt_cuda_context *ctx, const drt_film *slice_device, uint64_t slice_begin, uint64_t pixel_begin, uint64_t pixel_end,
                              const drt_film *film_host, void *stream);

/* A BAND of drt_cuda_render_device_scatter: the same part [band_begin, band_end) (pixel offsets inside a slice) of EVERY owner's slice,
 * i.e. pixels o * slice_pixels + band_begin ... for o = 0 .. count - 1.  Rendering a frame band by band lets every owner merge
 * (drt_cuda_film_merge_slices_local on the band's part of its slice) and read back band b on a second stream while band b + 1
 * renders: the PCIe read-back hides under the render.  Needs >= 32 samples per pixel.  keep_stats != 0 adds this launch's work
 * counters to the previous launch's (one drt_cuda_get_stats for all bands of a frame). */
int  drt_cuda_render_device_scatter_band(drt_cuda_context *ctx, const drt_render_params *params, const drt_film *staging_device, int count, int rank,
                                         uint64_t slice_pixels, uint64_t band_begin, uint64_t band_end, int keep_stats, void *stream);

/* Device-side arrival flags, the exchange's only synchronisation (no host barrier between the render and the merge):
 * _signal: one tiny kernel on `stream` that, after everything enqueued before it on the stream has completed, fences system-wide and
 *          stores `value` to each of the `count` flag words targets[i] (device pointers, local or peer memory);
 * _wait:   one tiny kernel on `stream` that returns when each of the `count` consecutive LOCAL words at flags_device holds a value
 *          >= `value` (epochs compared modulo 2^32), so work enqueued after it sees the data the signals announced.  A wait gives up
 *          after 20 s; _timeouts returns how many did since the context was created (non-zero = a peer never arrived). */
int  drt_cuda_flags_signal(drt_cuda_context *ctx, uint32_t *const *targets, int count, uint32_t value, void *stream);
int  drt_cuda_flags_wait(drt_cuda_context *ctx, const uint32_t *flags_device, int count, uint32_t value, void *stream);
int  drt_cuda_flags_timeouts(drt_cuda_context *ctx, uint32_t *timeouts);

/* Page-locked host memory (portable across devices) for film planes: read-backs into it run as DMA and overlap with rendering. */
int  drt_cuda_host_alloc(size_t bytes, void **out_host);
int  drt_cuda_host_free(void *host_ptr);

/* Measured FP32 FMA throughput of this device (TFLOP/s, FFMA counted as 2 flops): the roofline denominator
 * MEASURED_PEAKS.json does not carry.  packed=1 uses fma.rn.f32x2. */
int  drt_cuda_measure_fp32_peak(drt_cuda_context *ctx, int packed, double *tflops);

#ifdef __cplusplus
}
#endif
#endif
