/*
 * csrc/drt_context.cuh -- private to the library: the context behind drt_cuda_context*, the error helpers and the launchers the
 * C-ABI translation units (drt_capi.cu, drt_exchange.cu) share.
 */
#pragma once
#include <cuda_runtime.h>
#include <stdarg.h>
#include <stdint.h>
#include <stdio.h>
#include "drt_cuda.h"
#include "drt_device.cuh"

cudaError_t drt_launch_render(const RenderLaunch &L, bool f64_geometry, int mode, int nslots, int grid, int warps, size_t smem, cudaStream_t stream);
size_t      drt_render_smem_bytes(const RenderLaunch &L, bool f64_geometry, int warps, int nslots);
void        drt_launch_film_to_rgb(const void *tables, const float *plane, const float *filter, int normalise_by_max, uint32_t npix,
                                   float *rgb, uint32_t *bgra, int grid, cudaStream_t stream);
void        drt_launch_film_merge(FilmPtrs dst, FilmPtrs src, uint32_t n, size_t npix, int grid, cudaStream_t stream);
void        drt_launch_fma_peak(int packed, float *out, int iters, int grid, cudaStream_t stream);
void        drt_launch_film_gather_merge(const void *tables, int count, const FilmPtrs *films, FilmPtrs dst, uint32_t pixel_begin, uint32_t pixel_end, uint32_t src_base, uint32_t dst_base,
                                         uint32_t *bgra_sum, uint32_t *bgra_mean, uint32_t *bgra_var, int grid, cudaStream_t stream);
/* drt_denoise.cu: the guide planes (Y, v, usable as 1 / 0, npix each) of a film, then the filter of drt_cuda_film_denoise from them */
void        drt_launch_denoise_guide(const float *yw, const float *mean, const float *m2, const float *filter, uint32_t npix, int n, float *guide,
                                     int grid, cudaStream_t stream);
cudaError_t drt_launch_denoise_filter(const float *mean, const float *guide, uint32_t width, uint32_t height, int n, int search_radius,
                                      int patch_radius, float strength, float *out, cudaStream_t stream);
size_t      drt_denoise_smem_bytes(int n, int search_radius, int patch_radius);
size_t      drt_rgb_tables_bytes(void);
size_t      drt_rgb_tables_yw_offset(void);   /* byte offset of the luminance weights cmf_y * ref_white (adaptive sampling) */
void        drt_fill_rgb_tables(void *dst_host, const drt_tables *t);

int drt_fail(int code, const char *fmt, ...);   /* records the message drt_cuda_last_error() returns (thread-local), returns code */
#define fail drt_fail

#define CU(call) do { cudaError_t e_ = (call); if(e_ != cudaSuccess) return fail(DRT_CUDA_E_CUDA, "%s: %s", #call, cudaGetErrorString(e_)); } while(0)

#define DRT_RING 64

struct drt_cuda_context
{
    int    device = 0;
    int    num_sms = 0;
    size_t smem_optin = 0;
    bool   have_scene = false;
    bool   f64_geometry = false;
    int    n = 0, nslots = 0, nlights = 0, eval_words = 1;
    bool   hit_bound = false;      /* hit_u/v: film-plane bound (in pixel units of the uploaded camera) of everything a camera ray can hit */
    double hit_u0 = 0, hit_u1 = 0, hit_v0 = 0, hit_v1 = 0;
    int    scene_mode = 0;        /* the render kernel the uploaded scene gets (scene_kernel_mode in drt_capi.cu) */
    void  *d_geom32 = nullptr, *d_geom64 = nullptr;
    SpdIndex *d_index = nullptr;
    float *d_pool = nullptr;
    uint32_t pool_words = 0;
    size_t pool_capacity = 0;
    void  *d_rgb_tables = nullptr;
    /* Work counters and the task counter are PER CALL, taken round-robin from two small rings, so that renders of one context that
     * are in flight on different streams (a user stream, render_host's band streams, the legacy stream of sample_paths) never
     * share a counter: stats_ring[i] belongs to the i-th most recent render call (the bands of one render_host call share one),
     * counter_ring[i] to one kernel launch.  A slot is reused after DRT_RING calls; get_stats reads the latest call's block.
     * (The library's growing buffers d_film / d_dump / d_slice are reallocated with cudaFree, which waits for the device.) */
    DeviceStats *d_stats_ring = nullptr;
    unsigned int *d_counter_ring = nullptr;
    uint64_t stats_calls = 0, counter_launches = 0;
    DeviceStats *d_stats = nullptr;       /* the current call's block inside d_stats_ring */
    /* library-owned film + dump buffers for the host-buffer entry points */
    float *d_film = nullptr; size_t film_bytes = 0;
    float *d_dump = nullptr; size_t dump_bytes = 0;
    float *d_deep = nullptr; size_t deep_bytes = 0;     /* overflow rows of deep renders (RenderLaunch::deep) */
    float *d_slice = nullptr; size_t slice_bytes = 0;   /* merged planes of this rank's slice before they are copied to the root */
    float *d_denoise = nullptr; size_t denoise_bytes = 0;   /* the denoise guide planes (drt_denoise.cu) */
    /* recorded after each denoise filter; the next denoise call's stream waits on it before its guide overwrites d_denoise, so calls
     * on different streams take the guide planes one after the other */
    cudaEvent_t denoise_done = nullptr;
    uint64_t launches = 0;
    size_t upload_bytes = 0;
    uint64_t last_launches = 0;
    /* render_host pipelines the frame in row bands: render on one stream, read finished bands back on the other */
    cudaStream_t band_render = nullptr, band_copy = nullptr;
    cudaEvent_t  band_done[16] = {};
    /* multi-GPU exchange (drt_exchange.cu): count of flag waits that gave up (device word), the in-process state of render_host_multi */
    unsigned int *d_wait_timeouts = nullptr;
    struct drt_multi_state *multi = nullptr;
};


void drt_exchange_release(drt_cuda_context *ctx);   /* frees what drt_exchange.cu hung on the context */
int drt_ensure_buffer(float **buf, size_t *have, size_t need);
/* The library's layout of a device film of npix pixels and n wavelengths at base: the sum, mean, m2 and filter planes one after the other. */
static inline drt_film film_planes(float *base, size_t npix, int n)
{
    const size_t plane = npix * (size_t)n;
    return drt_film{ base, base + 3 * plane, base + plane, base + 2 * plane };
}
/* film_planes in one of the context's growing buffers (buf, have: d_film, film_bytes or d_slice, slice_bytes), grown first if need be */
int drt_library_film(const drt_cuda_context *ctx, float **buf, size_t *have, size_t npix, drt_film *out);

static inline bool film_complete(const drt_film *f) { return f && f->sum && f->filter && f->mean && f->m2; }
static inline FilmPtrs film_ptrs(const drt_film &f) { return FilmPtrs{ f.sum, f.filter, f.mean, f.m2 }; }
