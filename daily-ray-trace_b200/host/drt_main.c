/*
 * host/drt_main.c -- thin Linux main replacing win32_main.c:123-156 and the platform layer (win32_platform.c).
 *
 * Same contract as the reference executable: run it in a directory that holds config.cfg, scenes/, spectra/ and
 * output/; it reads config.cfg, renders input_scene, writes the three .spd films and converts each to a .bmp
 * (win32_main.c:129-152).  The render itself goes through the C ABI of include/drt_cuda.h; the timed region is the
 * reference's render_timer scope (sampling + film accumulation, daily_ray_trace.c:709-752; file I/O excluded).
 *
 *   drt_raytrace [config.cfg] [--device N] [--gpus G] [--seed S] [--strict] [--f64-geometry] [--cpu-images] [--adaptive REL [--min-spp M]] [--denoise]
 * --gpus G renders on devices N .. N+G-1: the samples of every pixel are split over them (drt_cuda_render_host_multi_images).
 * The three .bmp images come from the devices with the film (converted from the merged film there, fused into the multi-GPU merge
 * kernel); --cpu-images converts them the reference's way instead: by reading the .spd files back (spd_file_to_rgb_f64_pixels,
 * daily_ray_trace.c:1-28, in f64 -- bytes may differ by 1 from the device's f32 conversion).
 * --adaptive REL samples adaptively (drt_cuda_render_host_adaptive): a pixel stops once the error bound of its luminance is at most REL
 * times the luminance and it has at least M samples (--min-spp, default 64, at most num_pixel_samples); num_pixel_samples is the cap.
 * One device only, and the .bmp images are converted from the .spd files as with --cpu-images.
 * --denoise also filters the film with non-local means at the default parameters (drt_cuda_film_denoise_host on the first device) and
 * writes denoised.spd (the format of average.spd) and denoised.bmp next to average.spd; the other files are those of a run without it.
 */
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <time.h>
#include "drt_host.h"
#include "drt_cuda.h"

static double now_ms(void)
{
    struct timespec ts;
    clock_gettime(CLOCK_MONOTONIC, &ts);
    return (double)ts.tv_sec * 1e3 + (double)ts.tv_nsec * 1e-6;
}

static int die_host(const char *what) { fprintf(stderr, "ERROR: %s: %s\n", what, drt_host_last_error()); return 1; }
static int die_cuda(const char *what) { fprintf(stderr, "ERROR: %s: %s\n", what, drt_cuda_last_error()); return 1; }

static int spd_to_bmp(const char *spd, const char *bmp, const drt_tables *t)
{
    uint32_t w = 0, h = 0;
    double *rgb = NULL;
    if(drt_spd_to_rgb(spd, t, &w, &h, &rgb) != DRT_OK) return -1;
    int rc = drt_write_bmp_rgb(bmp, w, h, rgb);
    free(rgb);
    return rc;
}

int main(int argc, char **argv)
{
    const char *config_path = "config.cfg";
    int device = 0, gpus = 1, flags = DRT_PARSE_LEGACY_COMPAT, precision = DRT_GEOMETRY_F32, cpu_images = 0, adaptive = 0, denoise = 0;
    unsigned long long seed = 0;
    drt_adaptive ad = { 0.f, 64u };
    for(int i = 1; i < argc; i += 1)
    {
        if(strcmp(argv[i], "--device") == 0 && i + 1 < argc) device = atoi(argv[++i]);
        else if(strcmp(argv[i], "--gpus") == 0 && i + 1 < argc) gpus = atoi(argv[++i]);
        else if(strcmp(argv[i], "--seed") == 0 && i + 1 < argc) seed = strtoull(argv[++i], NULL, 0);
        else if(strcmp(argv[i], "--strict") == 0) flags = DRT_PARSE_STRICT;
        else if(strcmp(argv[i], "--f64-geometry") == 0) precision = DRT_GEOMETRY_F64;
        else if(strcmp(argv[i], "--cpu-images") == 0) cpu_images = 1;
        else if(strcmp(argv[i], "--denoise") == 0) denoise = 1;
        else if(strcmp(argv[i], "--adaptive") == 0 && i + 1 < argc) { adaptive = 1; ad.rel_error = strtof(argv[++i], NULL); }
        else if(strcmp(argv[i], "--min-spp") == 0 && i + 1 < argc) ad.min_samples = (uint32_t)strtoul(argv[++i], NULL, 0);
        else config_path = argv[i];
    }
    if(adaptive && gpus != 1)
    {
        /* with the samples of a pixel split over devices no device sees the merged film the stopping rule needs */
        fprintf(stderr, "ERROR: --adaptive renders on one GPU: it cannot be combined with --gpus %d\n", gpus);
        return 1;
    }
    if(adaptive) cpu_images = 1;

    drt_config cfg;
    if(drt_parse_config_file(config_path, &cfg) != DRT_OK) return die_host("config");
    printf("CONFIG ARGS:\n");
    printf("Num pixel samples:   %u\nOutput width:        %u\nOutput height:       %u\n", cfg.num_pixel_samples, cfg.output_width, cfg.output_height);
    printf("Min wavelength:      %f\nMax wavelength:      %f\nWavelength interval: %f\n", cfg.min_wl, cfg.max_wl, cfg.wl_interval);
    printf("Input scene path:    %s\nOutput spd path:     %s\nAverage spd path:    %s\nVariance spd path:   %s\n", cfg.input_scene, cfg.output_spd, cfg.average_spd, cfg.variance_spd);
    printf("Output bmp path:     %s\nAverage bmp path:    %s\nVariance bmp path:   %s\n\n", cfg.output_bmp, cfg.average_bmp, cfg.variance_bmp);

    static drt_tables tables;
    static drt_scene scene;
    static drt_camera camera;
    if(drt_load_tables(&cfg, ".", &tables) != DRT_OK) return die_host("spectral tables");
    if(drt_load_scene_file(".", cfg.input_scene, &tables, flags, cfg.output_width, cfg.output_height, &scene, &camera) != DRT_OK) return die_host("scene");

    if(gpus < 1 || gpus > 16) { fprintf(stderr, "ERROR: --gpus %d (1..16)\n", gpus); return 1; }
    drt_cuda_context *ctxs[16] = { NULL };
    for(int g = 0; g < gpus; g += 1)
    {
        if(drt_cuda_create(device + g, &ctxs[g]) != DRT_CUDA_OK) return die_cuda("cuda");
        if(drt_cuda_upload_scene(ctxs[g], &scene, &camera, &tables) != DRT_CUDA_OK) return die_cuda("upload");
        drt_cuda_set_geometry_precision(ctxs[g], precision);
    }

    /* host film and images in page-locked memory (read-backs run as DMA, all devices at once); pageable memory if that is refused */
    size_t npix = (size_t)cfg.output_width * cfg.output_height, n = (size_t)scene.num_wavelengths;
    drt_film film;
    uint32_t *images[3] = { NULL, NULL, NULL };
    void *blocks[7] = { NULL };
    const size_t sizes[7] = { npix * n * 4, npix * n * 4, npix * n * 4, npix * 4, npix * 4, npix * 4, npix * 4 };
    int pinned = 1;
    for(int i = 0; i < 7 && pinned; i += 1) if(drt_cuda_host_alloc(sizes[i] ? sizes[i] : 4, &blocks[i]) != DRT_CUDA_OK) pinned = 0;
    if(!pinned)
        for(int i = 0; i < 7; i += 1) { if(blocks[i]) drt_cuda_host_free(blocks[i]); blocks[i] = malloc(sizes[i] ? sizes[i] : 4); }
    for(int i = 0; i < 7; i += 1) if(!blocks[i]) { fprintf(stderr, "ERROR: out of host memory\n"); return 1; }
    film.sum = (float *)blocks[0]; film.mean = (float *)blocks[1]; film.m2 = (float *)blocks[2]; film.filter = (float *)blocks[3];
    for(int i = 0; i < 3; i += 1) images[i] = (uint32_t *)blocks[4 + i];

    drt_render_params prm;
    memset(&prm, 0, sizeof(prm));
    prm.width = cfg.output_width; prm.height = cfg.output_height;
    prm.sample_begin = 0; prm.sample_end = cfg.num_pixel_samples;
    prm.max_depth = cfg.max_cast_depth; prm.pixel_scheme = cfg.pixel_scheme; prm.seed = seed;

    if(adaptive && ad.min_samples > cfg.num_pixel_samples) ad.min_samples = cfg.num_pixel_samples;

    printf("Starting render...\n");
    double t0 = now_ms();
    int rrc = adaptive   ? drt_cuda_render_host_adaptive(ctxs[0], &prm, &ad, &film)
            : cpu_images ? drt_cuda_render_host_multi(ctxs, gpus, &prm, &film)
                         : drt_cuda_render_host_multi_images(ctxs, gpus, &prm, &film, images[0], images[1], images[2]);
    if(rrc != DRT_CUDA_OK) return die_cuda("render");
    double ms = now_ms() - t0;
    drt_cuda_stats st;
    memset(&st, 0, sizeof(st));
    for(int g = 0; g < gpus; g += 1)
    {
        drt_cuda_stats one;
        if(drt_cuda_get_stats(ctxs[g], &one) != DRT_CUDA_OK) return die_cuda("stats");
        st.paths += one.paths; st.closest_rays += one.closest_rays; st.shadow_rays += one.shadow_rays;
    }
    printf("Avg sample time: %fms\n", ms / (double)cfg.num_pixel_samples);
    printf("Total render time: %fms\n", ms);
    printf("Camera paths: %llu (%.3f Mpaths/s), rays: %llu (%.3f Mrays/s)\n", (unsigned long long)st.paths, (double)st.paths / ms * 1e-3,
           (unsigned long long)(st.closest_rays + st.shadow_rays), (double)(st.closest_rays + st.shadow_rays) / ms * 1e-3);
    if(adaptive)
        printf("Adaptive sampling: rel_error %g, min %u, cap %u samples per pixel; mean %.2f samples per pixel\n", (double)ad.rel_error,
               ad.min_samples, cfg.num_pixel_samples, npix ? (double)st.paths / (double)npix : 0.0);
    printf("Render complete.\n");

    if(drt_write_spd_sum(cfg.output_spd, &tables, prm.width, prm.height, film.sum, film.filter) != DRT_OK) return die_host("output spd");
    if(drt_write_spd_plain(cfg.average_spd, &tables, prm.width, prm.height, film.mean, 0) != DRT_OK) return die_host("average spd");
    if(drt_write_spd_plain(cfg.variance_spd, &tables, prm.width, prm.height, film.m2, 1) != DRT_OK) return die_host("variance spd");
    printf("Converting...\n");
    if(cpu_images)
    {
        if(spd_to_bmp(cfg.output_spd, cfg.output_bmp, &tables) != 0) return die_host("output bmp");
        if(spd_to_bmp(cfg.average_spd, cfg.average_bmp, &tables) != 0) return die_host("average bmp");
        if(spd_to_bmp(cfg.variance_spd, cfg.variance_bmp, &tables) != 0) return die_host("variance bmp");
    }
    else
    {
        if(drt_write_bmp(cfg.output_bmp, prm.width, prm.height, images[0]) != DRT_OK) return die_host("output bmp");
        if(drt_write_bmp(cfg.average_bmp, prm.width, prm.height, images[1]) != DRT_OK) return die_host("average bmp");
        if(drt_write_bmp(cfg.variance_bmp, prm.width, prm.height, images[2]) != DRT_OK) return die_host("variance bmp");
    }
    printf("Converted.\n");

    if(denoise)
    {
        /* denoised.spd / .bmp in the directory of average_spd (a path of the config file: '\\' or '/' separated) */
        char spd[80], bmp[80];
        const char *slash = strrchr(cfg.average_spd, '\\'), *fwd = strrchr(cfg.average_spd, '/');
        if(fwd && (!slash || fwd > slash)) slash = fwd;
        const int dir = slash ? (int)(slash - cfg.average_spd) + 1 : 0;
        snprintf(spd, sizeof(spd), "%.*sdenoised.spd", dir, cfg.average_spd);
        snprintf(bmp, sizeof(bmp), "%.*sdenoised.bmp", dir, cfg.average_spd);
        const size_t bytes = npix * n * 4;
        float *out = (float *)malloc(bytes ? bytes : 4);
        if(!out) { fprintf(stderr, "ERROR: out of host memory\n"); return 1; }
        const drt_denoise opt = { 7u, 3u, 0.45f };
        t0 = now_ms();
        if(drt_cuda_film_denoise_host(ctxs[0], &film, prm.width, prm.height, &opt, out) != DRT_CUDA_OK) return die_cuda("denoise");
        printf("Denoise time: %fms (non-local means, search radius %u, patch radius %u, strength %g)\n", now_ms() - t0, opt.search_radius,
               opt.patch_radius, (double)opt.strength);
        if(drt_write_spd_plain(spd, &tables, prm.width, prm.height, out, 0) != DRT_OK) return die_host("denoised spd");
        if(spd_to_bmp(spd, bmp, &tables) != 0) return die_host("denoised bmp");
        free(out);
    }

    for(int i = 0; i < 7; i += 1) { if(pinned) drt_cuda_host_free(blocks[i]); else free(blocks[i]); }
    for(int g = 0; g < gpus; g += 1) drt_cuda_destroy(ctxs[g]);
    return 0;
}
