/*
 * csrc/drt_exchange.cu -- the multi-GPU film exchange without host synchronisation (SURVEY.md 8e).
 *
 * The path shards by SAMPLE INDEX: every GPU renders its share of the samples of every pixel, and the partial films are combined
 * once per render.  The exchange is three stream-ordered steps per rank, none of which involves the host:
 *
 *   render + scatter   drt_cuda_render_device_scatter (drt_capi.cu): the render kernel stores each finished pixel straight into
 *                      the staging film of the rank that OWNS the pixel's slice (peer stores over NVLink under the render)
 *   signal / wait      flag_signal_kernel: after its render a rank publishes an epoch number into one word of every owner's flag
 *                      block (system-scope fence, then release stores over NVLink); flag_wait_kernel: an owner polls its LOCAL
 *                      flag words until every rank's epoch has arrived (acquire loads).  These replace the two host barriers
 *                      of round 1 (0.2 + 0.3 ms of the 1.6 ms fixed exchange cost at 8 GPUs).
 *   merge (sharded)    drt_cuda_film_merge_slices_local: every owner merges the N partial films of its slice from local memory
 *                      (Chan's count / mean / M2 update) into ITS OWN merged slice and writes only the three 8-bit images to the
 *                      root.  The merged spectral film stays sharded over the owners: each owner reads its slice back to the
 *                      host over its own PCIe link (drt_cuda_film_read_slice) -- nothing funnels through one GPU.
 *
 * A wait gives up after DRT_FLAG_TIMEOUT_NS (a peer that died must not hang the device); the give-ups are counted in a device
 * word that drt_cuda_flags_timeouts reads, and callers treat a non-zero count as a failed exchange.
 *
 * drt_cuda_render_host_multi is the same exchange inside ONE process (what `drt_raytrace --gpus G` calls).
 */
#include <stdlib.h>
#include <string.h>
#include "drt_context.cuh"

#define DRT_FLAG_TIMEOUT_NS 20000000000ull   /* 20 s: far beyond any render share, short of the driver's patience */

namespace drt {

struct FlagTargets { uint32_t *p[DRT_MAX_PEERS]; };

/* One thread per target.  The kernel boundary orders this kernel after every store of the kernels before it on the stream (the
 * scattered film pixels); the fence makes them visible system-wide before the flag that announces them. */
__global__ void flag_signal_kernel(FlagTargets t, int count, uint32_t value)
{
    if((int)threadIdx.x < count)
    {
        __threadfence_system();
        asm volatile("st.release.sys.global.u32 [%0], %1;" :: "l"(t.p[threadIdx.x]), "r"(value) : "memory");
    }
}

/* One thread per flag word; epochs only grow, compared modulo 2^32. */
__global__ void flag_wait_kernel(const uint32_t *flags, int count, uint32_t value, unsigned int *timeouts)
{
    if((int)threadIdx.x < count)
    {
        unsigned long long t0;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t0));
        for(;;)
        {
            uint32_t v;
            asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(flags + threadIdx.x) : "memory");
            if((int32_t)(v - value) >= 0) break;
            unsigned long long t1;
            asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t1));
            if(t1 - t0 > DRT_FLAG_TIMEOUT_NS) { atomicAdd(timeouts, 1u); break; }
            __nanosleep(200);
        }
    }
    __threadfence_system();
}

} // namespace drt

static int wait_word(drt_cuda_context *ctx)
{
    if(ctx->d_wait_timeouts) return DRT_CUDA_OK;
    CU(cudaMalloc(&ctx->d_wait_timeouts, sizeof(unsigned int)));
    CU(cudaMemset(ctx->d_wait_timeouts, 0, sizeof(unsigned int)));
    return DRT_CUDA_OK;
}

extern "C" int drt_cuda_flags_signal(drt_cuda_context *ctx, uint32_t *const *targets, int count, uint32_t value, void *stream)
{
    if(!ctx || !targets || count < 1 || count > DRT_MAX_PEERS) return fail(DRT_CUDA_E_ARG, "bad argument (1..%d flag words)", DRT_MAX_PEERS);
    CU(cudaSetDevice(ctx->device));
    drt::FlagTargets t;
    memset(&t, 0, sizeof(t));
    for(int i = 0; i < count; i += 1)
    {
        if(!targets[i]) return fail(DRT_CUDA_E_ARG, "flag target %d is NULL", i);
        t.p[i] = targets[i];
    }
    drt::flag_signal_kernel<<<1, 32, 0, (cudaStream_t)stream>>>(t, count, value);
    CU(cudaGetLastError());
    ctx->launches += 1;
    return DRT_CUDA_OK;
}

extern "C" int drt_cuda_flags_wait(drt_cuda_context *ctx, const uint32_t *flags_device, int count, uint32_t value, void *stream)
{
    if(!ctx || !flags_device || count < 1 || count > DRT_MAX_PEERS) return fail(DRT_CUDA_E_ARG, "bad argument (1..%d flag words)", DRT_MAX_PEERS);
    CU(cudaSetDevice(ctx->device));
    int rc = wait_word(ctx);
    if(rc != DRT_CUDA_OK) return rc;
    drt::flag_wait_kernel<<<1, 32, 0, (cudaStream_t)stream>>>(flags_device, count, value, ctx->d_wait_timeouts);
    CU(cudaGetLastError());
    ctx->launches += 1;
    return DRT_CUDA_OK;
}

extern "C" int drt_cuda_flags_timeouts(drt_cuda_context *ctx, uint32_t *timeouts)
{
    if(!ctx || !timeouts) return fail(DRT_CUDA_E_ARG, "NULL argument");
    *timeouts = 0;
    if(!ctx->d_wait_timeouts) return DRT_CUDA_OK;
    CU(cudaSetDevice(ctx->device));
    CU(cudaMemcpy(timeouts, ctx->d_wait_timeouts, sizeof(uint32_t), cudaMemcpyDeviceToHost));
    return DRT_CUDA_OK;
}

extern "C" int drt_cuda_film_merge_slices_local(drt_cuda_context *ctx, const drt_film *slice_device, const drt_film *staging, int count, uint64_t slice_pixels,
                                                uint32_t width, uint32_t height, uint64_t pixel_begin, uint64_t pixel_end,
                                                uint32_t *bgra_sum, uint32_t *bgra_mean, uint32_t *bgra_var, void *stream)
{
    if(!ctx || !slice_device || !staging || count < 1 || count > DRT_MAX_PEERS) return fail(DRT_CUDA_E_ARG, "bad argument (1..%d ranks)", DRT_MAX_PEERS);
    if(!film_complete(slice_device)) return fail(DRT_CUDA_E_ARG, "NULL slice film");
    if(!film_complete(staging)) return fail(DRT_CUDA_E_ARG, "NULL staging film");
    if(!ctx->have_scene) return fail(DRT_CUDA_E_STATE, "upload a scene first");
    const uint64_t npix = (uint64_t)width * height;
    if(pixel_begin > pixel_end || pixel_end > npix || pixel_end - pixel_begin > slice_pixels || npix > 0xffffffffull) return fail(DRT_CUDA_E_ARG, "bad pixel range");
    if((bgra_sum || bgra_mean || bgra_var) && !(bgra_sum && bgra_mean && bgra_var)) return fail(DRT_CUDA_E_ARG, "give all three image buffers or none");
    CU(cudaSetDevice(ctx->device));
    if(pixel_end == pixel_begin) return DRT_CUDA_OK;
    const size_t n = (size_t)ctx->n;
    FilmPtrs films[DRT_MAX_PEERS];
    for(int g = 0; g < count; g += 1)   /* rank g's partial film of this slice: staging pixels [g * slice, (g + 1) * slice) */
        films[g] = FilmPtrs{ staging->sum + (size_t)g * slice_pixels * n, staging->filter + (size_t)g * slice_pixels,
                             staging->mean + (size_t)g * slice_pixels * n, staging->m2 + (size_t)g * slice_pixels * n };
    /* staging and slice film are indexed from the first pixel of the owner's slice; [pixel_begin, pixel_end) may be a part (a band) of it */
    const uint64_t slice_begin = (pixel_begin / slice_pixels) * slice_pixels;
    if(pixel_end - slice_begin > slice_pixels) return fail(DRT_CUDA_E_ARG, "pixel range crosses a slice boundary");
    drt_launch_film_gather_merge(ctx->d_rgb_tables, count, films, film_ptrs(*slice_device), (uint32_t)pixel_begin, (uint32_t)pixel_end, (uint32_t)slice_begin,
                                 (uint32_t)slice_begin, bgra_sum, bgra_mean, bgra_var, ctx->num_sms * 8, (cudaStream_t)stream);
    CU(cudaGetLastError());
    ctx->launches += 1;
    return DRT_CUDA_OK;
}

extern "C" int drt_cuda_film_read_slice(drt_cuda_context *ctx, const drt_film *slice_device, uint64_t slice_begin, uint64_t pixel_begin, uint64_t pixel_end,
                                        const drt_film *film_host, void *stream)
{
    if(!ctx || !slice_device || !film_complete(film_host)) return fail(DRT_CUDA_E_ARG, "NULL argument");
    if(!ctx->have_scene) return fail(DRT_CUDA_E_STATE, "upload a scene first");
    if(pixel_begin > pixel_end || slice_begin > pixel_begin) return fail(DRT_CUDA_E_ARG, "bad pixel range");
    CU(cudaSetDevice(ctx->device));
    const size_t n = (size_t)ctx->n, spx = (size_t)(pixel_end - pixel_begin), at = (size_t)pixel_begin * n, from = (size_t)(pixel_begin - slice_begin);
    if(spx == 0) return DRT_CUDA_OK;
    cudaStream_t s = (cudaStream_t)stream;
    CU(cudaMemcpyAsync(film_host->sum + at, slice_device->sum + from * n, spx * n * 4, cudaMemcpyDeviceToHost, s));
    CU(cudaMemcpyAsync(film_host->mean + at, slice_device->mean + from * n, spx * n * 4, cudaMemcpyDeviceToHost, s));
    CU(cudaMemcpyAsync(film_host->m2 + at, slice_device->m2 + from * n, spx * n * 4, cudaMemcpyDeviceToHost, s));
    CU(cudaMemcpyAsync(film_host->filter + pixel_begin, slice_device->filter + from, spx * 4, cudaMemcpyDeviceToHost, s));
    return DRT_CUDA_OK;
}

extern "C" int drt_cuda_film_read_rows(drt_cuda_context *ctx, const drt_film *film_device, uint32_t width, uint32_t height, int count, int rank,
                                       const drt_film *film_host, void *stream)
{
    if(!ctx || !film_complete(film_device) || !film_complete(film_host)) return fail(DRT_CUDA_E_ARG, "NULL argument");
    if(count < 1 || count > DRT_MAX_PEERS || rank < 0 || rank >= count) return fail(DRT_CUDA_E_ARG, "bad row shard: rank %d of %d (1..%d ranks)", rank, count, DRT_MAX_PEERS);
    if(!ctx->have_scene) return fail(DRT_CUDA_E_STATE, "upload a scene first");
    CU(cudaSetDevice(ctx->device));
    if(width == 0 || (uint32_t)rank >= height) return DRT_CUDA_OK;
    /* rows rank, rank + count, ...: one strided copy per plane, row pitch count rows in both films */
    const size_t rows = (height - (uint32_t)rank + (uint32_t)count - 1) / (uint32_t)count, n = (size_t)ctx->n;
    const size_t row = (size_t)width * n * 4, at = (size_t)rank * width * n, frow = (size_t)width * 4, fat = (size_t)rank * width;
    cudaStream_t s = (cudaStream_t)stream;
    CU(cudaMemcpy2DAsync(film_host->sum + at, row * count, film_device->sum + at, row * count, row, rows, cudaMemcpyDeviceToHost, s));
    CU(cudaMemcpy2DAsync(film_host->mean + at, row * count, film_device->mean + at, row * count, row, rows, cudaMemcpyDeviceToHost, s));
    CU(cudaMemcpy2DAsync(film_host->m2 + at, row * count, film_device->m2 + at, row * count, row, rows, cudaMemcpyDeviceToHost, s));
    CU(cudaMemcpy2DAsync(film_host->filter + fat, frow * count, film_device->filter + fat, frow * count, frow, rows, cudaMemcpyDeviceToHost, s));
    return DRT_CUDA_OK;
}

extern "C" int drt_cuda_host_alloc(size_t bytes, void **out)
{
    if(!out || bytes == 0) return fail(DRT_CUDA_E_ARG, "bad argument");
    cudaError_t e = cudaHostAlloc(out, bytes, cudaHostAllocPortable);
    if(e != cudaSuccess) { *out = nullptr; return fail(e == cudaErrorNoDevice || e == cudaErrorInsufficientDriver ? DRT_CUDA_E_NO_DEVICE : DRT_CUDA_E_CUDA, "cudaHostAlloc(%zu): %s", bytes, cudaGetErrorString(e)); }
    return DRT_CUDA_OK;
}

extern "C" int drt_cuda_host_free(void *ptr)
{
    if(!ptr) return DRT_CUDA_OK;
    CU(cudaFreeHost(ptr));
    return DRT_CUDA_OK;
}

/* ------------------------------------------------------------------ one process, several devices */

struct drt_multi_state
{
    int      count = 0;
    uint32_t width = 0, height = 0;
    int      n = 0;
    bool     peers = false;                 /* every device can address every other one */
    int      device[DRT_MAX_PEERS] = {};
    drt_film staging[DRT_MAX_PEERS] = {};   /* on device g: count * slice pixels (the scattered exchange), or the whole film (no peer access) */
    drt_film slice[DRT_MAX_PEERS] = {};     /* on device g: its merged slice */
    uint32_t *flags[DRT_MAX_PEERS] = {};    /* on device g: one arrival word per rank */
    uint32_t *images[DRT_MAX_PEERS] = {};   /* on device g: the three 8-bit images of its slice, 3 x slice pixels (device 0 without peers: 3 x all pixels) */
    cudaStream_t stream[DRT_MAX_PEERS] = {};  /* render + scatter + signal */
    cudaStream_t copy[DRT_MAX_PEERS] = {};    /* wait + merge + read-back of a band, while the next band renders */
    uint32_t epoch = 0;
};

static void multi_free(drt_multi_state *m)
{
    if(!m) return;
    for(int g = 0; g < m->count; g += 1)
    {
        if(cudaSetDevice(m->device[g]) != cudaSuccess) { cudaGetLastError(); continue; }
        cudaFree(m->staging[g].sum); cudaFree(m->staging[g].mean); cudaFree(m->staging[g].m2); cudaFree(m->staging[g].filter);
        cudaFree(m->slice[g].sum); cudaFree(m->slice[g].mean); cudaFree(m->slice[g].m2); cudaFree(m->slice[g].filter);
        cudaFree(m->flags[g]); cudaFree(m->images[g]);
        if(m->stream[g]) cudaStreamDestroy(m->stream[g]);
        if(m->copy[g]) cudaStreamDestroy(m->copy[g]);
    }
    delete m;
}

void drt_exchange_release(drt_cuda_context *ctx)
{
    cudaFree(ctx->d_wait_timeouts); ctx->d_wait_timeouts = nullptr;
    multi_free(ctx->multi); ctx->multi = nullptr;
}

static int multi_prepare(drt_cuda_context **ctxs, int count, uint32_t width, uint32_t height, uint64_t slice, drt_multi_state **out)
{
    drt_multi_state *m = ctxs[0]->multi;
    bool same = m && m->count == count && m->width == width && m->height == height && m->n == ctxs[0]->n;
    for(int g = 0; same && g < count; g += 1) same = m->device[g] == ctxs[g]->device;
    if(same) { *out = m; return DRT_CUDA_OK; }
    multi_free(m);
    ctxs[0]->multi = nullptr;
    m = new drt_multi_state();
    m->count = count; m->width = width; m->height = height; m->n = ctxs[0]->n;
    for(int g = 0; g < count; g += 1) m->device[g] = ctxs[g]->device;
    m->peers = true;
    for(int g = 0; g < count && m->peers; g += 1)
        for(int h = 0; h < count && m->peers; h += 1)
        {
            if(h == g) continue;
            int can = 0;
            if(cudaDeviceCanAccessPeer(&can, ctxs[g]->device, ctxs[h]->device) != cudaSuccess || !can) { cudaGetLastError(); m->peers = false; }
        }
    int rc = DRT_CUDA_OK;
    const uint64_t npix = (uint64_t)width * height;
    for(int g = 0; g < count && rc == DRT_CUDA_OK; g += 1)
    {
        if(cudaSetDevice(ctxs[g]->device) != cudaSuccess) { rc = fail(DRT_CUDA_E_CUDA, "cudaSetDevice(%d)", ctxs[g]->device); break; }
        for(int h = 0; h < count && m->peers; h += 1)
        {
            if(h == g) continue;
            cudaError_t e = cudaDeviceEnablePeerAccess(ctxs[h]->device, 0);
            if(e == cudaErrorPeerAccessAlreadyEnabled) cudaGetLastError();
            else if(e != cudaSuccess) { rc = fail(DRT_CUDA_E_CUDA, "cudaDeviceEnablePeerAccess: %s", cudaGetErrorString(e)); break; }
        }
        if(rc != DRT_CUDA_OK) break;
        if(cudaStreamCreateWithFlags(&m->stream[g], cudaStreamNonBlocking) != cudaSuccess ||
           cudaStreamCreateWithFlags(&m->copy[g], cudaStreamNonBlocking) != cudaSuccess) { rc = fail(DRT_CUDA_E_CUDA, "cudaStreamCreate on device %d", ctxs[g]->device); break; }
        if(m->peers)
        {
            const uint32_t rows = (uint32_t)((slice * (uint64_t)count + width - 1) / width);
            const uint32_t srows = (uint32_t)((slice + width - 1) / width);
            rc = drt_cuda_film_alloc(ctxs[g], width, rows, &m->staging[g]);
            if(rc == DRT_CUDA_OK) rc = drt_cuda_film_alloc(ctxs[g], width, srows, &m->slice[g]);
            if(rc == DRT_CUDA_OK) rc = drt_cuda_buffer_alloc(ctxs[g], DRT_MAX_PEERS * sizeof(uint32_t), (void **)&m->flags[g]);
            if(rc == DRT_CUDA_OK) rc = drt_cuda_buffer_alloc(ctxs[g], 3 * (size_t)slice * sizeof(uint32_t), (void **)&m->images[g]);
        }
        else
        {
            /* no peer access: every device renders a whole local film; device 0 also holds a landing film for the others' */
            rc = drt_cuda_film_alloc(ctxs[g], width, height, &m->staging[g]);
            if(rc == DRT_CUDA_OK && g == 0) rc = drt_cuda_film_alloc(ctxs[0], width, height, &m->slice[0]);
            if(rc == DRT_CUDA_OK && g == 0) rc = drt_cuda_buffer_alloc(ctxs[0], 3 * (size_t)npix * sizeof(uint32_t), (void **)&m->images[0]);
        }
    }
    if(rc != DRT_CUDA_OK) { multi_free(m); return rc; }
    ctxs[0]->multi = m;
    *out = m;
    return DRT_CUDA_OK;
}

extern "C" int drt_cuda_render_host_multi_images(drt_cuda_context **ctxs, int count, const drt_render_params *params, const drt_film *out,
                                                 uint32_t *bgra_sum_host, uint32_t *bgra_mean_host, uint32_t *bgra_var_host);

extern "C" int drt_cuda_render_host_multi(drt_cuda_context **ctxs, int count, const drt_render_params *params, const drt_film *out)
{
    return drt_cuda_render_host_multi_images(ctxs, count, params, out, nullptr, nullptr, nullptr);
}

/* the three images of a whole film that sits on one device: three conversion kernels + three copies */
static int images_of_film(drt_cuda_context *ctx, const drt_film *film_device, uint32_t width, uint32_t height, uint32_t *scratch_device,
                          uint32_t *const host[3], cudaStream_t stream)
{
    const size_t npix = (size_t)width * height;
    for(int which = 0; which < 3; which += 1)
    {
        int rc = drt_cuda_film_to_rgb(ctx, film_device, width, height, which, nullptr, scratch_device + (size_t)which * npix, stream);
        if(rc != DRT_CUDA_OK) return rc;
        CU(cudaMemcpyAsync(host[which], scratch_device + (size_t)which * npix, npix * 4, cudaMemcpyDeviceToHost, stream));
    }
    return DRT_CUDA_OK;
}

extern "C" int drt_cuda_render_host_multi_images(drt_cuda_context **ctxs, int count, const drt_render_params *params, const drt_film *out,
                                                 uint32_t *bgra_sum_host, uint32_t *bgra_mean_host, uint32_t *bgra_var_host)
{
    const bool want_images = bgra_sum_host || bgra_mean_host || bgra_var_host;
    if(want_images && !(bgra_sum_host && bgra_mean_host && bgra_var_host)) return fail(DRT_CUDA_E_ARG, "give all three image buffers or none");
    uint32_t *const host_images[3] = { bgra_sum_host, bgra_mean_host, bgra_var_host };
    if(!ctxs || count < 1 || count > DRT_MAX_PEERS || !params || !film_complete(out))
        return fail(DRT_CUDA_E_ARG, "bad argument (1..%d contexts)", DRT_MAX_PEERS);
    for(int g = 0; g < count; g += 1)
    {
        if(!ctxs[g] || !ctxs[g]->have_scene) return fail(DRT_CUDA_E_STATE, "context %d has no scene", g);
        if(ctxs[g]->n != ctxs[0]->n) return fail(DRT_CUDA_E_ARG, "context %d holds another scene", g);
        for(int h = 0; h < g; h += 1) if(ctxs[h]->device == ctxs[g]->device) return fail(DRT_CUDA_E_ARG, "contexts %d and %d share device %d", h, g, ctxs[g]->device);
    }
    const uint32_t spp = params->sample_end > params->sample_begin ? params->sample_end - params->sample_begin : 0;
    /* fewer samples than devices: the surplus devices have nothing to render */
    if(spp < (uint32_t)count) count = spp > 0 ? (int)spp : 1;
    if(count == 1)
    {
        int rc1 = drt_cuda_render_host(ctxs[0], params, out);
        if(rc1 != DRT_CUDA_OK || !want_images) return rc1;
        /* the film render_host just produced is still in the library's device planes */
        const size_t np1 = (size_t)params->width * params->height;
        const drt_film dev = film_planes(ctxs[0]->d_film, np1, ctxs[0]->n);
        uint32_t *scratch = nullptr;
        CU(cudaSetDevice(ctxs[0]->device));
        CU(cudaMalloc(&scratch, 3 * np1 * 4));
        rc1 = images_of_film(ctxs[0], &dev, params->width, params->height, scratch, host_images, nullptr);
        if(rc1 == DRT_CUDA_OK && cudaDeviceSynchronize() != cudaSuccess) rc1 = fail(DRT_CUDA_E_CUDA, "image conversion failed");
        cudaFree(scratch);
        return rc1;
    }
    const size_t n = (size_t)ctxs[0]->n, npix = (size_t)params->width * params->height;
    if(npix == 0) return fail(DRT_CUDA_E_ARG, "bad image rectangle");
    const uint64_t slice = (npix + (size_t)count - 1) / (size_t)count;
    drt_multi_state *m = nullptr;
    int rc = multi_prepare(ctxs, count, params->width, params->height, slice, &m);
    if(rc != DRT_CUDA_OK) return rc;
    auto share = [&](int g) {
        drt_render_params p = *params;
        p.sample_begin = params->sample_begin + (uint32_t)((uint64_t)spp * g / count);
        p.sample_end = params->sample_begin + (uint32_t)((uint64_t)spp * (g + 1) / count);
        return p;
    };
    if(m->peers)
    {
        /* Everything below is enqueued without waiting.  The frame is rendered in bands -- the same part of every owner's slice per
         * band -- on each device's render stream (render + scatter, signal); on its copy stream the device waits for the band's
         * arrival flags, merges the band's part of its slice and reads it back over its own PCIe link while the next band renders.
         * Band boundaries in 1/16 of a slice, ever smaller, so that little is left to merge and copy after the last render. */
        static const int cut16[] = { 0, 4, 8, 12, 14, 15, 16 };
        const bool banded = spp / (uint32_t)count >= 32u && slice >= 64;
        const int nbands = banded ? 6 : 1;
        for(int b = 0; b < nbands && rc == DRT_CUDA_OK; b += 1)
        {
            const uint64_t b0 = banded ? slice * (uint64_t)cut16[b] / 16 : 0, b1 = banded ? slice * (uint64_t)cut16[b + 1] / 16 : slice;
            if(b1 <= b0) continue;
            m->epoch += 1;
            /* all signals of a band are enqueued before any wait for it */
            for(int g = 0; g < count && rc == DRT_CUDA_OK; g += 1)
            {
                drt_render_params p = share(g);
                rc = banded ? drt_cuda_render_device_scatter_band(ctxs[g], &p, m->staging, count, g, slice, b0, b1, b > 0, m->stream[g])
                            : drt_cuda_render_device_scatter(ctxs[g], &p, m->staging, count, g, slice, m->stream[g]);
                uint32_t *targets[DRT_MAX_PEERS];
                for(int o = 0; o < count; o += 1) targets[o] = m->flags[o] + g;
                if(rc == DRT_CUDA_OK) rc = drt_cuda_flags_signal(ctxs[g], targets, count, m->epoch, m->stream[g]);
            }
            for(int g = 0; g < count && rc == DRT_CUDA_OK; g += 1)
            {
                const uint64_t s0 = (uint64_t)g * slice < npix ? (uint64_t)g * slice : npix, s1 = (uint64_t)(g + 1) * slice < npix ? (uint64_t)(g + 1) * slice : npix;
                const uint64_t p0 = s0 + b0 < s1 ? s0 + b0 : s1, p1 = s0 + b1 < s1 ? s0 + b1 : s1;
                rc = drt_cuda_flags_wait(ctxs[g], m->flags[g], count, m->epoch, m->copy[g]);
                if(p1 <= p0) continue;
                /* the merge kernel indexes the images with the global pixel number: hand it the slice's local buffers shifted by s0 */
                uint32_t *img = want_images ? m->images[g] : nullptr;
                if(rc == DRT_CUDA_OK) rc = drt_cuda_film_merge_slices_local(ctxs[g], &m->slice[g], &m->staging[g], count, slice, params->width, params->height, p0, p1,
                                                                             img ? img - s0 : nullptr, img ? img + slice - s0 : nullptr, img ? img + 2 * slice - s0 : nullptr, m->copy[g]);
                if(rc == DRT_CUDA_OK) rc = drt_cuda_film_read_slice(ctxs[g], &m->slice[g], s0, p0, p1, out, m->copy[g]);
                for(int which = 0; which < 3 && img && rc == DRT_CUDA_OK; which += 1)
                    if(cudaMemcpyAsync(host_images[which] + p0, img + (size_t)which * slice + (p0 - s0), (size_t)(p1 - p0) * 4, cudaMemcpyDeviceToHost, m->copy[g]) != cudaSuccess)
                        rc = fail(DRT_CUDA_E_CUDA, "image read-back on device %d", ctxs[g]->device);
            }
        }
        for(int g = 0; g < count; g += 1)
        {
            cudaSetDevice(ctxs[g]->device);
            if((cudaStreamSynchronize(m->stream[g]) != cudaSuccess || cudaStreamSynchronize(m->copy[g]) != cudaSuccess) && rc == DRT_CUDA_OK)
                rc = fail(DRT_CUDA_E_CUDA, "device %d: %s", ctxs[g]->device, cudaGetErrorString(cudaGetLastError()));
        }
        for(int g = 0; g < count && rc == DRT_CUDA_OK; g += 1)
        {
            uint32_t gave_up = 0;
            rc = drt_cuda_flags_timeouts(ctxs[g], &gave_up);
            if(rc == DRT_CUDA_OK && gave_up) rc = fail(DRT_CUDA_E_CUDA, "device %d gave up waiting for a peer's film (%u waits)", ctxs[g]->device, gave_up);
        }
        return rc;
    }
    /* No peer access between the devices: whole films, merged one after the other on device 0 (cudaMemcpyPeer stages through the
     * host where it must).  Slower, same result. */
    for(int g = 0; g < count && rc == DRT_CUDA_OK; g += 1)
    {
        drt_render_params p = share(g);
        rc = drt_cuda_render_device(ctxs[g], &p, &m->staging[g], 0, m->stream[g]);
    }
    for(int g = 0; g < count; g += 1)
    {
        cudaSetDevice(ctxs[g]->device);
        if(cudaStreamSynchronize(m->stream[g]) != cudaSuccess && rc == DRT_CUDA_OK) rc = fail(DRT_CUDA_E_CUDA, "render on device %d failed", ctxs[g]->device);
    }
    cudaSetDevice(ctxs[0]->device);
    for(int g = 1; g < count && rc == DRT_CUDA_OK; g += 1)
    {
        cudaError_t e = cudaMemcpyPeer(m->slice[0].sum, ctxs[0]->device, m->staging[g].sum, ctxs[g]->device, npix * n * 4);
        if(e == cudaSuccess) e = cudaMemcpyPeer(m->slice[0].mean, ctxs[0]->device, m->staging[g].mean, ctxs[g]->device, npix * n * 4);
        if(e == cudaSuccess) e = cudaMemcpyPeer(m->slice[0].m2, ctxs[0]->device, m->staging[g].m2, ctxs[g]->device, npix * n * 4);
        if(e == cudaSuccess) e = cudaMemcpyPeer(m->slice[0].filter, ctxs[0]->device, m->staging[g].filter, ctxs[g]->device, npix * 4);
        if(e != cudaSuccess) { rc = fail(DRT_CUDA_E_CUDA, "cudaMemcpyPeer from device %d: %s", ctxs[g]->device, cudaGetErrorString(e)); break; }
        rc = drt_cuda_film_merge(ctxs[0], &m->staging[0], &m->slice[0], params->width, params->height, nullptr);
        if(rc == DRT_CUDA_OK && cudaDeviceSynchronize() != cudaSuccess) rc = fail(DRT_CUDA_E_CUDA, "merge on device %d failed", ctxs[0]->device);
    }
    if(rc == DRT_CUDA_OK) rc = drt_cuda_film_read_slice(ctxs[0], &m->staging[0], 0, 0, npix, out, nullptr);
    if(rc == DRT_CUDA_OK && want_images) rc = images_of_film(ctxs[0], &m->staging[0], params->width, params->height, m->images[0], host_images, nullptr);
    if(rc == DRT_CUDA_OK && cudaDeviceSynchronize() != cudaSuccess) rc = fail(DRT_CUDA_E_CUDA, "film read-back failed");
    return rc;
}
