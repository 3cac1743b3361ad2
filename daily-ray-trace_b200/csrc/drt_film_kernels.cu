/*
 * csrc/drt_film_kernels.cu -- film epilogues and the FP32 peak probe.
 *
 *   film_to_rgb_kernel   K7: per pixel divide by the filter sum (daily_ray_trace.c:18-22), SPD -> XYZ -> "CIE RGB"
 *                        (spectrum.c:49-82), clamp + truncating 8-bit quantiser (win32_platform.c:136-147).
 *                        One warp per pixel, wavelengths across lanes, coalesced 128-byte row reads.
 *   film_merge_kernel    combines two films of the same pixels over disjoint sample sets: sum and filter add,
 *                        (count, mean, M2) merge by Chan et al.'s pairwise update.  `src` may be a peer GPU's memory
 *                        (P2P load over NVLink), which makes this the reduce step of sample-sharded multi-GPU renders.
 *   fma_peak_kernel      dependent-chain-free FFMA / FFMA2 loop used to MEASURE the FP32 roofline denominator.
 */
#include <cuda_runtime.h>
#include "drt_device.cuh"

namespace drt {

struct RgbTables
{
    int   n;
    float scale;                       /* wl_interval / sum(cmf_y * ref_white * wl_interval) */
    float xw[DRT_MAX_WAVELENGTHS];     /* cmf_x * ref_white */
    float yw[DRT_MAX_WAVELENGTHS];
    float zw[DRT_MAX_WAVELENGTHS];
};

__device__ __forceinline__ float warp_sum(float v)
{
#pragma unroll
    for(int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ float warp_max(float v)
{
#pragma unroll
    for(int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}

__global__ void __launch_bounds__(256) film_to_rgb_kernel(const RgbTables *tables, const float *plane, const float *filter,
                                                          int normalise_by_max, uint32_t npix, float *rgb, uint32_t *bgra)
{
    __shared__ RgbTables t;
    for(uint32_t i = threadIdx.x; i < sizeof(RgbTables) / 4; i += blockDim.x)
        reinterpret_cast<uint32_t *>(&t)[i] = reinterpret_cast<const uint32_t *>(tables)[i];
    __syncthreads();
    const uint32_t lane = threadIdx.x & 31u;
    const uint32_t warps = (gridDim.x * blockDim.x) >> 5;
    const uint32_t n = (uint32_t)t.n;
    for(uint32_t p = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; p < npix; p += warps)
    {
        const float *row = plane + (size_t)p * n;
        float v[DRT_MAX_SLOTS];
        float peak = 0.f;
#pragma unroll
        for(int k = 0; k < DRT_MAX_SLOTS; k += 1)
        {
            uint32_t wl = lane + k * 32;
            v[k] = (wl < n) ? row[wl] : 0.f;
            if(wl < n && v[k] > peak) peak = v[k];
        }
        float div = 1.f;
        if(filter) div = filter[p];
        if(normalise_by_max) div = warp_max(peak);      /* spectrum_normalise, spectrum.c:182-187 (0/0 -> NaN, Q17) */
        float x = 0.f, y = 0.f, z = 0.f;
#pragma unroll
        for(int k = 0; k < DRT_MAX_SLOTS; k += 1)
        {
            uint32_t wl = lane + k * 32;
            if(wl < n)
            {
                float s = v[k] / div;
                x = fmaf(t.xw[wl], s, x); y = fmaf(t.yw[wl], s, y); z = fmaf(t.zw[wl], s, z);
            }
        }
        x = warp_sum(x) * t.scale; y = warp_sum(y) * t.scale; z = warp_sum(z) * t.scale;
        float r = (2.3706743f * x) - (0.9000405f * y) - (0.4706338f * z);
        float gch = (-0.5138850f * x) + (1.4253036f * y) + (0.0885814f * z);
        float b = (0.0052982f * x) - (0.0146949f * y) + (1.0093968f * z);
        if(lane == 0)
        {
            if(rgb) { rgb[(size_t)p * 3 + 0] = r; rgb[(size_t)p * 3 + 1] = gch; rgb[(size_t)p * 3 + 2] = b; }
            if(bgra)
            {
                float ch[3] = { r, gch, b };
                uint32_t out = 0;
#pragma unroll
                for(int c = 0; c < 3; c += 1)
                {
                    float q = ch[c];
                    if(!(q == q)) q = 0.f;
                    q = fminf(fmaxf(q, 0.f), 1.f);
                    out |= ((uint32_t)(q * 255.0f) & 255u) << (8 * (2 - c));
                }
                bgra[p] = out;
            }
        }
    }
}

/* One thread per (pixel, wavelength); grid-stride, fully coalesced on both films. */
__global__ void __launch_bounds__(256) film_merge_kernel(FilmPtrs dst, FilmPtrs src, uint32_t n, size_t total)
{
    size_t stride = (size_t)gridDim.x * blockDim.x;
    for(size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += stride)
    {
        size_t p = i / n;
        float na = dst.filter[p], nb = src.filter[p];
        float nab = na + nb;
        float ma = dst.mean[i], mb = src.mean[i];
        float delta = mb - ma;
        /* correctly rounded: the build's -prec-div=false division can give nb / nb != 1, and merging into an empty film must be exact */
        float wb = (nab > 0.f) ? __fdiv_rn(nb, nab) : 0.f;
        dst.mean[i] = fmaf(delta, wb, ma);
        dst.m2[i] = dst.m2[i] + src.m2[i] + delta * delta * na * wb;
        dst.sum[i] = dst.sum[i] + src.sum[i];
    }
}

__global__ void __launch_bounds__(256) film_merge_filter_kernel(float *dst, const float *src, size_t npix)
{
    size_t stride = (size_t)gridDim.x * blockDim.x;
    for(size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < npix; i += stride) dst[i] = dst[i] + src[i];
}


/* Fused multi-GPU epilogue.  `set` holds the partial films of all ranks (own memory and peer memory mapped through
 * CUDA IPC / P2P); every warp takes pixels of [pixel_begin, pixel_end), reads each rank's (count, sum, mean, M2) row
 * straight over NVLink, combines them with Chan's update in registers, writes the merged planes to `dst` (which may
 * itself be the root rank's memory) and, in the same pass, converts the three images of win32_main.c:150-152
 * (sum/filter, mean, M2/max) to packed BGRA.  One kernel replaces reduce-scatter + gather + three conversions. */
struct FilmSet { int count; FilmPtrs film[16]; };

template <int CHUNK>
__global__ void __launch_bounds__(256) film_gather_merge_kernel(const RgbTables *tables, FilmSet set, FilmPtrs dst, uint32_t pixel_begin,
                                                                uint32_t pixel_end, uint32_t src_base, uint32_t dst_base, uint32_t *bgra_sum, uint32_t *bgra_mean, uint32_t *bgra_var)
{
    __shared__ RgbTables t;
    for(uint32_t i = threadIdx.x; i < sizeof(RgbTables) / 4; i += blockDim.x)
        reinterpret_cast<uint32_t *>(&t)[i] = reinterpret_cast<const uint32_t *>(tables)[i];
    __syncthreads();
    const uint32_t lane = threadIdx.x & 31u;
    const uint32_t warps = (gridDim.x * blockDim.x) >> 5;
    const uint32_t n = (uint32_t)t.n;
    for(uint32_t p = pixel_begin + ((blockIdx.x * blockDim.x + threadIdx.x) >> 5); p < pixel_end; p += warps)
    {
        float cnt = 0.f, sum[DRT_MAX_SLOTS], mean[DRT_MAX_SLOTS], m2[DRT_MAX_SLOTS];
#pragma unroll
        for(int k = 0; k < DRT_MAX_SLOTS; k += 1) { sum[k] = 0.f; mean[k] = 0.f; m2[k] = 0.f; }
        /* ranks are taken CHUNK at a time: all their loads (peer memory over NVLink) are issued before any is consumed */
        for(int g0 = 0; g0 < set.count; g0 += CHUNK)
        {
            float nb[CHUNK], rs[CHUNK][DRT_MAX_SLOTS], rm[CHUNK][DRT_MAX_SLOTS], rv[CHUNK][DRT_MAX_SLOTS];
#pragma unroll
            for(int c = 0; c < CHUNK; c += 1)
            {
                const bool on = g0 + c < set.count;
                const FilmPtrs &f = set.film[on ? g0 + c : g0];
                nb[c] = on ? f.filter[p - src_base] : 0.f;
#pragma unroll
                for(int k = 0; k < DRT_MAX_SLOTS; k += 1)
                {
                    uint32_t wl = lane + k * 32;
                    size_t at = (size_t)(p - src_base) * n + wl;   /* sources are indexed from src_base (0 for whole films, the slice start for staged slices) */
                    bool ld = on && wl < n;
                    rs[c][k] = ld ? f.sum[at] : 0.f; rm[c][k] = ld ? f.mean[at] : 0.f; rv[c][k] = ld ? f.m2[at] : 0.f;
                }
            }
#pragma unroll
            for(int c = 0; c < CHUNK; c += 1)
            {
                float nab = cnt + nb[c];
                float wb = (nab > 0.f) ? __fdiv_rn(nb[c], nab) : 0.f;   /* exact 1 for the first non-empty film (see film_merge_kernel) */
#pragma unroll
                for(int k = 0; k < DRT_MAX_SLOTS; k += 1)
                {
                    float delta = rm[c][k] - mean[k];
                    m2[k] = m2[k] + rv[c][k] + delta * delta * cnt * wb;
                    mean[k] = fmaf(delta, wb, mean[k]);
                    sum[k] += rs[c][k];
                }
                cnt = nab;
            }
        }
        float peak = 0.f;
#pragma unroll
        for(int k = 0; k < DRT_MAX_SLOTS; k += 1)
        {
            uint32_t wl = lane + k * 32;
            if(wl >= n) continue;
            size_t at = (size_t)(p - dst_base) * n + wl;   /* the destination is indexed from dst_base (0: a whole film) */
            dst.sum[at] = sum[k]; dst.mean[at] = mean[k]; dst.m2[at] = m2[k];
            if(m2[k] > peak) peak = m2[k];
        }
        if(lane == 0) dst.filter[p - dst_base] = cnt;
        if(!bgra_sum) continue;
        peak = warp_max(peak);
        float acc[9];
#pragma unroll
        for(int i = 0; i < 9; i += 1) acc[i] = 0.f;
#pragma unroll
        for(int k = 0; k < DRT_MAX_SLOTS; k += 1)
        {
            uint32_t wl = lane + k * 32;
            if(wl >= n) continue;
            float v[3] = { sum[k] / cnt, mean[k], m2[k] / peak };
#pragma unroll
            for(int img = 0; img < 3; img += 1)
            {
                acc[img * 3 + 0] = fmaf(t.xw[wl], v[img], acc[img * 3 + 0]);
                acc[img * 3 + 1] = fmaf(t.yw[wl], v[img], acc[img * 3 + 1]);
                acc[img * 3 + 2] = fmaf(t.zw[wl], v[img], acc[img * 3 + 2]);
            }
        }
#pragma unroll
        for(int i = 0; i < 9; i += 1) acc[i] = warp_sum(acc[i]) * t.scale;
        if(lane < 3)
        {
            float x = acc[lane * 3 + 0], y = acc[lane * 3 + 1], z = acc[lane * 3 + 2];
            float ch[3] = { (2.3706743f * x) - (0.9000405f * y) - (0.4706338f * z),
                            (-0.5138850f * x) + (1.4253036f * y) + (0.0885814f * z),
                            (0.0052982f * x) - (0.0146949f * y) + (1.0093968f * z) };
            uint32_t out = 0;
#pragma unroll
            for(int c = 0; c < 3; c += 1)
            {
                float q = ch[c];
                if(!(q == q)) q = 0.f;
                q = fminf(fmaxf(q, 0.f), 1.f);
                out |= ((uint32_t)(q * 255.0f) & 255u) << (8 * (2 - c));
            }
            uint32_t *img = (lane == 0) ? bgra_sum : (lane == 1) ? bgra_mean : bgra_var;
            img[p] = out;
        }
    }
}

template <int PACKED>
__global__ void __launch_bounds__(256) fma_peak_kernel(float *out, int iters, float a, float b)
{
    float acc[16];
#pragma unroll
    for(int k = 0; k < 16; k += 1) acc[k] = (float)(threadIdx.x + k);
    for(int i = 0; i < iters; i += 1)
    {
        if(PACKED)
        {
#pragma unroll
            for(int k = 0; k < 16; k += 2)
            {
                unsigned long long v, aa, bb;
                asm volatile("mov.b64 %0, {%1, %2};" : "=l"(v) : "f"(acc[k]), "f"(acc[k + 1]));
                asm volatile("mov.b64 %0, {%1, %1};" : "=l"(aa) : "f"(a));
                asm volatile("mov.b64 %0, {%1, %1};" : "=l"(bb) : "f"(b));
                asm volatile("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(v) : "l"(v), "l"(aa), "l"(bb));
                asm volatile("mov.b64 {%0, %1}, %2;" : "=f"(acc[k]), "=f"(acc[k + 1]) : "l"(v));
            }
        }
        else
        {
#pragma unroll
            for(int k = 0; k < 16; k += 1) acc[k] = fmaf(acc[k], a, b);
        }
    }
    float s = 0.f;
#pragma unroll
    for(int k = 0; k < 16; k += 1) s += acc[k];
    if(s == 123.456f) out[0] = s;   /* keeps the loop alive without writing */
}

} // namespace drt

void drt_launch_film_to_rgb(const void *tables, const float *plane, const float *filter, int normalise_by_max, uint32_t npix,
                            float *rgb, uint32_t *bgra, int grid, cudaStream_t stream)
{
    drt::film_to_rgb_kernel<<<grid, 256, 0, stream>>>(reinterpret_cast<const drt::RgbTables *>(tables), plane, filter,
                                                     normalise_by_max, npix, rgb, bgra);
}

void drt_launch_film_merge(FilmPtrs dst, FilmPtrs src, uint32_t n, size_t npix, int grid, cudaStream_t stream)
{
    drt::film_merge_kernel<<<grid, 256, 0, stream>>>(dst, src, n, npix * n);
    /* filter planes are read by the spectral merge above: update them only after it, on the same stream */
    drt::film_merge_filter_kernel<<<grid, 256, 0, stream>>>(dst.filter, src.filter, npix);
}

void drt_launch_fma_peak(int packed, float *out, int iters, int grid, cudaStream_t stream)
{
    if(packed) drt::fma_peak_kernel<1><<<grid, 256, 0, stream>>>(out, iters, 0.999f, 0.001f);
    else       drt::fma_peak_kernel<0><<<grid, 256, 0, stream>>>(out, iters, 0.999f, 0.001f);
}

void drt_launch_film_gather_merge(const void *tables, int count, const FilmPtrs *films, FilmPtrs dst, uint32_t pixel_begin, uint32_t pixel_end,
                                  uint32_t src_base, uint32_t dst_base, uint32_t *bgra_sum, uint32_t *bgra_mean, uint32_t *bgra_var, int grid, cudaStream_t stream)
{
    drt::FilmSet set;
    set.count = count;
    for(int i = 0; i < count && i < 16; i += 1) set.film[i] = films[i];
    if(count <= 2)
        drt::film_gather_merge_kernel<2><<<grid, 256, 0, stream>>>(reinterpret_cast<const drt::RgbTables *>(tables), set, dst, pixel_begin, pixel_end, src_base, dst_base,
                                                                  bgra_sum, bgra_mean, bgra_var);
    else
        drt::film_gather_merge_kernel<4><<<grid, 256, 0, stream>>>(reinterpret_cast<const drt::RgbTables *>(tables), set, dst, pixel_begin, pixel_end, src_base, dst_base,
                                                                  bgra_sum, bgra_mean, bgra_var);
}

size_t drt_rgb_tables_bytes(void) { return sizeof(drt::RgbTables); }
size_t drt_rgb_tables_yw_offset(void) { return offsetof(drt::RgbTables, yw); }

void drt_fill_rgb_tables(void *dst_host, const drt_tables *t)
{
    drt::RgbTables *r = reinterpret_cast<drt::RgbTables *>(dst_host);
    r->n = t->num_wavelengths;
    double norm = 0.0;
    for(int i = 0; i < t->num_wavelengths; i += 1) norm += (t->cmf_y[i] * t->ref_white[i]);
    norm *= t->wl_interval;
    r->scale = (float)(t->wl_interval / norm);
    for(int i = 0; i < DRT_MAX_WAVELENGTHS; i += 1)
    {
        bool in = i < t->num_wavelengths;
        r->xw[i] = in ? (float)(t->cmf_x[i] * t->ref_white[i]) : 0.f;
        r->yw[i] = in ? (float)(t->cmf_y[i] * t->ref_white[i]) : 0.f;
        r->zw[i] = in ? (float)(t->cmf_z[i] * t->ref_white[i]) : 0.f;
    }
}
