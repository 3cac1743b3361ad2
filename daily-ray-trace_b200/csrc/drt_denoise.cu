/*
 * csrc/drt_denoise.cu -- non-local-means denoising of a finished film guided by the film's own statistics (Rousselle, Knaus and
 * Zwicker, "Adaptive rendering with non-local means filtering", 2012).  drt_cuda.h states the filter; this file computes it.
 *
 *   denoise_guide_kernel   per pixel: luminance Y = sum w_l mean_l, its variance bound v = (sum w_l sqrt(max(0, M2_l / (n (n - 1)))))^2
 *                          and whether the pixel is usable (n >= 2, finite mean and M2, finite f32 Y and v), into three planes of the
 *                          context's scratch.  One warp per pixel, wavelengths across lanes (the adaptive rule's Y and err).
 *   denoise_filter_kernel  a CTA takes a 32 x 4 tile of output pixels and stages the guide of the tile and its r + f halo in shared
 *                          memory (border replicated).  It walks the search window one row of offsets (dy) at a time: the patch
 *                          distances of all 2r + 1 offsets of the row come from one separable box sum over the tile and its f halo,
 *                          then the spectra of the neighbours in that row are staged (all wavelengths, zero for unusable and outside
 *                          pixels) and accumulated.  Every thread holds the f32 sums of 4 adjacent pixels x up to 4 groups of 4
 *                          wavelengths in registers (packed f32x2), so each spectrum value read from shared memory feeds up to 4
 *                          pixels and each weight up to 16 wavelengths.  Sums run in a fixed order: no atomics, deterministic.
 */
#include <cuda_runtime.h>
#include "drt_device.cuh"

namespace drt {

constexpr int DN_TX = 32, DN_TY = 4, DN_TP = DN_TX * DN_TY;           /* output tile */
constexpr int DN_THREADS = 256;
constexpr int DN_KP = 4;                                              /* adjacent pixels of one row per thread */
constexpr int DN_SLOTS = DN_THREADS / (DN_TP / DN_KP);                /* threads per pixel group: 8 */
constexpr int DN_MAXG = (DRT_MAX_WAVELENGTHS + 4 * DN_SLOTS - 1) / (4 * DN_SLOTS);   /* groups of 4 wavelengths per thread */
static_assert(DN_THREADS % DN_TP == 0, "the distance pass gives every thread one fixed pixel");

/* Shared memory of denoise_filter_kernel in floats, for search radius r, patch radius f and n wavelengths. */
struct DenoiseLayout
{
    int np, gx, gy, ex, ey, sw;
    uint32_t w_off, s_off, u_off, words;
    __host__ __device__ DenoiseLayout(int r, int f, int n)
    {
        np = (n + 3) & ~3;                         /* staged spectra are float4 rows */
        gx = DN_TX + 2 * (r + f); gy = DN_TY + 2 * (r + f);   /* guide: tile + search + patch halo */
        ex = DN_TX + 2 * f; ey = DN_TY + 2 * f;    /* distance terms: tile + patch halo */
        sw = DN_TX + 2 * r;                        /* one staged row of neighbour spectra */
        const uint32_t spec = (uint32_t)(DN_TY * sw * np), eh = (uint32_t)((2 * r + 1) * (ex * ey + DN_TX * ey));
        w_off = (uint32_t)(3 * gx * gy + 3) & ~3u;                         /* Y, v, usable planes before it */
        s_off = w_off + (uint32_t)((2 * r + 2 * DN_KP - 1) * DN_TP);       /* weights [dx + r + KP - 1][pixel], zero outside |dx| <= r */
        u_off = (s_off + DN_TP + 3) & ~3u;                                  /* weight sums [pixel] */
        words = u_off + (spec > eh ? spec : eh);                            /* spectra of one dy, or the distance terms before them */
    }
};

namespace {
__device__ __forceinline__ unsigned long long dn_pk2(float a, float b) { unsigned long long r; asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(a), "f"(b)); return r; }
__device__ __forceinline__ void dn_upk2(unsigned long long v, float &a, float &b) { asm("mov.b64 {%0, %1}, %2;" : "=f"(a), "=f"(b) : "l"(v)); }
__device__ __forceinline__ void dn_fma2_acc(unsigned long long &acc, unsigned long long a, unsigned long long b)
{ asm("fma.rn.f32x2 %0, %1, %2, %0;" : "+l"(acc) : "l"(a), "l"(b)); }
}

__global__ void __launch_bounds__(256) denoise_guide_kernel(const float *yw, const float *mean, const float *m2, const float *filter,
                                                            uint32_t npix, uint32_t n, float *guide)
{
    const uint32_t lane = threadIdx.x & 31u;
    const uint32_t warps = (gridDim.x * blockDim.x) >> 5;
    for(uint32_t p = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; p < npix; p += warps)
    {
        const float cnt = filter[p];
        const float inv = 1.f / (cnt * (cnt - 1.f));
        float y = 0.f, e = 0.f;
        bool finite = true;
        for(uint32_t l = lane; l < n; l += 32)
        {
            const float m = mean[(size_t)p * n + l], s = m2[(size_t)p * n + l];
            finite = finite && isfinite(m) && isfinite(s);
            y = fmaf(yw[l], m, y);
            e = fmaf(yw[l], sqrtf(fmaxf(s * inv, 0.f)), e);   /* a negative M2 counts as zero variance */
        }
#pragma unroll
        for(int o = 16; o > 0; o >>= 1) { y += __shfl_xor_sync(0xffffffffu, y, o); e += __shfl_xor_sync(0xffffffffu, e, o); }
        const bool usable = __all_sync(0xffffffffu, finite) && cnt >= 2.f && isfinite(y) && isfinite(e * e);
        if(lane == 0)
        {
            guide[p] = usable ? y : 0.f;
            guide[npix + p] = usable ? e * e : 0.f;
            guide[2 * (size_t)npix + p] = usable ? 1.f : 0.f;
        }
    }
}

__global__ void __launch_bounds__(DN_THREADS) denoise_filter_kernel(const float *mean, const float *guide, uint32_t width, uint32_t height,
                                                                    uint32_t n, int r, int f, float kk, float *out)
{
    extern __shared__ __align__(16) float sm[];
    const DenoiseLayout L(r, f, (int)n);
    const int tid = threadIdx.x;
    const uint32_t tiles_x = (width + DN_TX - 1) / DN_TX;
    const int x0 = (int)(blockIdx.x % tiles_x) * DN_TX, y0 = (int)(blockIdx.x / tiles_x) * DN_TY;
    const int R = r + f, W = (int)width, H = (int)height;
    const size_t npix = (size_t)width * height;
    float *gY = sm, *gV = sm + L.gx * L.gy, *gU = sm + 2 * L.gx * L.gy;
    float *wt = sm + L.w_off, *wsum = sm + L.s_off, *u = sm + L.u_off;

    /* the guide of the tile and its halo, border replicated; the weight rows outside |dx| <= r are zero */
    for(int i = tid; i < L.gx * L.gy; i += DN_THREADS)
    {
        const int x = min(max(x0 - R + i % L.gx, 0), W - 1), y = min(max(y0 - R + i / L.gx, 0), H - 1);
        const size_t p = (size_t)y * width + x;
        gY[i] = guide[p]; gV[i] = guide[npix + p]; gU[i] = guide[2 * npix + p];
    }
    for(int i = tid; i < 2 * (DN_KP - 1) * DN_TP; i += DN_THREADS)
        wt[(i < (DN_KP - 1) * DN_TP ? 0 : (2 * r + 1) * DN_TP) + i] = 0.f;

    /* accumulation: pixels (px0 .. px0 + 3, ty) of the tile, wavelength groups 4 (slot + 8 g) .. + 3 */
    const int slot = tid % DN_SLOTS, pg = tid / DN_SLOTS;
    const int ty = pg / (DN_TX / DN_KP), px0 = (pg % (DN_TX / DN_KP)) * DN_KP, pix0 = ty * DN_TX + px0;
    unsigned long long acc[DN_MAXG][DN_KP][2];
#pragma unroll
    for(int g = 0; g < DN_MAXG; g += 1)
#pragma unroll
        for(int i = 0; i < DN_KP; i += 1) { acc[g][i][0] = 0ull; acc[g][i][1] = 0ull; }
    /* distances: one fixed pixel per thread, offsets dx = -r + (tid / TP) + 2 m */
    const int vpix = tid % DN_TP, vtx = vpix % DN_TX, vty = vpix / DN_TX;
    float wpart = 0.f;
    const int nd = 2 * r + 1, ecells = L.ex * L.ey, hcells = DN_TX * L.ey, side = 2 * f + 1;
    const float inv_area = 1.f / (float)(side * side);
    float *E = u, *Hs = u + nd * ecells;

    for(int dy = -r; dy <= r; dy += 1)
    {
        __syncthreads();   /* the guide is staged; the previous row's spectra are consumed */
        /* D(a, b) of every distance term of every offset of this row: a = tile + patch halo cell, b = a + (dx, dy) */
        for(int i = tid; i < nd * ecells; i += DN_THREADS)
        {
            const int dxi = i / ecells, c = i - dxi * ecells;
            const int ga = (c / L.ex + r) * L.gx + c % L.ex + r, gb = ga + dy * L.gx + dxi - r;
            const float ya = gY[ga], va = gV[ga], yb = gY[gb], vb = gV[gb], dY = ya - yb;
            E[i] = (dY * dY - (va + fminf(va, vb))) / (1e-10f + kk * (va + vb));
        }
        __syncthreads();
        for(int i = tid; i < nd * hcells; i += DN_THREADS)
        {
            const int dxi = i / hcells, c = i - dxi * hcells, hy = c / DN_TX, hx = c % DN_TX;
            const float *e = E + dxi * ecells + hy * L.ex + hx;
            float s = 0.f;
            for(int j = 0; j < side; j += 1) s += e[j];
            Hs[i] = s;
        }
        __syncthreads();
        for(int dxi = tid / DN_TP; dxi < nd; dxi += DN_THREADS / DN_TP)
        {
            const float *h = Hs + dxi * hcells + vty * DN_TX + vtx;
            float s = 0.f;
            for(int j = 0; j < side; j += 1) s += h[j * DN_TX];
            const int dx = dxi - r, qx = x0 + vtx + dx, qy = y0 + vty + dy;
            /* a NaN distance (inf - inf of two guides near FLT_MAX) takes weight 0: fmaxf would turn it into 0, a weight of 1 */
            const bool in = qx >= 0 && qx < W && qy >= 0 && qy < H && gU[(vty + dy + R) * L.gx + vtx + dx + R] != 0.f && !isnan(s);
            float w = in ? __expf(-fmaxf(0.f, s * inv_area)) : 0.f;
            if(dx == 0 && dy == 0) w = 1.f;
            wt[(dxi + DN_KP - 1) * DN_TP + vpix] = w;
            wpart += w;
        }
        __syncthreads();   /* the distance terms are consumed: their space takes the spectra */
        /* the spectra of row y0 + t + dy, x0 - r .. x0 + 31 + r, one warp per pixel; zero where the pixel takes no weight */
        for(int s = tid >> 5; s < DN_TY * L.sw; s += DN_THREADS / 32)
        {
            const int st = s / L.sw, sx = s % L.sw, qx = x0 - r + sx, qy = y0 + st + dy;
            const bool ok = qx >= 0 && qx < W && qy >= 0 && qy < H && gU[(st + dy + R) * L.gx + sx + f] != 0.f;
            const float *src = mean + ((size_t)qy * width + qx) * n;
            for(int l = tid & 31; l < L.np; l += 32) u[s * L.np + l] = (ok && l < (int)n) ? src[l] : 0.f;
        }
        __syncthreads();
        const float *srow = u + (ty * L.sw + px0) * L.np;
        for(int j = 0; j < 2 * r + DN_KP; j += 1, srow += L.np)
        {
            unsigned long long w2[DN_KP];
#pragma unroll
            for(int i = 0; i < DN_KP; i += 1) { const float w = wt[(j - i + DN_KP - 1) * DN_TP + pix0 + i]; w2[i] = dn_pk2(w, w); }
#pragma unroll
            for(int g = 0; g < DN_MAXG; g += 1)
            {
                const int wl = 4 * (slot + DN_SLOTS * g);
                if(wl >= (int)n) break;
                const float4 s = *reinterpret_cast<const float4 *>(srow + wl);
                const unsigned long long s01 = dn_pk2(s.x, s.y), s23 = dn_pk2(s.z, s.w);
#pragma unroll
                for(int i = 0; i < DN_KP; i += 1) { dn_fma2_acc(acc[g][i][0], w2[i], s01); dn_fma2_acc(acc[g][i][1], w2[i], s23); }
            }
        }
    }
    /* the weight sum of a pixel: the two threads of its even and odd offsets, in a fixed order */
    if(tid >= DN_TP) wsum[vpix] = wpart;
    __syncthreads();
    if(tid < DN_TP) wsum[vpix] += wpart;
    __syncthreads();

#pragma unroll
    for(int i = 0; i < DN_KP; i += 1)
    {
        const int x = x0 + px0 + i, y = y0 + ty;
        if(x >= W || y >= H) continue;
        const size_t at = ((size_t)y * width + x) * n;
        const bool usable = gU[(ty + R) * L.gx + px0 + i + R] != 0.f;
        const float ws = wsum[pix0 + i];
#pragma unroll
        for(int g = 0; g < DN_MAXG; g += 1)
        {
            const int wl = 4 * (slot + DN_SLOTS * g);
            if(wl >= (int)n) break;
            float v[4];
            dn_upk2(acc[g][i][0], v[0], v[1]); dn_upk2(acc[g][i][1], v[2], v[3]);
#pragma unroll
            for(int c = 0; c < 4; c += 1)
                if(wl + c < (int)n) out[at + wl + c] = usable ? __fdiv_rn(v[c], ws) : mean[at + wl + c];   /* unusable: copied bit for bit */
        }
    }
}

} // namespace drt

void drt_launch_denoise_guide(const float *yw, const float *mean, const float *m2, const float *filter, uint32_t npix, int n, float *guide,
                              int grid, cudaStream_t stream)
{
    drt::denoise_guide_kernel<<<grid, 256, 0, stream>>>(yw, mean, m2, filter, npix, (uint32_t)n, guide);
}

size_t drt_denoise_smem_bytes(int n, int search_radius, int patch_radius)
{
    return (size_t)drt::DenoiseLayout(search_radius, patch_radius, n).words * sizeof(float);
}

cudaError_t drt_launch_denoise_filter(const float *mean, const float *guide, uint32_t width, uint32_t height, int n, int search_radius,
                                      int patch_radius, float strength, float *out, cudaStream_t stream)
{
    const size_t smem = drt_denoise_smem_bytes(n, search_radius, patch_radius);
    cudaError_t e = cudaFuncSetAttribute(drt::denoise_filter_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if(e != cudaSuccess) return e;
    const uint64_t tiles = (uint64_t)((width + drt::DN_TX - 1) / drt::DN_TX) * ((height + drt::DN_TY - 1) / drt::DN_TY);
    drt::denoise_filter_kernel<<<(unsigned)tiles, drt::DN_THREADS, smem, stream>>>(mean, guide, width, height, (uint32_t)n, search_radius,
                                                                                  patch_radius, strength * strength, out);
    return cudaGetLastError();
}
