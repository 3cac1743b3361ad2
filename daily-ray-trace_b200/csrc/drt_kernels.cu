/*
 * csrc/drt_kernels.cu -- dispatch to the render kernel instantiations and the launch geometry they are compiled for.
 * The kernel itself is the template in drt_render.cuh.
 */
#include <cuda_runtime.h>
#include "drt_device.cuh"

#define DRT_DECLARE(NAME) cudaError_t NAME(const RenderLaunch &L, bool paired, int nslots, int grid, int warps, size_t smem, cudaStream_t stream)
DRT_DECLARE(drt_launch_render_f32_fast);    DRT_DECLARE(drt_launch_render_f32_fast_deep);
DRT_DECLARE(drt_launch_render_f32_classed); DRT_DECLARE(drt_launch_render_f32_classed_deep);
DRT_DECLARE(drt_launch_render_f32_general); DRT_DECLARE(drt_launch_render_f32_general_deep);
DRT_DECLARE(drt_launch_render_f64);         DRT_DECLARE(drt_launch_render_f64_deep);
#define DRT_DECLARE_ADAPTIVE(NAME) cudaError_t NAME(const RenderLaunch &L, int nslots, int grid, int warps, size_t smem, cudaStream_t stream)
DRT_DECLARE_ADAPTIVE(drt_launch_render_f32_fast_adaptive);    DRT_DECLARE_ADAPTIVE(drt_launch_render_f32_fast_adaptive_deep);
DRT_DECLARE_ADAPTIVE(drt_launch_render_f32_classed_adaptive); DRT_DECLARE_ADAPTIVE(drt_launch_render_f32_classed_adaptive_deep);
DRT_DECLARE_ADAPTIVE(drt_launch_render_f32_general_adaptive); DRT_DECLARE_ADAPTIVE(drt_launch_render_f32_general_adaptive_deep);

/* f64 geometry is the branch-flip diagnostic: it always runs the general kernel.  A launch whose records overflow to global memory
 * (L.deep_stride != 0) takes the deep instantiation of its mode.  Adaptive launches (L.adaptive; f32 geometry and one pixel per task,
 * which the C ABI checks) take render_kernel_adaptive. */
cudaError_t drt_launch_render(const RenderLaunch &L, bool f64_geometry, int mode, int nslots, int grid, int warps, size_t smem, cudaStream_t stream)
{
    const bool paired = L.pixels_per_task == 1, deep = L.deep_stride != 0;
    if(L.adaptive)
    {
        if(f64_geometry || !paired) return cudaErrorInvalidValue;
        if(mode == 1) return deep ? drt_launch_render_f32_fast_adaptive_deep(L, nslots, grid, warps, smem, stream) : drt_launch_render_f32_fast_adaptive(L, nslots, grid, warps, smem, stream);
        if(mode == 2) return deep ? drt_launch_render_f32_classed_adaptive_deep(L, nslots, grid, warps, smem, stream) : drt_launch_render_f32_classed_adaptive(L, nslots, grid, warps, smem, stream);
        return deep ? drt_launch_render_f32_general_adaptive_deep(L, nslots, grid, warps, smem, stream) : drt_launch_render_f32_general_adaptive(L, nslots, grid, warps, smem, stream);
    }
    if(f64_geometry) return deep ? drt_launch_render_f64_deep(L, paired, nslots, grid, warps, smem, stream) : drt_launch_render_f64(L, paired, nslots, grid, warps, smem, stream);
    if(mode == 1) return deep ? drt_launch_render_f32_fast_deep(L, paired, nslots, grid, warps, smem, stream) : drt_launch_render_f32_fast(L, paired, nslots, grid, warps, smem, stream);
    if(mode == 2) return deep ? drt_launch_render_f32_classed_deep(L, paired, nslots, grid, warps, smem, stream) : drt_launch_render_f32_classed(L, paired, nslots, grid, warps, smem, stream);
    return deep ? drt_launch_render_f32_general_deep(L, paired, nslots, grid, warps, smem, stream) : drt_launch_render_f32_general(L, paired, nslots, grid, warps, smem, stream);
}

int drt_render_cta_warps(bool f64_geometry, int mode)
{
    if(f64_geometry) return DRT_CTA_WARPS;
    return mode == 1 ? DRT_FAST_WARPS : mode == 2 ? DRT_CLASSED_WARPS : DRT_CTA_WARPS;
}

int drt_render_min_ctas(bool f64_geometry, int mode)
{
    if(f64_geometry) return DRT_GENERAL_CTAS;
    return mode == 1 ? DRT_MIN_CTAS : mode == 2 ? DRT_CLASSED_CTAS : DRT_GENERAL_CTAS;
}

size_t drt_render_smem_bytes(const RenderLaunch &L, bool f64_geometry, int warps, int nslots)
{
    size_t geom = f64_geometry ? sizeof(GeomT<double>) : sizeof(GeomT<float>);
    size_t off = (geom + 15) & ~size_t(15);
    off += (sizeof(SpdIndex) + 15) & ~size_t(15);
    off += (size_t)L.pool_words * 4;
    off += 16 * 8;
    off = (off + 15) & ~size_t(15);
    off += (size_t)warps * L.path_stride * DRT_WARP * 4;
    off += (size_t)warps * (3 * (size_t)nslots + 2) * DRT_WARP * 4;   /* film parking */
    return off;
}
