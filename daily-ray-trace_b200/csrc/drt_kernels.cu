/*
 * csrc/drt_kernels.cu -- dispatch to the render kernel instantiations and the shared memory a launch of them needs.
 * The kernel itself is the template in drt_render.cuh, its launch shapes are DRT_RENDER_SHAPE in drt_device.cuh.
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

/* the carve of the kernel body, without its pointers */
size_t drt_render_smem_bytes(const RenderLaunch &L, bool f64_geometry, int warps, int nslots)
{
#define DRT_SMEM_NO_POINTER(T, NAME, AT)
    DRT_RENDER_SMEM_CARVE(DRT_SMEM_NO_POINTER, f64_geometry ? sizeof(GeomT<double>) : sizeof(GeomT<float>), L.pool_words, warps, L.path_stride, nslots)
#undef DRT_SMEM_NO_POINTER
    return off;
}
