/* csrc/drt_kernels_fast_adaptive.cu -- instantiates drt::render_kernel_adaptive<float, NS, 1, DEEP> (drt_render.cuh) for NS = 2, 3, 5, 8,
 * shallow and deep: adaptive sampling in kernel mode 1. */
#include "drt_render.cuh"

DRT_DEFINE_ADAPTIVE_LAUNCHERS(drt_launch_render_f32_fast_adaptive, 1)
