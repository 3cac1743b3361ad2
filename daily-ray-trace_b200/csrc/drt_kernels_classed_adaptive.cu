/* csrc/drt_kernels_classed_adaptive.cu -- instantiates drt::render_kernel_adaptive<float, NS, 2, DEEP> (drt_render.cuh) for NS = 2, 3, 5, 8,
 * shallow and deep: adaptive sampling in kernel mode 2. */
#define DRT_PHILOX_ROLLED 1   /* this kernel is bound by instruction fetch (hot code > 32 KB): smaller beats straight-line */
#include "drt_render.cuh"

DRT_DEFINE_ADAPTIVE_LAUNCHERS(drt_launch_render_f32_classed_adaptive, 2)
