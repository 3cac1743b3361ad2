/*
 * csrc/drt_device.cuh -- device-side scene layout and launch descriptors.
 *
 * The reference's AoS scene with function pointers (daily_ray_trace.h:78-170) becomes three flat blocks that
 * every CTA stages once into shared memory:
 *   GeomT<R>   surfaces SoA (precomputed plane frames), per-material scalars and lobe lists, in the arithmetic
 *              type R of the geometric phase (float by default, double for the branch-flip diagnostic)
 *   SpdIndex   material -> row of the spectrum pool for each of its six SPDs (row 0 is all zeros)
 *   pool       nrows x NPAD floats, NPAD = 32 * (wavelength slots per lane)
 */
#pragma once
#include <stdint.h>
#include "drt_scene.h"

#define DRT_WARP 32
#define DRT_MAX_SLOTS 4            /* ceil(DRT_MAX_WAVELENGTHS / 32): full-warp wavelength layout of the film epilogue kernels */
#define DRT_HALF 16                /* phase 2 of the render kernel: a path is shaded by a HALF warp, lane l16 holds wavelengths l16 + 16k */
#define DRT_MAX_HALF_SLOTS 8       /* ceil(DRT_MAX_WAVELENGTHS / 16) */
#ifndef DRT_CTA_WARPS
#define DRT_CTA_WARPS 8      /* warps per CTA of the general kernel */
#endif
#ifndef DRT_FAST_WARPS
#define DRT_FAST_WARPS 14     /* warps per CTA of the ALLFAST kernel: 2 CTAs x 14 warps x 72 registers per SM (measured: 8 warps 6.7, 12: 9.70, 14: 9.79, 16: 9.65 G paths/s) */
#endif
#ifndef DRT_CLASSED_WARPS
#define DRT_CLASSED_WARPS 16   /* warps per CTA of the classed kernel: 2 CTAs x 16 warps x 64 registers (measured on cornell_plane_light, G paths/s at
                                * 64 spp: 10 warps 3.96, 12: 4.09, 14: 4.34, 16: 4.53; with the phase gates 16 x 2: 5.04, 32 x 1: 4.97, 28 x 1: 4.79) */
#endif
#ifndef DRT_CLASSED_CTAS
#define DRT_CLASSED_CTAS 2     /* resident CTAs per SM the classed / the general kernel is compiled for */
#endif
#ifndef DRT_GENERAL_CTAS
#define DRT_GENERAL_CTAS 2
#endif
#ifndef DRT_LOCKSTEP
#define DRT_LOCKSTEP 2         /* bit mask of kernel modes whose CTAs run their phases in lockstep (drt_render.cuh): bit 1 = the classed kernel
                                * (measured +15 %: its hot code is 38 KB against a 32 KB instruction cache); bit 0 = the general kernel
                                * (measured -26 % on stress_all: its phase-2 times differ too much between warps); bit 2 = the plastic-only kernel */
#endif
#ifndef DRT_GATE_PATIENCE_CYCLES
/* A phase gate gives up after this many SM clock cycles (about 10 ms at 1.97 GHz; a phase takes 50 - 200 us) and switches the
 * CTA's gates off: lockstep is a performance aid, never a dependency.  Multi-GPU renders (scatter_count > 1) start with the gates
 * off: bench.py --scene cornell_plane_light --gpus 2/4/8 did not complete in the round's last GPU session (cause not found before
 * the GPU budget ran out; the same kernel passes every single-device and in-process two-device test), and an untested multi-rank
 * combination is not worth 13 % -- see DESIGN.md section 9. */
#define DRT_GATE_PATIENCE_CYCLES 20000000ll
#endif
#ifndef DRT_GATE_SUSPEND_NS
#define DRT_GATE_SUSPEND_NS 20000u   /* suspend-time hint of a phase gate's mbarrier.try_wait */
#endif
#define DRT_CTA_THREADS (DRT_CTA_WARPS * DRT_WARP)
#ifndef DRT_MIN_CTAS
#define DRT_MIN_CTAS 2        /* resident CTAs per SM the render kernels are compiled for (__launch_bounds__) */
#endif

/* Spectral basis a BSDF evaluation is expressed in (eval_weights in drt_kernels.cu).  A material's lobe list fixes
 * which of the seven can ever be non-zero (bmask); only those weights are stored in a path record, in this order,
 * followed by the micro-normal cosine when BK_COND_MN is present. */
enum { DRT_CLASS_PLASTIC = 0, DRT_CLASS_SPECULAR = 1, DRT_CLASS_ROUGH = 2, DRT_CLASS_GENERAL = 3 };
enum { BK_CONST = 0, BK_DIFFUSE, BK_GLOSSY, BK_MIRROR, BK_DIEL_R, BK_COND_ON, BK_COND_MN, BK_COUNT };

/* one surface as four 16-byte (f32) / 32-byte (f64) vectors, so that the intersection loop issues vector shared-memory loads */
template <typename R> struct alignas(16) R4 { R x, y, z, w; };
template <typename R> struct alignas(8) R2 { R x, y; };

template <typename R>
struct GeomT
{
    /* intersectable surfaces regrouped by type: slots [0, nplanes) are planes, [nplanes, nplanes + nspheres) spheres;
     * sid[slot] is the surface's index in the scene (ties in distance go to the lower scene index, Q21).
     * The planes come in four groups: axis-aligned rectangles with normal +-x, +-y, +-z (nax[0..2] of them, every Cornell
     * wall), then planes in general position.  An axis-aligned rectangle with normal axis a and in-plane axes b < c is
     * AX4[slot] = { p_a, centre_b, half extent_b, centre_c }, AXH[slot] = { half extent_c, scene index as a number }. */
    int   nplanes, nspheres, pad2, pad3;
    int   nax[4];                  /* [3] unused */
    /* Inside each plane group the BOUNDARY planes come first: planes with the whole scene in one of their closed half-spaces (every
     * wall of a room).  A segment between two points of the scene can meet such a plane only at its end points, where the
     * reference's shadow test never reports a hit (origin pushed 1e-4 along the ray, Q2; far end excluded by vis_dist,
     * daily_ray_trace.c:244-250), so shadow rays skip them: nax_b[0..2] of the axis groups, nax_b[3] of the general planes. */
    int   nax_b[4];
    R4<R> AX4[DRT_MAX_SURFACES];
    R2<R> AXH[DRT_MAX_SURFACES];
    int   sid[DRT_MAX_SURFACES];
    R4<R> N4[DRT_MAX_SURFACES];    /* plane normal | w unused */
    R4<R> P4[DRT_MAX_SURFACES];    /* position | w = sphere radius */
    R4<R> U4[DRT_MAX_SURFACES];    /* normalised bounds vector u | w = |u| */
    R4<R> V4[DRT_MAX_SURFACES];    /* normalised bounds vector v | w = |v| */
    int nsurf, nlights, base_mat, escape_mat, nmat, n, eval_words, pad1;
    R   trans_num, trans_den;      /* (630 - w0), (w1 - w0) of value_at_wl, spectrum.c:150-162 */
    int type[DRT_MAX_SURFACES], mat[DRT_MAX_SURFACES], light_surf[DRT_MAX_SURFACES];
    R   px[DRT_MAX_SURFACES], py[DRT_MAX_SURFACES], pz[DRT_MAX_SURFACES], rad[DRT_MAX_SURFACES];
    R   nx[DRT_MAX_SURFACES], ny[DRT_MAX_SURFACES], nz[DRT_MAX_SURFACES];
    R   unx[DRT_MAX_SURFACES], uny[DRT_MAX_SURFACES], unz[DRT_MAX_SURFACES], ulen[DRT_MAX_SURFACES];
    R   vnx[DRT_MAX_SURFACES], vny[DRT_MAX_SURFACES], vnz[DRT_MAX_SURFACES], vlen[DRT_MAX_SURFACES];
    R   ux[DRT_MAX_SURFACES], uy[DRT_MAX_SURFACES], uz[DRT_MAX_SURFACES];
    R   vx[DRT_MAX_SURFACES], vy[DRT_MAX_SURFACES], vz[DRT_MAX_SURFACES];
    R   light_pdf[DRT_MAX_SURFACES];
    /* materials */
    int mflags[DRT_MAX_MATERIALS];   /* bit0 is_black_body, bit1 is_emissive */
    /* Shading class of the compact-record kernels (DRT_CLASS_*): what one bounce on this material needs in its 4-word record.
     *   PLASTIC   lobes all bp_diffuse / bp_glossy: NEE and sampled-direction weights (w_d, w_g) of the material's D, G block
     *   SPECULAR  lobes all match-gated (mirror, fs_conductor, fs_dielectric_R / _T) over ONE spectral basis X (mirror spectrum,
     *             dielectric R(on_dot) or conductor F(on_dot)): next-event estimation contributes nothing, the sampled direction
     *             multiplies the throughput by c0 + c1 X
     *   ROUGH     ct_conductor only: w F(cos) with the micro-normal cosine of each evaluation
     *   GENERAL   anything else (the general kernel) */
    int mclass[DRT_MAX_MATERIALS];
    /* SPECULAR: every lobe is gated on `in` being the exact reflection (match 1) or refraction (match 2) direction, so the
     * bdsf() sum over the lobe list -- stale scratch values included, Q7 -- is one of three constant pairs (c0, c1) of
     * c0 + c1 X, tabulated at upload by walking the lobe list exactly as eval_weights_general does: spec_c[m][match] */
    float spec_c[DRT_MAX_MATERIALS][3][2];
    float ct_mult[DRT_MAX_MATERIALS];   /* ROUGH: how many times ct_conductor_bdsf is listed */
    int bmask[DRT_MAX_MATERIALS];    /* bit k: basis kind k can be produced by this material's lobe list */
    int nlobes[DRT_MAX_MATERIALS], dirf[DRT_MAX_MATERIALS];
    unsigned char lobes[DRT_MAX_MATERIALS][DRT_MAX_LOBES];
    R   shin[DRT_MAX_MATERIALS], rough[DRT_MAX_MATERIALS];
    R   n630[DRT_MAX_MATERIALS];                                  /* value_at_wl(refract, 630) */
    R   refr_a[DRT_MAX_MATERIALS], refr_b[DRT_MAX_MATERIALS];     /* refract samples bracketing 630 nm */
    /* camera, daily_ray_trace.h:158-170 */
    R   fwd[3], right[3], up[3], ap_pos[3], film_bl[3];
    R   ap_radius, focal_depth, pixel_w, pixel_h;
    R   lens_rot[9];
};

struct SpdIndex
{
    int n, nslots, npad, nrows;
    int row[DRT_MAX_MATERIALS][DRT_SPD_COUNT];
    /* Plastic bounces under a scene's only light (every kernel mode): word offset (multiple of 4) of the material's D, G block, 0 if
     * it has none -- the diffuse and glossy rows D, G, each times its lobe's multiplicity, laid out so that a half-warp lane fetches a
     * slot pair with one 16-byte load that lands in f32x2 register pairs.  For lane l, chunk p (a float4 at index p*16 + l) =
     * { D[2p], D[2p+1], G[2p], G[2p+1] }, and for an odd last slot s the last chunk = { D[s], G[s], 0, 0 }: ceil(nslots / 2) * 64
     * words.  light_pairs = word offset of the light's emission E in the same pairing: float2 { E[2p], E[2p+1] } at index p*16 + l,
     * { E[s], 0 } for an odd last slot. */
    int plastic2[DRT_MAX_MATERIALS];
    int light_pairs, pad[3];
    /* Fresnel inputs per wavelength, precomputed in f64 at upload for the two orientations a surface can be met in (0: from the
     * base medium, 1: from inside, Q11), as plain pool rows (word offsets; 0 = absent): with ir / tr / te the incident refraction,
     * transmitting refraction and transmitting extinction of bdsf.c:44-101,
     *   [0] rel  = ir / tr                                    dielectric (fresnel_dielectric_rel)
     *   [1] condA = (tr / ir)^2 - (te / ir)^2   [2] condB = 4 (tr / ir)^2 (te / ir)^2          conductor (fresnel_conductor_ab) */
    int fres[DRT_MAX_MATERIALS][2][3];
};

struct FilmPtrs { float *sum, *filter, *mean, *m2; };
#define DRT_MAX_PEERS 16

struct DeviceStats
{
    unsigned long long paths, closest_rays, shadow_rays, shaded_bounces, rng_draws;
    unsigned long long terminated_at_depth[8];
    unsigned long long reached_depth_cap;
#ifdef DRT_PHASE_CLOCKS
    /* diagnostic builds only: SM-clock cycles the warps spent in each part of a batch (DRT_PHASE_* in drt_render.cuh) */
    unsigned long long phase_clocks[4];
#endif
};

/* Path record in shared memory, one row per path slot (word w of slot s at rec[s*path_stride + w]; path_stride is 4 times an
 * odd number, so the 16-byte stores of 32 lanes and the scalar stores of 8 consecutive lanes are bank-conflict free):
 *   word 0            number of bounce records
 *   word 1            vignette factor
 *   words 2, 3        unused (bounces start 16-byte aligned)
 *   per bounce, general   [0] header: kind(2) | 0<<2 | surface material(5)<<3 | media swapped<<8 | light visibility mask(16)<<16
 *                         [1] on_dot
 *                         nlights x { eval weights (eval_words), light scale k }      next-event estimation
 *                         eval weights (eval_words)                                   sampled direction, x 1/pdf
 *   per bounce, fast      two-lobe plastic under the scene's only light:
 *                         [0] header: kind(2) | 1<<2 | D, G block word offset (SpdIndex::plastic2, a multiple of 4)<<2
 *                         [1] w_diffuse * k  [2] w_glossy * k   (next-event estimation, 0 when the light is hidden)
 *                         [4] w_diffuse / pdf [5] w_glossy / pdf (sampled direction)
 *   bounce_words is a multiple of 4 and at least 8.
 * Compact records of the plastic-only and the classed kernel (one light, which is the scene's only emitter):
 *   word 0, 1         number of bounce records | (emitter material + 1) << 16, vignette factor
 *   from word 2       one 16-bit header per bounce: class (bits 0-1, DRT_CLASS_*) and
 *                       PLASTIC   the word offset of the material's D, G block (SpdIndex::plastic2, a multiple of 4: class bits 0)
 *                       SPECULAR  basis << 2 (0 mirror spectrum, 1 dielectric R, 2 conductor F) | inside << 4 | material << 5
 *                       ROUGH     inside << 4 | material << 5
 *   from head_words   per bounce four words:
 *                       PLASTIC   { w_diffuse k, w_glossy k (next-event estimation), w_diffuse / pdf, w_glossy / pdf (sampled direction) }
 *                       SPECULAR  { c0 / pdf, c1 / pdf, on_dot, - }
 *                       ROUGH     { w k, micro-normal cosine (next-event estimation; w = 0 when the light is hidden), w / pdf, cosine } */
struct RenderLaunch
{
    const void     *geom;          /* GeomT<float> or GeomT<double> in global memory */
    const SpdIndex *spd_index;
    const float    *pool;
    FilmPtrs        film;
    float          *path_dump;     /* optional per-path spectra, [pixel_local][sample][N] */
    float          *record_dump;   /* optional per-path record words, [pixel_local][sample][path_words] (diagnostics) */
    DeviceStats    *stats;
    unsigned int   *task_counter;
    uint32_t width, height;
    uint32_t x0, y0, x1, y1;       /* pixel rectangle rendered (whole image for a film render) */
    uint32_t sample_begin, sample_end;
    uint32_t max_depth;
    int32_t  pixel_scheme;
    uint64_t seed;
    int32_t  accumulate;
    int32_t  nlights;
    uint32_t pixels_per_task;      /* contiguous rectangle pixels claimed per warp task */
    uint32_t eval_words;           /* stored weights per BSDF evaluation (scene-wide maximum) */
    uint32_t bounce_words;         /* 2 + nlights*(eval_words+1) + eval_words */
    uint32_t head_words;           /* words before the first bounce: 4, or roundup4(2 + ceil(max_depth / 2)) for compact records */
    uint32_t path_words;           /* head_words + max_depth*bounce_words */
    uint32_t path_stride;          /* words between the records of consecutive slots: >= path_words, 4 * odd */
    uint32_t geom_bytes, pool_words;
    /* Deep renders: only the first smem_depth bounces of a path live in its shared-memory record (as many as fit with the kernel's
     * full number of warps); bounces from smem_depth on go to the slot's OVERFLOW ROW in global memory: row (warp * 32 + slot) of
     * `deep`, deep_stride words each -- (max_depth - smem_depth) bounces of bounce_words words, and for compact records their 16-bit
     * headers from word deep_hdr_off.  The rows are written and read once per path by the warp that owns them, so they stay in L2.
     * smem_depth = max_depth (and deep = NULL) for renders whose records fit, i.e. every shipped configuration. */
    uint32_t smem_depth, deep_stride, deep_hdr_off;
    float   *deep;
    /* scattered film store (multi-GPU, drt_cuda_render_device_scatter): pixel p belongs to rank p / scatter_slice, and this
     * rank's partial film of it is written -- over NVLink when the owner is a peer -- into the owner's staging film at pixel
     * scatter_rank * scatter_slice + p % scatter_slice, so every owner ends up with all ranks' partial films of its slice in
     * local memory.  scatter_count = 0: plain store to `film`. */
    /* Pixels outside [hit_x0, hit_x1) x [hit_y0, hit_y1) cannot see any surface (pinhole camera: a conservative screen-space
     * bound of the scene's projection, computed at upload); their camera paths all end on the escape material at depth 0
     * (cast_ray :451-452), so they are counted, not traced.  The full image when no bound is known. */
    uint32_t hit_x0, hit_y0, hit_x1, hit_y1;
    uint32_t scatter_count, scatter_rank, scatter_slice;
    /* Band of a scattered render (drt_cuda_render_device_scatter_band): the launch covers, for every owner o, the pixels
     * [o * band_period + band_base, + band_chunk) -- the same part of every owner's slice -- so that the owners can merge and read
     * back band b while band b + 1 renders.  Task t is pixel (t / band_chunk) * band_period + band_base + t % band_chunk (tasks past
     * the end of the image are empty).  band_chunk = 0: the plain row-major walk of the rectangle. */
    uint32_t band_chunk, band_period, band_base;
    uint32_t task_rotate;          /* tasks are walked from this index (mod the task count): with scatter_rank * slice every rank starts in its own
                                    * slice, so at any moment each owner receives from one peer instead of from all of them */
    FilmPtrs scatter[DRT_MAX_PEERS];
    /* Adaptive sampling (drt_cuda_render_*_adaptive, render_kernel_adaptive): a pixel stops at the end of a batch once its count is
     * >= min_samples and the bound on the standard error of its luminance is <= rel_error times the luminance (pixel_converged in
     * drt_render.cuh).  luminance_w: the per-wavelength weights cmf_y * ref_white of the film-to-RGB tables, in device memory.
     * adaptive = 0: every pixel takes all samples [sample_begin, sample_end). */
    const float *luminance_w;
    float    rel_error;
    uint32_t min_samples;
    uint32_t adaptive;
};
