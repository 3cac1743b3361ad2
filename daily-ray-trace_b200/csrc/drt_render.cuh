/*
 * csrc/drt_render.cuh -- the render hot path as one persistent sm_100a kernel (a template; instantiated by the
 * drt_kernels_{fast,classed,general,f64}[_deep].cu translation units, dispatched by drt_kernels.cu).
 *
 * What the reference does per camera path (sample_scene -> cast_ray -> ..., src/daily_ray_trace.c:432-618) is split
 * along the one axis that never feeds back: NOTHING geometric depends on wavelength (refraction uses n(630 nm) only,
 * Q10; reflect-or-transmit draws against R(630 nm), bdsf.c:241-247).  So every warp alternates two phases:
 *
 *   phase 1 "trace"   one THREAD per path.  Camera ray + per-path Philox stream (K1), closest hit over the SoA scene in
 *                     shared memory (K2), light sampling + shadow rays (K3), direction sampling (K4).  All spectral
 *                     quantities are reduced to a handful of scalar WEIGHTS per BSDF evaluation (eval_weights) and
 *                     written as a compact path record to shared memory.
 *   phase 2 "shade"   one HALF WARP per path, wavelengths across its 16 lanes (5 slots per lane for N = 69), two paths per
 *                     warp at a time.  The record is a broadcast read, spectra are conflict-free shared-memory rows,
 *                     throughput / radiance live in registers,
 *                     and the pixel's film (sum, Welford mean and M2, daily_ray_trace.c:732-743) stays on chip for ALL
 *                     samples of the pixel: each film plane is written to HBM exactly once, coalesced (K6).
 *
 * No path state goes to global memory (deep renders excepted, see DEEP); HBM traffic is the film write, so the kernel is bound by
 * FP32 issue, not by the 1.2 KB-per-bounce queue traffic of a global-memory wavefront (SURVEY.md 8d).
 *
 * Template parameters: R = float (default) or double (branch-flip diagnostic) arithmetic of phase 1; NS = wavelength slots per
 * half-warp lane (2, 3, 5, 8); PAIRED = one pixel per task (spp >= 32) or 32/spp pixels; MODE, chosen at scene upload:
 *   1 plastic-only  every surface material is a bp_diffuse / bp_glossy plastic under ONE light that is the scene's only emitter:
 *                   compact 4-word bounce records replayed backwards in units of the light's emission E (replay_compact),
 *                   the film updated once per batch (BatchStats); 72 registers, 2 CTAs x 14 warps per SM
 *   2 classed       the same records for plastics, single-basis specular materials (mirror, fs_conductor, glass R / T) and
 *                   ct_conductor (GeomT::mclass); its hot code exceeds the 32 KB instruction cache, so the warps of a CTA run their
 *                   phases in lockstep behind mbarrier gates (LOCKSTEP); 64 registers, 2 CTAs x 16 warps
 *   0 general       any lobe list, any sampler, any number of lights, emissive escape material: general records, 2 CTAs x 8 warps
 * DEEP = the instantiation for renders whose records do not fit in shared memory at full occupancy: bounces past
 * RenderLaunch::smem_depth overflow to per-slot rows in global memory (L2-resident), so max_cast_depth x lights is unbounded.
 * Work the kernel proves unnecessary on the host's word (drt_capi.cu, exact): shadow rays do not test boundary planes
 * (GeomT::nax_b), pixels outside the scene's screen-space bound are counted instead of traced (RenderLaunch::hit_*).
 * Quirk numbers (Qn) refer to SURVEY.md Appendix A; the CPU restatement of the same lines is oracle/drt_oracle.c.
 */
#pragma once
#include <cuda_runtime.h>
#include <math_constants.h>
#include "drt_device.cuh"
#include "drt_rng.h"

namespace drt {

/* ------------------------------------------------------------------ small vector algebra in the phase-1 type R */

template <typename R> struct V3 { R x, y, z; };

template <typename R> __device__ __forceinline__ V3<R> mk(R x, R y, R z) { V3<R> v; v.x = x; v.y = y; v.z = z; return v; }
template <typename R> __device__ __forceinline__ V3<R> operator+(V3<R> a, V3<R> b) { return mk<R>(a.x + b.x, a.y + b.y, a.z + b.z); }
template <typename R> __device__ __forceinline__ V3<R> operator-(V3<R> a, V3<R> b) { return mk<R>(a.x - b.x, a.y - b.y, a.z - b.z); }
template <typename R> __device__ __forceinline__ V3<R> operator*(V3<R> a, R f) { return mk<R>(f * a.x, f * a.y, f * a.z); }
template <typename R> __device__ __forceinline__ V3<R> neg(V3<R> a) { return mk<R>(-a.x, -a.y, -a.z); }
template <typename R> __device__ __forceinline__ R dot(V3<R> a, V3<R> b) { return a.x * b.x + a.y * b.y + a.z * b.z; }
template <typename R> __device__ __forceinline__ V3<R> cross(V3<R> a, V3<R> b)
{
    return mk<R>(a.y * b.z - a.z * b.y, a.z * b.x - a.x * b.z, a.x * b.y - a.y * b.x);
}

/* MUFU.RCP alone (<= 1 ulp), for arguments known to be in range */
__device__ __forceinline__ float r_rcp_fast(float x) { float r; asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x)); return r; }
__device__ __forceinline__ float  r_sqrt(float x)  { float r; asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x)); return r; }   /* MUFU.SQRT alone */
__device__ __forceinline__ double r_sqrt(double x) { return sqrt(x); }
__device__ __forceinline__ float  r_abs(float x)   { return fabsf(x); }
__device__ __forceinline__ double r_abs(double x)  { return fabs(x); }
/* The transcendental library routines are large; one out-of-line copy each keeps the kernel inside the instruction cache. */
/* f32: x^y = 2^(y log2 x) on the SFU (MUFU.LG2 / MUFU.EX2); relative error ~ |y| * 1.7e-7, i.e. 5e-6 at shininess 32 and 2e-5
 * at 100, against the 1e-3 parity tolerance.  The accurate powf costs ~7.5 warp-instructions per path (5 % of the kernel). */
__device__ __forceinline__ float  r_pow(float x, float y)   { return (x <= 0.f) ? ((y == 0.f) ? 1.f : 0.f) : exp2f(y * __log2f(x)); }
static __device__ __noinline__ double r_pow(double x, double y) { return pow(x, y); }
/* sin and cos of pi*t: the reference's angles are all multiples of pi (2*pi*v, pi/4*ratio, rng.c:18,40-46) */
static __device__ __noinline__ void r_sincospi(float t, float *s, float *c)    { sincospif(t, s, c); }
static __device__ __noinline__ void r_sincospi(double t, double *s, double *c) { sincos(3.14159265358979323846 * t, s, c); }

template <typename R> struct Num;
template <> struct Num<float>
{
    static __device__ __forceinline__ float pi()  { return 3.14159265358979323846f; }
    static __device__ __forceinline__ float inf() { return CUDART_INF_F; }
    static __device__ __forceinline__ float fudge() { return 0.0001f; }
    /* rng() of rng.c:2-7: r31 / RAND_MAX, rounded once to f32 */
    static __device__ __forceinline__ float unit(uint32_t r31) { return __uint2float_rn(r31) * 4.6566128752457969e-10f; }
};
template <> struct Num<double>
{
    static __device__ __forceinline__ double pi()  { return 3.14159265358979323846; }
    static __device__ __forceinline__ double inf() { return CUDART_INF; }
    static __device__ __forceinline__ double fudge() { return 0.0001; }
    static __device__ __forceinline__ double unit(uint32_t r31) { return (double)r31 / 2147483647.0; }
};

/* a / b and 1 / sqrt(x) for operands known to be in range: f32 uses the bare MUFU.RCP / MUFU.RSQ (<= 1-2 ulp) instead of the
 * range-scaled sequences the compiler emits for '/' and sqrtf even under -prec-div=false (8-13 instructions per site) */
__device__ __forceinline__ float  r_div(float a, float b)   { return a * r_rcp_fast(b); }
__device__ __forceinline__ double r_div(double a, double b) { return a / b; }
__device__ __forceinline__ float  r_sqrt_fast(float x)  { float r; asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x)); return r; }   /* MUFU.SQRT */
__device__ __forceinline__ double r_sqrt_fast(double x) { return sqrt(x); }
__device__ __forceinline__ float  r_rsqrt(float x)  { float r; asm("rsqrt.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x)); return r; }
__device__ __forceinline__ double r_rsqrt(double x) { return 1.0 / sqrt(x); }

template <typename R> __device__ __forceinline__ V3<R> normalise(V3<R> v);
template <> __device__ __forceinline__ V3<double> normalise<double>(V3<double> v)   /* geometry.c: v / |v| */
{
    double len = sqrt(dot(v, v));
    return mk<double>(v.x / len, v.y / len, v.z / len);
}
template <> __device__ __forceinline__ V3<float> normalise<float>(V3<float> v)
{
    float inv = r_rsqrt(dot(v, v));
    return mk<float>(v.x * inv, v.y * inv, v.z * inv);
}
template <typename R> __device__ __forceinline__ V3<R> reflect(V3<R> v, V3<R> n)   /* geometry.c:85-90 */
{
    R f = R(2) * dot(v, n);
    return v - n * f;
}
template <typename R> __device__ __forceinline__ V3<R> transmit(V3<R> v, V3<R> n, R ir, R tr)   /* geometry.c:92-106 */
{
    R vn = dot(v, n);
    R rel = r_div(ir, tr);
    V3<R> m = n * vn;
    v = m - v;
    V3<R> perpend = neg(v * rel);
    R pd = -r_sqrt(R(1) - dot(perpend, perpend));
    return perpend + n * pd;
}

/* find_rotation_between_vectors((0,0,1), n) applied to q (geometry.c:263-295), in closed form:
 * R q = q + a x q + a x (a x q) / (1 + c) with a = (0,0,1) x n, c = n.z; antiparallel -> -q (Q14). */
template <typename R> __device__ __forceinline__ V3<R> rotate_from_z(V3<R> n, V3<R> q)
{
    V3<R> a = mk<R>(-n.y, n.x, R(0));
    R c = n.z;
    if(dot(a, a) == R(0) && c <= R(0)) return neg(q);
    V3<R> aq = cross(a, q);
    V3<R> aaq = cross(a, aq);
    R f = r_div(R(1), R(1) + c);
    return (q + aq) + aaq * f;
}

/* ------------------------------------------------------------------ per-path random stream (include/drt_rng.h) */

static __device__ __noinline__ uint4 philox_block(uint32_t block, uint32_t seed_lo, uint32_t seed_hi, uint32_t key0, uint32_t key1)
{
    uint32_t out[4];
    drt_philox4x32_10(block, 0u, seed_lo, seed_hi, key0, key1, out);
    return make_uint4(out[0], out[1], out[2], out[3]);
}

struct Rng
{
    uint32_t key0, key1, seed_lo, seed_hi, draws;
    uint4 buf;
    __device__ __forceinline__ void begin(uint64_t seed, uint32_t pixel, uint32_t sample)
    {
        key0 = pixel; key1 = sample; seed_lo = (uint32_t)seed; seed_hi = (uint32_t)(seed >> 32); draws = 0;
        buf = make_uint4(0u, 0u, 0u, 0u);
    }
    __device__ __forceinline__ uint32_t next31()
    {
        uint32_t lane = draws & 3u;
        if(lane == 0) buf = philox_block(draws >> 2, seed_lo, seed_hi, key0, key1);
        draws += 1;
        uint32_t w = (lane == 0) ? buf.x : (lane == 1) ? buf.y : (lane == 2) ? buf.z : buf.w;
        return w >> 1;
    }
    template <typename R> __device__ __forceinline__ R unit() { return Num<R>::unit(next31()); }
};

/* ------------------------------------------------------------------ K2: closest hit / any hit over the SoA scene */

/* line_sphere_intersection, geometry.c:123-146: smallest non-negative root of t^2 - b t + c = 0, else +inf. */
__device__ __forceinline__ double hit_sphere(V3<double> o, V3<double> d, V3<double> c, double r)
{
    V3<double> co = o - c;
    double b = -2.0 * dot(co, d);
    double cc = dot(co, co) - r * r;
    double disc = b * b - 4.0 * cc;
    if(disc < 0.0) return Num<double>::inf();
    double sq = sqrt(disc);
    double s0 = (b + sq) / 2.0;
    double s1 = (b - sq) / 2.0;
    if(s0 < 0.0 && s1 < 0.0) return Num<double>::inf();
    if(s0 >= 0.0 && s1 < 0.0) return s0;
    if(s1 >= 0.0 && s0 < 0.0) return s1;
    return (s0 <= s1) ? s0 : s1;
}
/* The same roots in f32.  b^2 - 4c loses |o-c|^2 * eps, which near a silhouette (and for the reference's shadow test
 * against the light's own sphere, margin 1e-4) decides hit or miss; the quarter discriminant r^2 - |co - (co.d) d|^2
 * is the same quantity with error ~ r^2 * eps (Haines et al., Ray Tracing Gems ch. 7). */
__device__ __forceinline__ float hit_sphere(V3<float> o, V3<float> d, V3<float> c, float r)
{
    V3<float> co = o - c;
    float half_b = -dot(co, d);                 /* = b / 2 */
    V3<float> perp = co + d * half_b;           /* component of co perpendicular to the ray */
    float qdisc = r * r - dot(perp, perp);      /* = disc / 4 */
    if(qdisc < 0.f) return Num<float>::inf();
    float sq = sqrtf(qdisc);
    float s0 = half_b + sq;
    float s1 = half_b - sq;
    if(s0 < 0.f && s1 < 0.f) return Num<float>::inf();
    if(s0 >= 0.f && s1 < 0.f) return s0;
    if(s1 >= 0.f && s0 < 0.f) return s1;
    return (s0 <= s1) ? s0 : s1;
}

/* line_plane_intersection, geometry.c:157-182, on the packed surface (n, p, u^ | |u|, v^ | |v|).  The bounds frame that the
 * reference recomputes on every call (:166-170) is precomputed by the host; bounds are inclusive (Q21). */
__device__ __forceinline__ double hit_plane(V3<double> o, V3<double> d, R4<double> n4, R4<double> p4, R4<double> u4, R4<double> v4)
{
    V3<double> n = mk<double>(n4.x, n4.y, n4.z), p = mk<double>(p4.x, p4.y, p4.z);
    double dn = dot(d, n);
    if(dn == 0.0) return Num<double>::inf();
    double l = dot(p - o, n) / dn;
    V3<double> j = (o + d * l) - p;
    double ju = dot(j, mk<double>(u4.x, u4.y, u4.z));
    double jv = dot(j, mk<double>(v4.x, v4.y, v4.z));
    bool inside = l >= 0.0 && 0.0 <= ju && ju <= u4.w && 0.0 <= jv && jv <= v4.w;
    return inside ? l : Num<double>::inf();
}
/* f32: the same test fused with the nearest-so-far update.  The in-plane offset is formed as d*l - (p - o), which reuses p - o;
 * l = ((p - o).n) / (d.n) uses MUFU.RCP without the range scaling of a full divide (|d.n| <= 1); the five inclusive bounds
 * l >= 0, 0 <= j.u^ <= |u|, 0 <= j.v^ <= |v| (Q21) collapse into one minimum that must be >= 0 (FMNMX3).  A ray parallel to
 * the plane (d.n == 0, geometry.c:160) gives l = +-inf or NaN: -inf fails the minimum, +inf and NaN fail l < best. */
__device__ __forceinline__ bool hit_plane_nearer(V3<float> o, V3<float> d, R4<float> n4, R4<float> p4, R4<float> u4, R4<float> v4, float best, float &l)
{
    V3<float> n = mk<float>(n4.x, n4.y, n4.z);
    float dn = dot(d, n);
    V3<float> po = mk<float>(p4.x - o.x, p4.y - o.y, p4.z - o.z);
    l = dot(po, n) * r_rcp_fast(dn);
    V3<float> j = mk<float>(fmaf(d.x, l, -po.x), fmaf(d.y, l, -po.y), fmaf(d.z, l, -po.z));
    float ju = dot(j, mk<float>(u4.x, u4.y, u4.z));
    float jv = dot(j, mk<float>(v4.x, v4.y, v4.z));
    float m = fminf(fminf(ju, u4.w - ju), fminf(fminf(jv, v4.w - jv), l));
    return m >= 0.f && l < best;
}
__device__ __forceinline__ bool hit_plane_nearer(V3<double> o, V3<double> d, R4<double> n4, R4<double> p4, R4<double> u4, R4<double> v4, double best, double &l)
{
    l = hit_plane(o, d, n4, p4, u4, v4);
    return l < best;
}

/* Nearest surface strictly closer than `limit` along the ray: its SLOT in the regrouped arrays, or -1 (the loops of
 * find_ray_intersection daily_ray_trace.c:340-364 and points_mutually_visible :246-268; points are skipped, strict < keeps
 * the lowest scene index on ties).  One shared out-of-line body serves closest-hit (limit = inf) and shadow rays
 * (limit = vis_dist).
 * `skip` = slot of the PLANE the ray starts on, or -1.  The reference tests that plane too and always misses it: the origin
 * is pushed 1e-4 along the ray first (Q2), so the plane lies at l = -1e-4 < 0 whatever the direction.  Its f64 rounding
 * cannot change that sign; f32 rounding at grazing angles could, so not testing the plane is both cheaper and closer to the
 * reference. */
__device__ __forceinline__ float  r_rcp(float x)  { return r_rcp_fast(x); }
__device__ __forceinline__ double r_rcp(double x) { return 1.0 / x; }
__device__ __forceinline__ float  r_min3(float a, float b, float c)    { return fminf(fminf(a, b), c); }   /* FMNMX3 */
__device__ __forceinline__ double r_min3(double a, double b, double c) { return fmin(fmin(a, b), c); }

/* One group of axis-aligned rectangles (normal along axis a; in-plane axes b < c): l = (p_a - o_a) / d_a and the hit point's
 * two in-plane coordinates against the rectangle's centre and half extents -- line_plane_intersection (geometry.c:157-182)
 * with the zero terms of its dot products dropped.  o?, d? are the ray's components along a, b, c; inv_da = 1 / d_a.
 * A ray parallel to the plane gives l = +-inf or NaN, which fail l >= 0 or l < best as in hit_plane_nearer. */
template <typename R>
__device__ __forceinline__ void nearest_axis_group(const GeomT<R> &g, int k0, int k1, R oa, R ob, R oc, R inv_da, R db, R dc, int skip,
                                                   R &best, R &best_sid, int &found)
{
#pragma unroll 1
    for(int k = k0; k < k1; k += 1)
    {
        const R4<R> q = g.AX4[k];
        const R2<R> h = g.AXH[k];
        const R l = (q.x - oa) * inv_da;
        const R eb = q.z - r_abs((ob + db * l) - q.y);
        const R ec = h.x - r_abs((oc + dc * l) - q.w);
        const R m = r_min3(eb, ec, l);
        /* nearer, or as near as the best so far but earlier in the scene (best_sid is -1 until something is found) */
        const bool take = (m >= R(0)) & ((l < best) | ((l == best) & (h.y < best_sid))) & (k != skip);   /* & and |: no branches */
        best = take ? l : best; best_sid = take ? h.y : best_sid; found = take ? k : found;
    }
}

template <typename R> __device__ __noinline__ int nearest_surface(const GeomT<R> &g, V3<R> o, V3<R> d, R limit, int skip, bool shadow, R *dist_out)
{
    R best = limit, best_sid = R(-1);
    int found = -1;
    /* rectangles by axis, planes in general position, spheres: no type switch inside the loops.  Slots of one group are in
     * scene order, so inside a group a strict < reproduces the reference's single in-order loop; a candidate that ties with
     * the current best (coplanar surfaces, a ray through a shared edge) replaces it only if its scene index is lower. */
    const int nx = g.nax[0], ny = nx + g.nax[1], nz = ny + g.nax[2];
    const int np = g.nplanes, ns = g.nspheres;
    /* shadow rays start every plane group after its boundary planes (GeomT::nax_b) */
    const int bx = shadow ? g.nax_b[0] : 0, by = shadow ? g.nax_b[1] : 0, bz = shadow ? g.nax_b[2] : 0, bg = shadow ? g.nax_b[3] : 0;
    nearest_axis_group<R>(g, bx, nx, o.x, o.y, o.z, r_rcp(d.x), d.y, d.z, skip, best, best_sid, found);
    nearest_axis_group<R>(g, nx + by, ny, o.y, o.x, o.z, r_rcp(d.y), d.x, d.z, skip, best, best_sid, found);
    nearest_axis_group<R>(g, ny + bz, nz, o.z, o.x, o.y, r_rcp(d.z), d.x, d.y, skip, best, best_sid, found);
#pragma unroll 1
    for(int k = nz + bg; k < np; k += 1)
    {
        if(k == skip) continue;
        R dist;
        const R sid = R(g.sid[k]);
        bool nearer = hit_plane_nearer(o, d, g.N4[k], g.P4[k], g.U4[k], g.V4[k], best, dist);
        if(!nearer && dist == best && sid < best_sid) nearer = hit_plane_nearer(o, d, g.N4[k], g.P4[k], g.U4[k], g.V4[k], limit, dist);
        if(nearer) { best = dist; best_sid = sid; found = k; }
    }
#pragma unroll 1
    for(int k = np; k < np + ns; k += 1)
    {
        R4<R> p4 = g.P4[k];
        R dist = hit_sphere(o, d, mk<R>(p4.x, p4.y, p4.z), p4.w);
        const R sid = R(g.sid[k]);
        if(dist < best || (dist == best && sid < best_sid)) { best = dist; best_sid = sid; found = k; }
    }
    *dist_out = best;
    return found;
}

template <typename R> struct Hit
{
    V3<R> pos, nrm, out;
    R on_dot;
    int surf_mat, inc_mat, trans_mat;
    int plane_slot;   /* slot of the plane that was hit (nearest_surface's `skip` for the rays leaving this point), -1 for a sphere */
};

/* find_ray_intersection, daily_ray_trace.c:334-403.  Returns false on a miss (escape material). */
template <typename R> __device__ __forceinline__ bool closest_hit(const GeomT<R> &g, V3<R> o, V3<R> d, int skip, Hit<R> &h)
{
    o = o + d * Num<R>::fudge();   /* Q2 */
    R best;
    int slot = nearest_surface<R>(g, o, d, Num<R>::inf(), skip, false, &best);
    if(slot < 0) return false;
    const int found = g.sid[slot];
    h.plane_slot = (slot < g.nplanes) ? slot : -1;
    h.pos = o + d * best;
    V3<R> n = mk<R>(g.nx[found], g.ny[found], g.nz[found]);
    bool is_plane = g.type[found] == DRT_GEO_PLANE;
    if(!is_plane) n = normalise(h.pos - mk<R>(g.px[found], g.py[found], g.pz[found]));
    h.out = neg(d);
    h.on_dot = dot(n, h.out);
    int sm = g.mat[found];
    h.surf_mat = sm; h.trans_mat = sm; h.inc_mat = g.base_mat;
    if(h.on_dot < R(0))
    {
        if(!is_plane) { h.trans_mat = g.base_mat; h.inc_mat = sm; }   /* Q11 */
        n = neg(n);
        h.on_dot = dot(n, h.out);
    }
    h.nrm = n;
    return true;
}

/* points_mutually_visible, daily_ray_trace.c:238-270 */
template <typename R> __device__ __forceinline__ bool visible(const GeomT<R> &g, V3<R> p0, V3<R> p1, int skip, V3<R> &dir)
{
    dir = normalise(p1 - p0);   /* also the direction to the light of direct_light_contribution :318 */
    V3<R> o = p0 + dir * Num<R>::fudge();
    V3<R> po = p1 - o;
    R vis_dist = r_sqrt(dot(po, po)) - Num<R>::fudge();
    R t;
    /* nothing but boundary planes in the scene (an empty room): no surface can lie between two of its points */
    if(g.nax_b[0] + g.nax_b[1] + g.nax_b[2] + g.nax_b[3] == g.nplanes && g.nspheres == 0) return true;
    return nearest_surface<R>(g, o, dir, vis_dist, skip, true, &t) < 0;
}

/* ------------------------------------------------------------------ BSDF evaluation reduced to basis weights
 *
 * bdsf() (daily_ray_trace.c:215-229) sums the material's lobes through ONE scratch spectrum that is zeroed once;
 * lobes that "do not write" leave the previous lobe's value in it (Q7).  Every lobe output is a scalar times one of
 * seven spectra: 1, diffuse, glossy, mirror, R_dielectric(on_dot), F_conductor(on_dot), F_conductor(mn_dot).  Walking
 * the lobe list with a 7-vector as the scratch reproduces the sum, stale values included, as 7 weights.  The weights
 * the material can produce (g.bmask) are stored to the path record `rec` (already offset to the slot) from word `at`. */
#define BMASK_PLASTIC ((1 << BK_DIFFUSE) | (1 << BK_GLOSSY))

template <typename R>
static __device__ __noinline__ void eval_weights_general(const GeomT<R> &g, int m, V3<R> nrm, V3<R> out, R on_dot, V3<R> in, int match, float scale,
                                                  float *rec, uint32_t at)
{
    const bool is_reflection = match & 1, is_transmission = match & 2;
    float cur[BK_COUNT], acc[BK_COUNT];
#pragma unroll
    for(int k = 0; k < BK_COUNT; k += 1) { cur[k] = 0.f; acc[k] = 0.f; }
    float mn_cos = 0.f;
    int nl = g.nlobes[m];
    for(int li = 0; li < nl; li += 1)
    {
        int lobe = g.lobes[m][li];
        bool wrote = true;
        int kind = BK_CONST;
        float val = 0.f, val_const = 0.f;
        switch(lobe)
        {
            case DRT_LOBE_BP_DIFFUSE:   /* bdsf.c:105-109 */
                kind = BK_DIFFUSE; val = (float)((R(1) / Num<R>::pi()) * r_abs(dot(nrm, in)));
                break;
            case DRT_LOBE_BP_GLOSSY:   /* bdsf.c:111-119 */
            {
                V3<R> bis = normalise(out + in);
                R nb = dot(nrm, bis);
                R coef = r_pow((R(0) > nb) ? R(0) : nb, g.shin[m]);
                kind = BK_GLOSSY; val = (float)(coef * r_abs(dot(nrm, in)));
                break;
            }
            case DRT_LOBE_MIRROR:   /* bdsf.c:121-132: zero on mismatch */
                kind = BK_MIRROR; val = is_reflection ? 1.f : 0.f;
                break;
            case DRT_LOBE_FS_CONDUCTOR:   /* bdsf.c:134-146: no write on mismatch (Q8: exact match == "came from the reflect formula") */
                kind = BK_COND_ON; val = 1.f; wrote = is_reflection;
                break;
            case DRT_LOBE_FS_DIELECTRIC_REFLECTANCE:   /* bdsf.c:148-159 */
                kind = BK_DIEL_R; val = 1.f; wrote = is_reflection;
                break;
            case DRT_LOBE_FS_DIELECTRIC_TRANSMITTANCE:   /* bdsf.c:161-172: 1 - R */
                kind = BK_DIEL_R; val = -1.f; val_const = 1.f; wrote = is_transmission;
                break;
            case DRT_LOBE_CT_CONDUCTOR:   /* bdsf.c:174-186 */
            {
                V3<R> mn = normalise(out + in);
                R mn_dot = r_abs(dot(nrm, mn));
                /* ggx_att(out, n, mn, rough) * 1/(4 on_dot), bdsf.c:3-42 */
                R rough = g.rough[m], r2 = rough * rough;
                R d = dot(nrm, mn), gg = R(0);
                if(d > R(0))
                {
                    R d2 = d * d, d4 = d2 * d2, tan_sq = r_div(R(1), d2) - R(1);
                    gg = r_div(r2, Num<R>::pi() * d4 * (r2 + tan_sq) * (r2 + tan_sq));
                }
                R v_mn = dot(out, mn), v_sn = dot(out, nrm);
                R quot = r_abs(r_div(v_mn, v_sn)), att = R(0);
                if(!(quot <= R(0)))
                {
                    R tan_sq = r_div(R(1), v_sn * v_sn) - R(1);
                    att = r_div(R(2), R(1) + r_sqrt(R(1) + r2 * tan_sq));
                }
                kind = BK_COND_MN; val = (float)((gg * att) * r_div(R(1), R(4) * on_dot));
                mn_cos = (float)mn_dot;
                break;
            }
            default: wrote = false; break;
        }
        if(wrote)
        {
#pragma unroll
            for(int k = 0; k < BK_COUNT; k += 1) cur[k] = (k == kind) ? val : 0.f;
            cur[BK_CONST] += val_const;
        }
#pragma unroll
        for(int k = 0; k < BK_COUNT; k += 1) acc[k] += cur[k];
    }
    const int mask = g.bmask[m];
#pragma unroll
    for(int k = 0; k < BK_COUNT; k += 1)
        if(mask & (1 << k)) { rec[at] = acc[k] * scale; at += 1; }
    if(mask & (1 << BK_COND_MN)) rec[at] = mn_cos;
}

/* Hot case inline: the two-lobe Blinn-Phong plastic (bp_diffuse_bdsf, bp_glossy_bdsf, bdsf.c:105-119) of every shipped wall
 * and ball needs two weights and no lobe walk; every other lobe list goes through the out-of-line general evaluator. */
template <typename R>
__device__ __forceinline__ void plastic_weights(const GeomT<R> &g, int m, V3<R> nrm, V3<R> out, V3<R> in, float scale, float &wd, float &wg)
{
    R cos_in = r_abs(dot(nrm, in));
    V3<R> bis = normalise(out + in);
    R nb = dot(nrm, bis);
    R coef = r_pow((R(0) > nb) ? R(0) : nb, g.shin[m]);
    wd = (float)((R(1) / Num<R>::pi()) * cos_in) * scale;
    wg = (float)(coef * cos_in) * scale;
}
/* ct_conductor_bdsf without its Fresnel factor (bdsf.c:174-186): ggx_att(out, n, m, rough) / (4 on_dot) with m = normalise(out + in),
 * D of bdsf.c:3-20 and G1(out) of :22-42, and the micro-normal cosine |n.m| the Fresnel factor is evaluated at.  One out-of-line copy
 * serves the next-event and the sampled-direction evaluation of the classed kernel. */
template <typename R>
static __device__ __noinline__ float2 ct_weight(const GeomT<R> &g, int m, V3<R> nrm, V3<R> out, R on_dot, V3<R> in)
{
    V3<R> mn = normalise(out + in);
    R d = dot(nrm, mn), gg = R(0);
    R rough = g.rough[m], r2 = rough * rough;
    if(d > R(0))
    {
        R d2 = d * d, d4 = d2 * d2, tan_sq = r_div(R(1), d2) - R(1);
        gg = r_div(r2, Num<R>::pi() * d4 * (r2 + tan_sq) * (r2 + tan_sq));
    }
    R v_mn = dot(out, mn), v_sn = dot(out, nrm);
    R quot = r_abs(r_div(v_mn, v_sn)), att = R(0);
    if(!(quot <= R(0)))
    {
        R tan_sq = r_div(R(1), v_sn * v_sn) - R(1);
        att = r_div(R(2), R(1) + r_sqrt(R(1) + r2 * tan_sq));
    }
    return make_float2((float)((gg * att) * r_div(R(1), R(4) * on_dot)) * g.ct_mult[m], (float)r_abs(d));
}

/* dielectric Fresnel at one wavelength, bdsf.c:44-66 (Q9 kept) */
template <typename T> __device__ __forceinline__ T fresnel_dielectric(T ir, T tr, T inc_cos)
{
    T inc_sin_sq = T(1) - inc_cos * inc_cos;
    T rel = r_div(ir, tr);
    T ts_sin_sq = rel * rel * inc_sin_sq;
    if(ts_sin_sq >= T(1)) return T(1);
    T ts_cos = r_sqrt_fast(T(1) - ts_sin_sq * ts_sin_sq);
    T tr_on = tr * inc_cos, tr_ts = tr * ts_cos, ir_on = ir * inc_cos, ir_ts = ir * ts_cos;
    T par = r_div(tr_on - ir_ts, tr_on + ir_ts);
    T per = r_div(ir_on - tr_ts, ir_on + tr_ts);
    return T(0.5) * (par * par + per * per);
}

/* ------------------------------------------------------------------ K4: the six direction samplers, bdsf.c:191-292 */

/* sin(pi u) and cos(pi u) for |u| <= 1/4, inline and without range reduction: minimax polynomials in v = u^2 whose float32
 * coefficients come from tools/fit_sincospi_quarter.py (numpy, float64 fit).  Under 1 ulp from float64 sin / cos on a dense grid and
 * on the float32 values next to 0 and +-1/4 (tests/test_trace_trim.py models this evaluation order). */
__device__ __forceinline__ void sincospi_quarter(float u, float &s, float &c)
{
    const float v = u * u;
    const float ps = fmaf(fmaf(-0x1.330cc6p-1f, v, 0x1.46805cp+1f), v, -0x1.4abc24p+2f);
    s = fmaf(u, 0x1.921fb6p+1f, (u * v) * ps);
    const float pc = fmaf(fmaf(fmaf(0x1.d9f7bcp-3f, v, -0x1.55c664p+0f), v, 0x1.03c1dep+2f), v, -0x1.3bd3ccp+2f);
    c = fmaf(v, pc, 1.f);
}

/* sin and cos of the concentric map's angle: pi/4 q, or pi/2 - pi/4 q for the `steep` octants (q = the smaller coordinate over the
 * larger, in [-1, 1]).  f32: sin(pi/2 - x) = cos(x), so both come from sincospi_quarter(q / 4) with s and c swapped; f64 (the branch-
 * flip diagnostic) keeps the library's sincos. */
__device__ __forceinline__ void disc_sincos(float q, bool steep, float &s, float &c)
{
    float a, b;
    sincospi_quarter(0.25f * q, a, b);
    s = steep ? b : a; c = steep ? a : b;
}
__device__ __forceinline__ void disc_sincos(double q, bool steep, double &s, double &c) { r_sincospi(steep ? 0.5 - 0.25 * q : 0.25 * q, &s, &c); }

template <typename R> __device__ __forceinline__ V3<R> sample_disc(Rng &rng)   /* uniform_sample_disc, rng.c:25-51 */
{
    R rx = rng.unit<R>();
    R ry = rng.unit<R>();
    R ox = R(2) * rx - R(1), oy = R(2) * ry - R(1);
    if(ox == R(0) && oy == R(0)) return mk<R>(R(0), R(0), R(0));
    R r, q;
    const bool steep = !(r_abs(ox) > r_abs(oy));
    if(!steep) { r = ox; q = r_div(oy, ox); }
    else       { r = oy; q = r_div(ox, oy); }
    R s, c;
    disc_sincos(q, steep, s, c);
    return mk<R>(r * c, r * s, R(0));
}

/* match: bit0 = `in` came out of the reflection formula, bit1 = out of the refraction formula (Q8) */
template <typename R> struct DirSample { V3<R> in; R inv_pdf; int match; Rng rng; };

/* Five of the six samplers, out of line and by value (the cosine-weighted one is inlined in sample_direction below). */
template <typename R>
static __device__ __noinline__ DirSample<R> sample_direction_general(const GeomT<R> &g, Hit<R> h, Rng rng)
{
    DirSample<R> out;
    V3<R> in = mk<R>(R(0), R(0), R(0));
    R inv_pdf = R(0);
    int match = 0;
    int m = h.surf_mat;
    switch(g.dirf[m])
    {
        case DRT_DIR_UNIFORM_HEMISPHERE:   /* :191-198; uniform_sample_sphere rng.c:14-23 has z = u >= 0 */
        {
            R u = rng.unit<R>();
            R v = rng.unit<R>();
            R r = r_sqrt(R(1) - u * u);
            R s, c;
            r_sincospi(R(2) * v, &s, &c);
            in = rotate_from_z<R>(h.nrm, mk<R>(r * c, r * s, u));
            inv_pdf = R(2) * Num<R>::pi();
            break;
        }
        /* DRT_DIR_COS_WEIGHTED_HEMISPHERE (:200-213) is handled inline by sample_direction below and never reaches this function */
        case DRT_DIR_SPECULAR:   /* :215-220 */
            in = reflect<R>(neg(h.out), h.nrm);
            inv_pdf = R(1);
            match = 1;
            break;
        case DRT_DIR_TRANSMIT:   /* :222-234 */
            in = transmit<R>(neg(h.out), h.nrm, g.n630[h.inc_mat], g.n630[h.trans_mat]);
            inv_pdf = R(1);
            match = ((in.x == in.x) && (in.y == in.y) && (in.z == in.z)) ? 2 : 0;
            break;
        case DRT_DIR_REFLECT_OR_TRANSMIT:   /* :236-259: reflect with probability R(630 nm) */
        {
            R ra = fresnel_dielectric<R>(g.refr_a[h.inc_mat], g.refr_a[h.trans_mat], h.on_dot);
            R rb = fresnel_dielectric<R>(g.refr_b[h.inc_mat], g.refr_b[h.trans_mat], h.on_dot);
            R rd = ra + (g.trans_num * r_div(rb - ra, g.trans_den));
            R f = rng.unit<R>();
            if(f < rd)
            {
                in = reflect<R>(neg(h.out), h.nrm);
                inv_pdf = r_div(R(1), rd);
                match = 1;
            }
            else
            {
                in = transmit<R>(neg(h.out), h.nrm, g.n630[h.inc_mat], g.n630[h.trans_mat]);
                inv_pdf = r_div(R(1), R(1) - rd);
                match = ((in.x == in.x) && (in.y == in.y) && (in.z == in.z)) ? 2 : 0;
            }
            break;
        }
        case DRT_DIR_CT:   /* :261-292 */
        {
            R rough = g.rough[m];
            do
            {
                R f = rng.unit<R>();
                R gq = rng.unit<R>();
                R tan_mn = r_div(rough * r_sqrt(f), r_sqrt(R(1) - f));
                R cos_mn = r_rsqrt(R(1) + tan_mn * tan_mn);
                R cm2 = cos_mn * cos_mn;
                R sin_mn = r_sqrt((cm2 < R(1)) ? R(1) - cm2 : R(0));   /* 1/sqrt(1+t^2) may round to 1+ulp with approximate division */
                R s, c;
                r_sincospi(R(2) * gq, &s, &c);
                V3<R> mn = rotate_from_z<R>(h.nrm, mk<R>(sin_mn * c, sin_mn * s, cos_mn));
                R sn_mn = dot(h.nrm, mn);
                if(sn_mn < R(0)) { mn = neg(mn); sn_mn = -sn_mn; }
                R o_mn = dot(h.out, mn);
                in = reflect<R>(neg(h.out), mn);
                R d = R(0);   /* ggx(n, mn, rough) * sn_mn */
                if(sn_mn > R(0))
                {
                    R r2 = rough * rough, d2 = sn_mn * sn_mn, d4 = d2 * d2, tan_sq = r_div(R(1), d2) - R(1);
                    d = r_div(r2, Num<R>::pi() * d4 * (r2 + tan_sq) * (r2 + tan_sq));
                }
                d = d * sn_mn;
                inv_pdf = r_div(R(4) * o_mn, d);
            }
            while(dot(in, h.nrm) < R(0));
            break;
        }
        default: break;
    }
    out.in = in; out.inv_pdf = inv_pdf; out.match = match; out.rng = rng;
    return out;
}

template <typename R>
__device__ __forceinline__ void sample_direction(const GeomT<R> &g, const Hit<R> &h, Rng &rng, V3<R> &in, R &inv_pdf, int &match)
{
    if(g.dirf[h.surf_mat] == DRT_DIR_COS_WEIGHTED_HEMISPHERE)   /* hot case inline, bdsf.c:200-213 */
    {
        V3<R> q;
        for(;;)
        {
            q = sample_disc<R>(rng);
            if(dot(q, q) < R(1)) break;   /* Q16 */
        }
        q.z = r_sqrt(R(1) - dot(q, q));
        in = rotate_from_z<R>(h.nrm, q);
        inv_pdf = r_div(Num<R>::pi(), dot(h.nrm, in));
        match = 0;
        return;
    }
    DirSample<R> s = sample_direction_general<R>(g, h, rng);
    in = s.in; inv_pdf = s.inv_pdf; match = s.match; rng = s.rng;
}

/* ------------------------------------------------------------------ path records in shared memory */

#define REC_NB   0
#define REC_VIG  1
#define REC_HDR16 2   /* ALLFAST records: 16-bit bounce headers from word 2 */
#define REC_HEAD 4    /* general records: first bounce */
#define KIND_SHADE 1u
#define KIND_EMIT  2u
/* bounce header word (record layout: RenderLaunch in drt_device.cuh):
 *   fast (two-lobe plastic, one light):  kind(2) | 1<<2 | D, G block word offset (SpdIndex::plastic2)<<2
 *   general:                             kind(2) | 0<<2 | surface material(5)<<3 | media swapped<<8 | light visibility mask(16)<<16
 * so the hot replay needs two 16-byte record reads per bounce and no material-table lookups. */
#define HDR_FAST 4u

/* ------------------------------------------------------------------ phase 1: trace one path, emit its record
 * `rec` points at this lane's record (16-byte aligned).  Returns the termination-histogram bin and a class bit. */

template <typename R, int MODE, bool DEEP>
__device__ __forceinline__ uint32_t trace_path(const GeomT<R> &g, const SpdIndex &ix, const RenderLaunch &L, float *rec, float *deep,
                                               uint32_t x, uint32_t y, uint32_t sample, uint32_t (&tally)[4])
{
    constexpr bool ALLFAST = MODE != 0;    /* compact records: the plastic-only kernel (1) and the classed kernel (2) */
    constexpr bool CLASSED = MODE == 2;
    Rng rng;
    rng.begin(L.seed, y * L.width + x, sample);

    /* K1: sample_pixel_point + sample_scene, daily_ray_trace.c:550-607 */
    R px = R(0), py = R(0);
    if(L.pixel_scheme == DRT_PIXEL_CENTER) { px = R(0.5); py = R(0.5); }
    else if(L.pixel_scheme == DRT_PIXEL_RANDOM) { px = rng.unit<R>(); py = rng.unit<R>(); }
    R film_x = (R(x) + px) * g.pixel_w;
    R film_y = (R(y) + py) * g.pixel_h;
    V3<R> fwd = mk<R>(g.fwd[0], g.fwd[1], g.fwd[2]);
    V3<R> ap = mk<R>(g.ap_pos[0], g.ap_pos[1], g.ap_pos[2]);
    V3<R> point = (mk<R>(g.right[0], g.right[1], g.right[2]) * film_x + mk<R>(g.up[0], g.up[1], g.up[2]) * film_y)
                  + mk<R>(g.film_bl[0], g.film_bl[1], g.film_bl[2]);
    V3<R> o, d;
    if(g.ap_radius > R(0))
    {
        V3<R> focus_dir = normalise(ap - point);
        focus_dir = focus_dir * r_div(g.focal_depth, dot(focus_dir, fwd));
        V3<R> focus_point = point + focus_dir;
        V3<R> disc = sample_disc<R>(rng) * g.ap_radius;
        V3<R> lens = mk<R>(g.lens_rot[0] * disc.x + g.lens_rot[3] * disc.y + g.lens_rot[6] * disc.z,
                           g.lens_rot[1] * disc.x + g.lens_rot[4] * disc.y + g.lens_rot[7] * disc.z,
                           g.lens_rot[2] * disc.x + g.lens_rot[5] * disc.y + g.lens_rot[8] * disc.z);
        o = ap + lens;
        d = normalise(focus_point - o);
    }
    else
    {
        o = point;
        d = normalise(ap - o);   /* Q1 */
    }
    rec[REC_VIG] = (float)dot(d, fwd);   /* Q20 */

    uint32_t nb = 0, closest = 0, shadow = 0, shaded = 0, end_depth = L.max_depth, general = 0, emitter = 0;
    int skip = -1;
    const uint32_t bw = L.bounce_words, ew = L.eval_words;
    for(uint32_t depth = 0; depth < L.max_depth; depth += 1)
    {
        Hit<R> h;
        closest += 1;
        bool found = closest_hit<R>(g, o, d, skip, h);
        int m = found ? h.surf_mat : g.escape_mat;
        int flags = g.mflags[m];
        /* this bounce's words: in the slot's shared-memory record, or (DEEP instantiations: renders whose records do not fit) -- past
         * the L.smem_depth bounces that fit there -- in the slot's global overflow row `deep` (RenderLaunch::deep) */
        const bool in_smem = !DEEP || nb < L.smem_depth;
        float *rb = in_smem ? rec + REC_HEAD + nb * bw : deep + (nb - L.smem_depth) * bw;
        if(flags & 1)   /* black body: escape or emitter, cast_ray :451-457 */
        {
            if(flags & 2)
            {
                if(ALLFAST) emitter = (uint32_t)(m + 1) << 16;   /* compact records: the closing emitter rides in word 0 */
                else { rb[0] = __uint_as_float(KIND_EMIT | ((uint32_t)m << 3)); nb += 1; }   /* Q6 */
            }
            end_depth = depth;
            break;
        }
        shaded += 1;
        /* Plastic (bp_diffuse + bp_glossy): two weights per evaluation, computed inline; under a single light the bounce also has a
         * fixed-size "fast" record (8 words in the general kernel, 4 in the compact-record kernels).  Shadow rays, direction sampling
         * and the weight arithmetic are shared by all materials so that a warp whose lanes sit on different materials does not run
         * them twice.  The classed kernel (MODE 2) gives specular and rough-conductor bounces 4-word records too (drt_device.cuh). */
        const int sm = h.surf_mat;
        const int cls = CLASSED ? g.mclass[sm] : DRT_CLASS_PLASTIC;
        const bool plastic = ALLFAST ? (cls == DRT_CLASS_PLASTIC) : (g.bmask[sm] == BMASK_PLASTIC && g.nlobes[sm] == 2);
        const bool fast = ALLFAST || (plastic && ix.plastic2[sm] != 0);
        const int nlights = ALLFAST ? 1 : g.nlights;
        float *recw = in_smem ? rec + L.head_words + 4u * nb : deep + 4u * (nb - L.smem_depth);   /* this bounce's four words in a compact record */
        if(CLASSED && cls == DRT_CLASS_ROUGH) { recw[0] = 0.f; recw[1] = 1.f; }   /* the light may turn out hidden */
        /* K3: direct_light_contribution, :272-332 -- every emissive surface in index order; draws come before visibility */
        uint32_t vis_mask = 0;
        float wd_n = 0.f, wg_n = 0.f;
        for(int j = 0; j < nlights; j += 1)
        {
            int ls = g.light_surf[j];
            int lt = g.type[ls];
            V3<R> lp = mk<R>(g.px[ls], g.py[ls], g.pz[ls]);
            R k;
            if(lt == DRT_GEO_POINT)
            {
                V3<R> to = lp - h.pos;
                R dist = r_sqrt(dot(to, to));
                k = (R(4) * Num<R>::pi() * dist * dist) * g.light_pdf[ls];   /* Q3 */
            }
            else if(lt == DRT_GEO_SPHERE)
            {
                R u = rng.unit<R>();
                R v = rng.unit<R>();
                R r = r_sqrt(R(1) - u * u);
                R s, c;
                r_sincospi(R(2) * v, &s, &c);
                lp = lp + mk<R>(r * c, r * s, u) * g.rad[ls];   /* Q5 */
                k = g.light_pdf[ls];
            }
            else
            {
                R u = rng.unit<R>();
                R v = rng.unit<R>();
                lp = (lp + mk<R>(g.ux[ls], g.uy[ls], g.uz[ls]) * u) + mk<R>(g.vx[ls], g.vy[ls], g.vz[ls]) * v;
                k = g.light_pdf[ls];
            }
            shadow += 1;
            V3<R> ldir;
            if(visible<R>(g, h.pos, lp, h.plane_slot, ldir))
            {
                const uint32_t e = 2 + (ew + 1) * (uint32_t)j;
                if(plastic)
                {
                    plastic_weights<R>(g, sm, h.nrm, h.out, ldir, fast ? (float)k : 1.f, wd_n, wg_n);
                    if(!fast) { rb[e] = wd_n; rb[e + 1] = wg_n; }
                }
                else if(CLASSED)
                {
                    /* rough conductor: w k and the micro-normal cosine; a specular material contributes nothing to next-event
                     * estimation (its lobes are gated on the exact reflection / refraction direction, Q8) */
                    if(cls == DRT_CLASS_ROUGH)
                    {
                        const float2 wc = ct_weight<R>(g, sm, h.nrm, h.out, h.on_dot, ldir);
                        recw[0] = wc.x * (float)k; recw[1] = wc.y;
                    }
                }
                else eval_weights_general<R>(g, sm, h.nrm, h.out, h.on_dot, ldir, 0, 1.f, rb, e);
                if(!fast) rb[e + ew] = (float)k;
                vis_mask |= 1u << j;
            }
        }
        /* K4: sample the next direction and evaluate the BSDF for it, cast_ray :464-472 */
        V3<R> in; R inv_pdf; int match;
        const uint32_t es = 2 + (ew + 1) * (uint32_t)nlights;
        float wd_s = 0.f, wg_s = 0.f;
        if(ALLFAST && plastic && depth + 1 == L.max_depth && g.dirf[sm] == DRT_DIR_COS_WEIGHTED_HEMISPHERE)
        {
            /* The last bounce's sampled direction is never cast, and the compact replay multiplies its weights by e = 0 (replay_compact):
             * it is not sampled, and its weights are 0.  The cosine sampler's two draws are still counted.  No draw follows them in
             * this path (the next path has a stream of its own), so only the draw counter sees them; it differs from the reference's
             * only when the disc sample would have been rejected (|q| rounds to 1, Q16). */
            rng.draws += 2;
            in = h.nrm;
        }
        else
        {
            sample_direction<R>(g, h, rng, in, inv_pdf, match);
            if(plastic) plastic_weights<R>(g, sm, h.nrm, h.out, in, (float)inv_pdf, wd_s, wg_s);
            else if(!CLASSED) eval_weights_general<R>(g, sm, h.nrm, h.out, h.on_dot, in, match, (float)inv_pdf, rb, es);
        }
        if(ALLFAST)
        {
            uint32_t hdr16;
            if(plastic)
            {
                /* four weights per bounce; the 16-bit header (class 0 | D, G block word offset, a multiple of 4) apart */
                *reinterpret_cast<float4 *>(recw) = make_float4(wd_n, wg_n, wd_s, wg_s);
                hdr16 = (uint32_t)ix.plastic2[sm];
            }
            else
            {
                general = 1;   /* sorts the path among those whose replay leaves the plastic loop */
                const uint32_t inside = (h.inc_mat != g.base_mat) ? 1u : 0u;
                if(cls == DRT_CLASS_ROUGH)
                {
                    const float2 wc = ct_weight<R>(g, sm, h.nrm, h.out, h.on_dot, in);
                    recw[2] = wc.x * (float)inv_pdf; recw[3] = wc.y;
                    hdr16 = (uint32_t)DRT_CLASS_ROUGH | (inside << 4) | ((uint32_t)sm << 5);
                }
                else
                {
                    /* (c0 + c1 X) / pdf over the material's one spectral basis X, constants tabulated per match (GeomT::spec_c) */
                    const int mask = g.bmask[sm], mt = match & 3;
                    recw[0] = g.spec_c[sm][mt < 3 ? mt : 0][0] * (float)inv_pdf;
                    recw[1] = g.spec_c[sm][mt < 3 ? mt : 0][1] * (float)inv_pdf;
                    recw[2] = (float)h.on_dot;
                    const uint32_t basis = (mask & (1 << BK_MIRROR)) ? 0u : (mask & (1 << BK_DIEL_R)) ? 1u : 2u;
                    hdr16 = (uint32_t)DRT_CLASS_SPECULAR | (basis << 2) | (inside << 4) | ((uint32_t)sm << 5);
                }
            }
            if(nb == 0u)
            {
                /* every term of the path carries the first bounce's next-event or sampled-direction weights, so the vignette factor
                 * (dot(ray direction, forward), sample_scene :612-615) is folded into them here, once per path by one thread, instead
                 * of multiplying the finished spectrum in the replay (a path without a shaded bounce is scaled there) */
                const float vig = rec[REC_VIG];
                const uint32_t c = hdr16 & 3u;
                recw[0] *= vig;
                if(c != (uint32_t)DRT_CLASS_ROUGH) recw[1] *= vig;
                if(c != (uint32_t)DRT_CLASS_SPECULAR) recw[2] *= vig;
                if(c == (uint32_t)DRT_CLASS_PLASTIC) recw[3] *= vig;
            }
            if(in_smem) reinterpret_cast<uint16_t *>(rec + REC_HDR16)[nb] = (uint16_t)hdr16;
            else reinterpret_cast<uint16_t *>(deep + L.deep_hdr_off)[nb - L.smem_depth] = (uint16_t)hdr16;
        }
        else if(fast)
        {
            float4 *r4 = reinterpret_cast<float4 *>(rb);
            r4[0] = make_float4(__uint_as_float(KIND_SHADE | HDR_FAST | ((uint32_t)ix.plastic2[sm] << 2)), wd_n, wg_n, 0.f);
            r4[1] = make_float4(wd_s, wg_s, 0.f, 0.f);
        }
        else
        {
            general = 1;
            if(plastic) { rb[es] = wd_s; rb[es + 1] = wg_s; }
            uint32_t swapped = (h.inc_mat != g.base_mat) ? 1u : 0u;
            rb[0] = __uint_as_float(KIND_SHADE | ((uint32_t)sm << 3) | (swapped << 8) | (vis_mask << 16));
            rb[1] = (float)h.on_dot;
        }
        nb += 1;
        d = in;
        o = h.pos;
        skip = h.plane_slot;
    }
    rec[REC_NB] = __uint_as_float(nb | emitter);
    tally[0] += closest; tally[1] += shadow; tally[2] += shaded; tally[3] += rng.draws;
    /* bits 0-7: histogram bin (depth of termination, 8 = hit the cap); bit 8: the record has a bounce that needs the general shader */
    return ((end_depth < L.max_depth) ? (end_depth < 7 ? end_depth : 7) : 8) | (general << 8);
}

/* ------------------------------------------------------------------ packed f32x2 arithmetic (sm_100 fma.rn.f32x2)
 * The replay is bound by instruction issue, not by the FMA pipe: one packed instruction does the work of two for the
 * wavelength slots (0,1), (2,3); an odd last slot stays scalar.  Results are bit-identical to the scalar forms. */
__device__ __forceinline__ unsigned long long pk2(float a, float b) { unsigned long long r; asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(a), "f"(b)); return r; }
__device__ __forceinline__ void upk2(unsigned long long v, float &a, float &b) { asm("mov.b64 {%0, %1}, %2;" : "=f"(a), "=f"(b) : "l"(v)); }
__device__ __forceinline__ unsigned long long fma2(unsigned long long a, unsigned long long b, unsigned long long c)
{ unsigned long long r; asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(a), "l"(b), "l"(c)); return r; }
__device__ __forceinline__ unsigned long long mul2(unsigned long long a, unsigned long long b)
{ unsigned long long r; asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b)); return r; }
/* acc += a * b and x *= t in place: the loop-carried accumulators keep their registers */
__device__ __forceinline__ void fma2_acc(unsigned long long &acc, unsigned long long a, unsigned long long b)
{ asm("fma.rn.f32x2 %0, %1, %2, %0;" : "+l"(acc) : "l"(a), "l"(b)); }
__device__ __forceinline__ void mul2_by(unsigned long long &x, unsigned long long t)
{ asm("mul.rn.f32x2 %0, %0, %1;" : "+l"(x) : "l"(t)); }
__device__ __forceinline__ void add2_acc(unsigned long long &acc, unsigned long long x)
{ asm("add.rn.f32x2 %0, %0, %1;" : "+l"(acc) : "l"(x)); }
__device__ __forceinline__ unsigned long long add2(unsigned long long a, unsigned long long b)
{ unsigned long long r; asm("add.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b)); return r; }

/* o = a*b + c,  o = s*b + c,  o = a*b,  o = s*b  over NS wavelength slots */
template <int NS> __device__ __forceinline__ void v_fma(float (&o)[NS], const float (&a)[NS], const float (&b)[NS], const float (&c)[NS])
{
#pragma unroll
    for(int k = 0; k + 1 < NS; k += 2) upk2(fma2(pk2(a[k], a[k + 1]), pk2(b[k], b[k + 1]), pk2(c[k], c[k + 1])), o[k], o[k + 1]);
    if(NS & 1) o[NS - 1] = fmaf(a[NS - 1], b[NS - 1], c[NS - 1]);
}
template <int NS> __device__ __forceinline__ void v_fma_s(float (&o)[NS], float s, const float (&b)[NS], const float (&c)[NS])
{
#pragma unroll
    for(int k = 0; k + 1 < NS; k += 2) upk2(fma2(pk2(s, s), pk2(b[k], b[k + 1]), pk2(c[k], c[k + 1])), o[k], o[k + 1]);
    if(NS & 1) o[NS - 1] = fmaf(s, b[NS - 1], c[NS - 1]);
}
template <int NS> __device__ __forceinline__ void v_mul(float (&o)[NS], const float (&a)[NS], const float (&b)[NS])
{
#pragma unroll
    for(int k = 0; k + 1 < NS; k += 2) upk2(mul2(pk2(a[k], a[k + 1]), pk2(b[k], b[k + 1])), o[k], o[k + 1]);
    if(NS & 1) o[NS - 1] = a[NS - 1] * b[NS - 1];
}
template <int NS> __device__ __forceinline__ void v_mul_s(float (&o)[NS], float s, const float (&b)[NS])
{
#pragma unroll
    for(int k = 0; k + 1 < NS; k += 2) upk2(mul2(pk2(s, s), pk2(b[k], b[k + 1])), o[k], o[k + 1]);
    if(NS & 1) o[NS - 1] = s * b[NS - 1];
}
template <int NS> __device__ __forceinline__ void v_add(float (&o)[NS], const float (&a)[NS], const float (&b)[NS])
{
#pragma unroll
    for(int k = 0; k + 1 < NS; k += 2) upk2(add2(pk2(a[k], a[k + 1]), pk2(b[k], b[k + 1])), o[k], o[k + 1]);
    if(NS & 1) o[NS - 1] = a[NS - 1] + b[NS - 1];
}
/* a - b as b * (-1) + a: one packed instruction per slot pair (a packed add has no negate modifier, and negating b first costs
 * one more instruction per slot); exact, so bit-identical to the subtraction */
template <int NS> __device__ __forceinline__ void v_sub(float (&o)[NS], const float (&a)[NS], const float (&b)[NS])
{
    const unsigned long long m1 = pk2(-1.f, -1.f);
#pragma unroll
    for(int k = 0; k + 1 < NS; k += 2) upk2(fma2(pk2(b[k], b[k + 1]), m1, pk2(a[k], a[k + 1])), o[k], o[k + 1]);
    if(NS & 1) o[NS - 1] = a[NS - 1] - b[NS - 1];
}

/* ------------------------------------------------------------------ phase 2: spectral replay of one record by a HALF warp
 *
 * A path is shaded by 16 lanes: lane l16 = lane & 15 holds wavelengths l16, l16+16, ... (NS register slots; 5 for N = 69,
 * 86 % of the slots carry a wavelength against 72 % for a 32-lane layout), and the two halves of a warp replay two
 * paths at once, sharing every address, header-decode and loop instruction.  `col` is the record column of the path (word w at
 * col[w*32]); every read of it is a shared-memory broadcast.  SpdIndex.row holds WORD OFFSETS into the pool. */

template <int NS> struct Spec { float v[NS]; };
template <int NS> struct ShadeState { Spec<NS> thr, dst; };

/* Fresnel terms on the rows precomputed at upload (SpdIndex::fres): the formulas of fresnel_dielectric above and of
 * fs_conductor_reflectance (bdsf.c:78-101) with the per-wavelength ratios taken out (rel = ir / tr;  A = eta^2 - kappa^2,
 * B = 4 eta^2 kappa^2 with eta = tr / ir, kappa = te / ir), numerator and denominator of the dielectric amplitudes divided by tr
 * (bdsf.c:44-76, Q9 kept).  Scalar and out of line: each formula exists once in a kernel however many wavelength slots a lane holds
 * -- the kernels that contain them are bound by instruction fetch, so small code beats straight-line code. */
static __device__ __noinline__ float fresnel_dielectric_rel(float rel, float inc_cos)
{
    const float inc_sin_sq = 1.f - inc_cos * inc_cos;
    const float ts_sin_sq = rel * rel * inc_sin_sq;
    if(ts_sin_sq >= 1.f) return 1.f;
    const float ts_cos = r_sqrt_fast(1.f - ts_sin_sq * ts_sin_sq);
    const float a = rel * ts_cos, b = rel * inc_cos;
    const float par = r_div(inc_cos - a, inc_cos + a);
    const float per = r_div(b - ts_cos, b + ts_cos);
    return 0.5f * (par * par + per * per);
}
static __device__ __noinline__ float fresnel_conductor_ab(float A, float B, float inc_cos)
{
    const float cos_sq = inc_cos * inc_cos, sin_sq = 1.f - cos_sq;
    const float r = A - sin_sq;
    const float apb_sq = r_sqrt_fast(fmaf(r, r, B));
    const float a = r_sqrt_fast(fmaxf(0.5f * (apb_sq + r), 0.f));   /* clamp: see fresnel_conductor */
    const float s = apb_sq + cos_sq;
    const float t = 2.f * a * inc_cos;
    const float u = fmaf(cos_sq, apb_sq, sin_sq * sin_sq);
    const float v = t * sin_sq;
    const float par = r_div(s - t, s + t);
    const float per = r_div(par * (u - v), u + v);
    return 0.5f * (par + per);
}

/* The same two Fresnel terms for TWO wavelength slots at once (packed f32x2 arithmetic; the square roots and reciprocals stay one
 * MUFU per element): the classed kernel's specular and rough-conductor bounces evaluate them for the slot pairs (0,1), (2,3), ... */
static __device__ __noinline__ unsigned long long fresnel_conductor_ab2(unsigned long long A2, unsigned long long B2, float inc_cos)
{
    const float cos_sq = inc_cos * inc_cos, sin_sq = 1.f - cos_sq;
    const unsigned long long m1 = pk2(-1.f, -1.f), cs2 = pk2(cos_sq, cos_sq);
    const unsigned long long r2 = add2(A2, pk2(-sin_sq, -sin_sq));
    float q0, q1;
    upk2(fma2(r2, r2, B2), q0, q1);
    const unsigned long long apb2 = pk2(r_sqrt_fast(q0), r_sqrt_fast(q1));
    upk2(mul2(add2(apb2, r2), pk2(0.5f, 0.5f)), q0, q1);
    const unsigned long long a2 = pk2(r_sqrt_fast(fmaxf(q0, 0.f)), r_sqrt_fast(fmaxf(q1, 0.f)));   /* clamp: see fresnel_conductor_ab */
    const unsigned long long s2 = add2(apb2, cs2);
    const unsigned long long t2 = mul2(a2, pk2(2.f * inc_cos, 2.f * inc_cos));
    const unsigned long long u2 = fma2(apb2, cs2, pk2(sin_sq * sin_sq, sin_sq * sin_sq));
    const unsigned long long v2 = mul2(t2, pk2(sin_sq, sin_sq));
    upk2(add2(s2, t2), q0, q1);
    const unsigned long long par2 = mul2(fma2(t2, m1, s2), pk2(r_rcp_fast(q0), r_rcp_fast(q1)));
    upk2(add2(u2, v2), q0, q1);
    const unsigned long long per2 = mul2(mul2(par2, fma2(v2, m1, u2)), pk2(r_rcp_fast(q0), r_rcp_fast(q1)));
    return mul2(add2(par2, per2), pk2(0.5f, 0.5f));
}
static __device__ __noinline__ unsigned long long fresnel_dielectric_rel2(unsigned long long rel2, float inc_cos)
{
    const float inc_sin_sq = 1.f - inc_cos * inc_cos;
    const unsigned long long m1 = pk2(-1.f, -1.f), c2 = pk2(inc_cos, inc_cos);
    const unsigned long long ts2 = mul2(mul2(rel2, rel2), pk2(inc_sin_sq, inc_sin_sq));
    float t0, t1, q0, q1;
    upk2(ts2, t0, t1);
    upk2(fma2(mul2(ts2, m1), ts2, pk2(1.f, 1.f)), q0, q1);
    const unsigned long long tc2 = pk2(r_sqrt_fast(fmaxf(q0, 0.f)), r_sqrt_fast(fmaxf(q1, 0.f)));   /* negative only under total reflection, replaced below */
    const unsigned long long a2 = mul2(rel2, tc2), b2 = mul2(rel2, c2);
    upk2(add2(c2, a2), q0, q1);
    const unsigned long long par2 = mul2(fma2(a2, m1, c2), pk2(r_rcp_fast(q0), r_rcp_fast(q1)));
    upk2(add2(b2, tc2), q0, q1);
    const unsigned long long per2 = mul2(fma2(tc2, m1, b2), pk2(r_rcp_fast(q0), r_rcp_fast(q1)));
    float f0, f1;
    upk2(mul2(fma2(per2, per2, mul2(par2, par2)), pk2(0.5f, 0.5f)), f0, f1);
    return pk2(t0 >= 1.f ? 1.f : f0, t1 >= 1.f ? 1.f : f1);   /* total internal reflection (bdsf.c:52) */
}

/* One BSDF evaluation expanded over this lane's wavelengths, any lobe list: the stored weights of the seven spectral bases
 * (eval_weights_general) times the bases.  `mask` is warp-uniform; a Fresnel basis whose weight is zero (every match-gated lobe under
 * next-event estimation) is not evaluated. */
template <int NS>
__device__ __forceinline__ Spec<NS> eval_spectrum_general(const float *col, uint32_t at, int mask, const SpdIndex &ix, const float *pool_lane,
                                                          int surf_mat, int inside, float on_dot)
{
    float w_const = 0.f, w_d = 0.f, w_g = 0.f, w_m = 0.f, w_r = 0.f, w_a = 0.f, w_b = 0.f, c_b = 0.f;
    if(mask & (1 << BK_CONST))   { w_const = col[at]; at += 1; }
    if(mask & (1 << BK_DIFFUSE)) { w_d = col[at]; at += 1; }
    if(mask & (1 << BK_GLOSSY))  { w_g = col[at]; at += 1; }
    if(mask & (1 << BK_MIRROR))  { w_m = col[at]; at += 1; }
    if(mask & (1 << BK_DIEL_R))  { w_r = col[at]; at += 1; }
    if(mask & (1 << BK_COND_ON)) { w_a = col[at]; at += 1; }
    if(mask & (1 << BK_COND_MN)) { w_b = col[at]; c_b = col[at + 1]; }
    const float *dr = pool_lane + ix.row[surf_mat][DRT_SPD_DIFFUSE];     /* absent spectra point at the all-zero row */
    const float *gr = pool_lane + ix.row[surf_mat][DRT_SPD_GLOSSY];
    const float *mr = pool_lane + ix.row[surf_mat][DRT_SPD_MIRROR];
    Spec<NS> f;
#pragma unroll
    for(int k = 0; k < NS; k += 1)
        f.v[k] = fmaf(w_m, mr[k * DRT_HALF], fmaf(w_g, gr[k * DRT_HALF], fmaf(w_d, dr[k * DRT_HALF], w_const)));
    if(w_r != 0.f)
    {
        const float *rel = pool_lane + ix.fres[surf_mat][inside][0];
#pragma unroll
        for(int k = 0; k + 1 < NS; k += 2)
        {
            float r0, r1;
            upk2(fresnel_dielectric_rel2(pk2(rel[k * DRT_HALF], rel[(k + 1) * DRT_HALF]), on_dot), r0, r1);
            f.v[k] = fmaf(w_r, r0, f.v[k]); f.v[k + 1] = fmaf(w_r, r1, f.v[k + 1]);
        }
        if(NS & 1) f.v[NS - 1] = fmaf(w_r, fresnel_dielectric_rel(rel[(NS - 1) * DRT_HALF], on_dot), f.v[NS - 1]);
    }
    if(w_a != 0.f || w_b != 0.f)
    {
        const float *ra = pool_lane + ix.fres[surf_mat][inside][1], *rb = pool_lane + ix.fres[surf_mat][inside][2];
#pragma unroll 1
        for(int t = 0; t < 2; t += 1)   /* F(on_dot) of fs_conductor_bdsf, F(micro-normal cosine) of ct_conductor_bdsf: one loop body */
        {
            const float w = t ? w_b : w_a, cs = t ? c_b : on_dot;
            if(w == 0.f) continue;
#pragma unroll
            for(int k = 0; k + 1 < NS; k += 2)
            {
                float r0, r1;
                upk2(fresnel_conductor_ab2(pk2(ra[k * DRT_HALF], ra[(k + 1) * DRT_HALF]), pk2(rb[k * DRT_HALF], rb[(k + 1) * DRT_HALF]), cs), r0, r1);
                f.v[k] = fmaf(w, r0, f.v[k]); f.v[k + 1] = fmaf(w, r1, f.v[k + 1]);
            }
            if(NS & 1) f.v[NS - 1] = fmaf(w, fresnel_conductor_ab(ra[(NS - 1) * DRT_HALF], rb[(NS - 1) * DRT_HALF], cs), f.v[NS - 1]);
        }
    }
    return f;
}

/* One shaded bounce of cast_ray (daily_ray_trace.c:458-473) for any material and any number of lights, out of line. */
template <int NS, typename G>
static __device__ __noinline__ ShadeState<NS> shade_bounce_general(const float *col, uint32_t base, uint32_t hdr, const G &g, const SpdIndex &ix,
                                                            const float *pool_lane, uint32_t ew, int nlights, ShadeState<NS> st)
{
    const int surf_mat = (hdr >> 3) & 31;
    const int mask = g.bmask[surf_mat];
    const bool swapped = (hdr >> 8) & 1u;
    const int inside = swapped ? 1 : 0;   /* the orientation of the Fresnel rows: 1 = incident medium is the surface's material (Q11) */
    const uint32_t vis = hdr >> 16;
    const float on_dot = col[base + 1];
    float contrib[NS];
#pragma unroll
    for(int k = 0; k < NS; k += 1) contrib[k] = 0.f;
#pragma unroll 1
    for(int j = 0; j < nlights; j += 1)
    {
        if(!((vis >> j) & 1u)) continue;
        uint32_t e = base + 2 + (ew + 1) * (uint32_t)j;
        Spec<NS> f = eval_spectrum_general<NS>(col, e, mask, ix, pool_lane, surf_mat, inside, on_dot);
        float kk = col[e + ew];
        const float *erow = pool_lane + ix.row[g.mat[g.light_surf[j]]][DRT_SPD_EMISSION];
#pragma unroll
        for(int k = 0; k < NS; k += 1) contrib[k] = ((contrib[k] + f.v[k]) * erow[k * DRT_HALF]) * kk;   /* Q4 */
    }
#pragma unroll
    for(int k = 0; k < NS; k += 1) st.dst.v[k] = fmaf(st.thr.v[k], contrib[k], st.dst.v[k]);
    Spec<NS> f = eval_spectrum_general<NS>(col, base + 2 + (ew + 1) * (uint32_t)nlights, mask, ix, pool_lane, surf_mat, inside, on_dot);
#pragma unroll
    for(int k = 0; k < NS; k += 1) st.thr.v[k] *= f.v[k];
    return st;
}

/* ------------------------------------------------------------------ classed kernel: specular and rough-conductor bounces */
/* One bounce of class SPECULAR or ROUGH (record layout: RenderLaunch in drt_device.cuh) on the backward replay's packed state r2 / r1
 * (the slot pairs and the odd last slot; see replay_compact).  Inline (the struct-passing call cost 4 %), the Fresnel formulas
 * themselves out of line. */
template <int NS>
__device__ __forceinline__ void shade_special(uint32_t hdr, float4 w, const float *pool_lane, const SpdIndex &ix,
                                              unsigned long long (&r2)[NS / 2 > 0 ? NS / 2 : 1], float &r1)
{
    constexpr int NP = NS / 2;
    const int cls = (int)(hdr & 3u), inside = (int)((hdr >> 4) & 1u), mat = (int)((hdr >> 5) & 31u);
    if(cls == DRT_CLASS_SPECULAR)
    {
        /* r = (c0 + c1 X) / pdf * r: the bounce emits nothing (cast_ray :467-469); X = mirror spectrum, dielectric R(on_dot) or
         * conductor F(on_dot) */
        const uint32_t basis = (hdr >> 2) & 3u;
        const float *x0 = pool_lane + (basis == 0u ? ix.row[mat][DRT_SPD_MIRROR] : basis == 1u ? ix.fres[mat][inside][0] : ix.fres[mat][inside][1]);
        const float *x1 = pool_lane + ix.fres[mat][inside][2];
        const unsigned long long c0 = pk2(w.x, w.x), c1 = pk2(w.y, w.y);
#pragma unroll
        for(int k = 0; k < NP; k += 1)
        {
            unsigned long long x = pk2(x0[(2 * k) * DRT_HALF], x0[(2 * k + 1) * DRT_HALF]);
            if(basis == 1u) x = fresnel_dielectric_rel2(x, w.z);
            else if(basis == 2u) x = fresnel_conductor_ab2(x, pk2(x1[(2 * k) * DRT_HALF], x1[(2 * k + 1) * DRT_HALF]), w.z);
            mul2_by(r2[k], fma2(c1, x, c0));
        }
        if(NS & 1)
        {
            float x = x0[(NS - 1) * DRT_HALF];
            if(basis == 1u) x = fresnel_dielectric_rel(x, w.z);
            else if(basis == 2u) x = fresnel_conductor_ab(x, x1[(NS - 1) * DRT_HALF], w.z);
            r1 *= fmaf(w.y, x, w.x);
        }
    }
    else
    {
        const float *ra = pool_lane + ix.fres[mat][inside][1], *rb = pool_lane + ix.fres[mat][inside][2];
        /* the rows are re-read for the second evaluation: keeping them in registers across the calls spills */
        auto rows2 = [&](int k, unsigned long long &a2, unsigned long long &b2)
        {
            a2 = pk2(ra[(2 * k) * DRT_HALF], ra[(2 * k + 1) * DRT_HALF]); b2 = pk2(rb[(2 * k) * DRT_HALF], rb[(2 * k + 1) * DRT_HALF]);
        };
        const float a1 = (NS & 1) ? ra[(NS - 1) * DRT_HALF] : 0.f, b1 = (NS & 1) ? rb[(NS - 1) * DRT_HALF] : 0.f;
        /* r = w / pdf F(cos_s) r + w k F(cos_n), cast_ray :458-469; the second term only when the light is visible */
        const unsigned long long ws = pk2(w.z, w.z);
#pragma unroll
        for(int k = 0; k < NP; k += 1) { unsigned long long a2, b2; rows2(k, a2, b2); mul2_by(r2[k], mul2(ws, fresnel_conductor_ab2(a2, b2, w.w))); }
        if(NS & 1) r1 *= w.z * fresnel_conductor_ab(a1, b1, w.w);
        if(w.x != 0.f)
        {
            const unsigned long long wn = pk2(w.x, w.x);
#pragma unroll
            for(int k = 0; k < NP; k += 1) { unsigned long long a2, b2; rows2(k, a2, b2); fma2_acc(r2[k], wn, fresnel_conductor_ab2(a2, b2, w.y)); }
            if(NS & 1) r1 = fmaf(w.x, fresnel_conductor_ab(a1, b1, w.y), r1);
        }
    }
}

/* One 16-bit bounce header of a compact record, zero-extended into a 32-bit register.  A plain 16-bit load keeps the loop-carried
 * header as a 16-bit value, which costs two more instructions per bounce to merge and widen.  Deep renders keep the generic load:
 * their headers may lie in the global overflow row. */
template <bool DEEP> __device__ __forceinline__ uint32_t load_hdr16(const uint16_t *p)
{
    if constexpr(DEEP) return *p;
    uint32_t v;
    asm volatile("ld.shared.u16 %0, [%1];" : "=r"(v) : "r"((uint32_t)__cvta_generic_to_shared(p)));
    return v;
}

/* Compact records (modes 1 and 2; RenderLaunch in drt_device.cuh: header halves from word 2, four weights per bounce).  The light is
 * the scene's only emitter, so every term of cast_ray's radiance (daily_ray_trace.c:446-473) is E times the light-free factors, and
 * the path's contribution is E * r with, for a plastic bounce b (NEE weights n_b, sampled-direction weights s_b),
 *     n_b = wd_n k D + wg_n k G    (NEE: bdsf * k, :322-327; the weights are 0 when the light is hidden)
 *     s_b = wd_s/pdf D + wg_s/pdf G (:467-469)
 *     r   = n_0 + s_0 (n_1 + s_1 (... (n_last + s_last e)))       e = 1 if the path ends on the light (:453-457), else 0.
 * This evaluates r from the last bounce back to the first (Horner form), four f32x2 operations per slot pair and bounce:
 *     r = D (wd_n + wd_s r) + G (wg_n + wg_s r)
 * and two for the last bounce, whose r = e is a constant.  The vignette factor (:612-615) rides in bounce 0's weights (trace_path);
 * a path that meets the light without a shaded bounce has r = vignette.  r is returned as f32x2 register pairs for wavelength slots
 * (0,1), (2,3), ... (r2) plus one scalar for an odd last slot (r1); E is applied once per batch (PixelFilm::add_batch). */
template <int NS, int MODE, bool DEEP>
__device__ __forceinline__ void replay_compact(const float *col, const float *deep, uint32_t nb, const SpdIndex &ix, const float *pool, const float *pool_lane,
                                               uint32_t lane16, const RenderLaunch &L, unsigned long long (&r2)[NS / 2 > 0 ? NS / 2 : 1], float &r1)
{
    constexpr bool CLASSED = MODE == 2;
    constexpr int NP = NS / 2;
    const uint32_t nshade = nb & 0xffffu;
    if(nshade == 0u)   /* the camera ray met the light */
    {
        const float v = col[REC_VIG];
#pragma unroll
        for(int k = 0; k < NP; k += 1) r2[k] = pk2(v, v);
        r1 = v;
        return;
    }
    /* The bounces come in at most two spans: the first L.smem_depth in the slot's shared-memory record, the rest (deep renders only)
     * in the slot's global overflow row, which is walked first.  b counts down through the current span; `rest` bounces of the
     * shared-memory span are left when the overflow row is done. */
    int b = (int)nshade - 1;
    int rest = 0;
    const uint16_t *hp = reinterpret_cast<const uint16_t *>(col + REC_HDR16) + b;   /* this bounce's header and weights */
    const float4 *wp = reinterpret_cast<const float4 *>(col + L.head_words) + b;
    if(DEEP && nshade > L.smem_depth)
    {
        rest = (int)L.smem_depth;
        b = (int)(nshade - L.smem_depth) - 1;
        hp = reinterpret_cast<const uint16_t *>(deep + L.deep_hdr_off) + b;
        wp = reinterpret_cast<const float4 *>(deep) + b;
    }
    /* The previous bounce's header is in flight while this one is shaded (the D, G block address depends on it; the weights are
     * loaded together with the block and need no head start).  Before the first bounce of the shared-memory span this reads (and
     * never uses) the record's head words; in deep renders the step back stops at the span's first bounce, since the word before an
     * overflow row may lie outside the allocation. */
    auto step_back = [&]() { const int s = (!DEEP || b > 0) ? 1 : 0; hp -= s; wp -= s; };
    uint32_t hdr = load_hdr16<DEEP>(hp);
    const float e = (nb >> 16) ? 1.f : 0.f;
    if(!CLASSED || (hdr & 3u) == 0u)
    {
        /* the last bounce, a plastic: r = (wd_n + wd_s e) D + (wg_n + wg_s e) G */
        const float4 w = *wp;   /* wd_n k, wg_n k, wd_s / pdf, wg_s / pdf */
        const float4 *blk = reinterpret_cast<const float4 *>(pool + hdr) + lane16;
        const float wd = fmaf(w.z, e, w.x), wg = fmaf(w.w, e, w.y);
        const unsigned long long wd2 = pk2(wd, wd), wg2 = pk2(wg, wg);
        step_back();
        hdr = load_hdr16<DEEP>(hp);
        b -= 1;
#pragma unroll
        for(int k = 0; k < NP; k += 1)
        {
            const float4 dg = blk[k * DRT_HALF];
            r2[k] = fma2(wg2, pk2(dg.z, dg.w), mul2(wd2, pk2(dg.x, dg.y)));
        }
        if(NS & 1)
        {
            const float2 q = *reinterpret_cast<const float2 *>(blk + NP * DRT_HALF);   /* D, G of the last slot */
            r1 = fmaf(wg, q.y, wd * q.x);
        }
    }
    else
    {
#pragma unroll
        for(int k = 0; k < NP; k += 1) r2[k] = pk2(e, e);
        r1 = e;
    }
#pragma unroll 1
    for(;;)
    {
#pragma unroll 1
        for(; b >= 0; b -= 1)
        {
            const float4 w = *wp;
            if constexpr(CLASSED)
            {
                if(hdr & 3u)   /* a specular or rough-conductor bounce */
                {
                    shade_special<NS>(hdr, w, pool_lane, ix, r2, r1);
                    step_back();
                    hdr = load_hdr16<DEEP>(hp);
                    continue;
                }
            }
            const float4 *blk = reinterpret_cast<const float4 *>(pool + hdr) + lane16;
            const unsigned long long wdn = pk2(w.x, w.x), wgn = pk2(w.y, w.y), wds = pk2(w.z, w.z), wgs = pk2(w.w, w.w);
            step_back();
            hdr = load_hdr16<DEEP>(hp);
#pragma unroll
            for(int k = 0; k < NP; k += 1)
            {
                const float4 dg = blk[k * DRT_HALF];
                r2[k] = fma2(pk2(dg.z, dg.w), fma2(wgs, r2[k], wgn), mul2(pk2(dg.x, dg.y), fma2(wds, r2[k], wdn)));
            }
            if(NS & 1)
            {
                const float2 q = *reinterpret_cast<const float2 *>(blk + NP * DRT_HALF);
                r1 = fmaf(q.y, fmaf(w.w, r1, w.y), q.x * fmaf(w.z, r1, w.x));
            }
        }
        if(!DEEP || rest == 0) break;
        b = rest - 1;
        rest = 0;
        hp = reinterpret_cast<const uint16_t *>(col + REC_HDR16) + b;
        wp = reinterpret_cast<const float4 *>(col + L.head_words) + b;
        hdr = load_hdr16<DEEP>(hp);
    }
}

/* cast_ray's spectral arithmetic (daily_ray_trace.c:446-473) replayed forward from a general record `col` (nb >= 1 bounces);
 * returns the path contribution already multiplied by the vignette factor (:612-615).
 * Throughput and radiance are held as f32x2 register pairs for wavelength slots (0,1), (2,3), ... plus one scalar for an
 * odd last slot.  The hot bounce (two-lobe plastic under the scene's only light) is
 *     radiance   += throughput * (wd_n k * DE + wg_n k * GE)        (NEE: bdsf * emission * k, :322-327; weights are 0 when shadowed)
 *     throughput *= wd_s/pdf * D + wg_s/pdf * G                      (:467-469)
 * with D, G from the material's D, G block (16-byte loads) and E from the light's slot pairs (SpdIndex::plastic2, light_pairs);
 * DE = D*E and GE = G*E are formed here. */
template <int NS, bool DEEP, typename G>
__device__ __forceinline__ void replay_path(const float *col, const float *deep, uint32_t nb, const G &g, const SpdIndex &ix, const float *pool, const float *pool_lane,
                                            uint32_t lane16, const RenderLaunch &L, float (&c)[NS])
{
    constexpr int NP = NS / 2;
    unsigned long long thr2[NP > 0 ? NP : 1], dst2[NP > 0 ? NP : 1];
    float thr1 = 1.f, dst1 = 0.f;
#pragma unroll
    for(int k = 0; k < NP; k += 1) { thr2[k] = pk2(1.f, 1.f); dst2[k] = pk2(0.f, 0.f); }
    const uint32_t bw = L.bounce_words, ew = L.eval_words;
    const float *p = (!DEEP || L.smem_depth) ? col + REC_HEAD : deep;
    float4 a_next = *reinterpret_cast<const float4 *>(p);
    for(uint32_t b = 0; b < nb; b += 1)
    {
        const float4 a = a_next;
        const float *pc = p;
        p = (DEEP && b + 1 == L.smem_depth) ? deep : p + bw;   /* past the bounces that fit in shared memory: the slot's global overflow row */
        if(b + 1 < nb) a_next = *reinterpret_cast<const float4 *>(p);   /* next header in flight while this bounce is shaded */
        const uint32_t hdr = __float_as_uint(a.x);
        if((hdr & HDR_FAST) != 0u)
        {
            const float4 s4 = *reinterpret_cast<const float4 *>(pc + 4);
            const float4 *blk = reinterpret_cast<const float4 *>(pool) + (hdr >> 4) + lane16;
            const float2 *ep = reinterpret_cast<const float2 *>(pool + ix.light_pairs) + lane16;
            const unsigned long long wdn = pk2(a.y, a.y), wgn = pk2(a.z, a.z), wds = pk2(s4.x, s4.x), wgs = pk2(s4.y, s4.y);
#pragma unroll
            for(int k = 0; k < NP; k += 1)
            {
                const float4 dg = blk[k * DRT_HALF];
                const float2 e = ep[k * DRT_HALF];
                const unsigned long long d2 = pk2(dg.x, dg.y), g2 = pk2(dg.z, dg.w), e2 = pk2(e.x, e.y);
                unsigned long long f = fma2(wgn, mul2(g2, e2), mul2(wdn, mul2(d2, e2)));
                dst2[k] = fma2(thr2[k], f, dst2[k]);
                unsigned long long t = fma2(wgs, g2, mul2(wds, d2));
                thr2[k] = mul2(thr2[k], t);
            }
            if(NS & 1)
            {
                const float2 q = *reinterpret_cast<const float2 *>(blk + NP * DRT_HALF);   /* D, G of the last slot */
                const float e = ep[NP * DRT_HALF].x;
                dst1 = fmaf(thr1, fmaf(a.z, q.y * e, a.y * (q.x * e)), dst1);
                thr1 *= fmaf(s4.y, q.y, s4.x * q.x);
            }
            continue;
        }
        if((hdr & 3u) == KIND_EMIT)   /* the path ran into an emitter, cast_ray :453-457 */
        {
            const float *row = pool_lane + ix.row[(hdr >> 3) & 31][DRT_SPD_EMISSION];
#pragma unroll
            for(int k = 0; k < NP; k += 1) dst2[k] = fma2(thr2[k], pk2(row[(2 * k) * DRT_HALF], row[(2 * k + 1) * DRT_HALF]), dst2[k]);
            if(NS & 1) dst1 = fmaf(thr1, row[(NS - 1) * DRT_HALF], dst1);
            break;
        }
        ShadeState<NS> st;
#pragma unroll
        for(int k = 0; k < NP; k += 1) { upk2(thr2[k], st.thr.v[2 * k], st.thr.v[2 * k + 1]); upk2(dst2[k], st.dst.v[2 * k], st.dst.v[2 * k + 1]); }
        if(NS & 1) { st.thr.v[NS - 1] = thr1; st.dst.v[NS - 1] = dst1; }
        st = shade_bounce_general<NS, G>(pc, 0u, hdr, g, ix, pool_lane, ew, L.nlights, st);
#pragma unroll
        for(int k = 0; k < NP; k += 1) { thr2[k] = pk2(st.thr.v[2 * k], st.thr.v[2 * k + 1]); dst2[k] = pk2(st.dst.v[2 * k], st.dst.v[2 * k + 1]); }
        if(NS & 1) { thr1 = st.thr.v[NS - 1]; dst1 = st.dst.v[NS - 1]; }
    }
    const float vig = col[REC_VIG];
    const unsigned long long vig2 = pk2(vig, vig);
#pragma unroll
    for(int k = 0; k < NP; k += 1) upk2(mul2(dst2[k], vig2), c[2 * k], c[2 * k + 1]);
    if(NS & 1) c[NS - 1] = dst1 * vig;
}

/* The replayed samples of one pixel in one batch that a half warp shaded, in units of the light's emission (replay_compact: sample
 * = E * r): count, S = sum of r and the shifted sum of squares Q = sum of (r - K)^2 about the half's first sample K, which keeps the
 * M2 of a pixel whose samples barely differ from cancelling (PixelFilm::add_batch).  Three f32x2 operations per slot pair and
 * sample, against the five of a per-sample Welford update and the E multiply. */
template <int NS> struct BatchStats
{
    static constexpr int NP = NS / 2, NP1 = NP > 0 ? NP : 1;
    unsigned long long s2[NP1], q2[NP1], k2[NP1];
    float s1, q1, k1;
    uint32_t cnt;
    __device__ __forceinline__ void clear()
    {
        cnt = 0u; s1 = 0.f; q1 = 0.f; k1 = 0.f;
#pragma unroll
        for(int k = 0; k < NP; k += 1) { s2[k] = pk2(0.f, 0.f); q2[k] = pk2(0.f, 0.f); k2[k] = pk2(0.f, 0.f); }
    }
    /* `first`: this is the half's first sample of the batch, which becomes the shift K */
    __device__ __forceinline__ void add(const unsigned long long (&r2)[NP1], float r1, bool first)
    {
        const unsigned long long m1 = pk2(-1.f, -1.f);
        if(first)
        {
#pragma unroll
            for(int k = 0; k < NP; k += 1) k2[k] = r2[k];
            k1 = r1;
        }
        cnt += 1u;
#pragma unroll
        for(int k = 0; k < NP; k += 1)
        {
            add2_acc(s2[k], r2[k]);
            const unsigned long long d = fma2(k2[k], m1, r2[k]);
            q2[k] = fma2(d, d, q2[k]);
        }
        if(NS & 1)
        {
            s1 += r1;
            const float d = r1 - k1;
            q1 = fmaf(d, d, q1);
        }
    }
};

/* film of one pixel held by a half warp: lane l16 owns wavelengths l16, l16+16, ...; when both halves work on the same
 * pixel each holds the partial film of its samples and merge_halves() combines them (Chan et al.) before the store */
template <int NS> struct PixelFilm
{
    float sum[NS], mean[NS], m2[NS], cnt;
    bool  lit;      /* some sample of this pixel was non-zero (uniform within the half warp) */
    __device__ __forceinline__ void clear()
    {
        cnt = 0.f; lit = false;
#pragma unroll
        for(int k = 0; k < NS; k += 1) { sum[k] = 0.f; mean[k] = 0.f; m2[k] = 0.f; }
    }
    /* The film is live for all samples of the pixel but idle while the warp traces (phase 1, the register-hungry phase): it is
     * parked in shared memory for the duration, word w of lane l at s[w*32 + l], which lowers the kernel's register need
     * and so raises the number of resident warps. */
    __device__ __forceinline__ void park(float *s) const
    {
        s[0] = cnt; s[DRT_WARP] = lit ? 1.f : 0.f;
#pragma unroll
        for(int k = 0; k < NS; k += 1) { s[(2 + k) * DRT_WARP] = sum[k]; s[(2 + NS + k) * DRT_WARP] = mean[k]; s[(2 + 2 * NS + k) * DRT_WARP] = m2[k]; }
    }
    __device__ __forceinline__ void unpark(const float *s)
    {
        cnt = s[0]; lit = s[DRT_WARP] != 0.f;
#pragma unroll
        for(int k = 0; k < NS; k += 1) { sum[k] = s[(2 + k) * DRT_WARP]; mean[k] = s[(2 + NS + k) * DRT_WARP]; m2[k] = s[(2 + 2 * NS + k) * DRT_WARP]; }
    }
    /* K6: film accumulation + Welford, daily_ray_trace.c:732-743 (filter weight is the constant 1, Q20) */
    __device__ __forceinline__ void add(const float (&c)[NS])
    {
        cnt += 1.f; lit = true;
        float inv = r_rcp_fast(cnt);
        float delta[NS], rest[NS];
        v_add<NS>(sum, sum, c);
        v_sub<NS>(delta, c, mean);
        v_fma_s<NS>(mean, inv, delta, mean);
        v_sub<NS>(rest, c, mean);
        v_fma<NS>(m2, delta, rest, m2);
    }
    /* k paths that contributed nothing, in one step: the pairwise update with a batch of k zeros (count k, mean 0, M2 0).
     * An exact no-op on a pixel that has seen no light yet. */
    __device__ __forceinline__ void add_zeros(uint32_t k)
    {
        const float n0 = cnt;
        cnt += (float)k;
        if(!lit || k == 0u) return;
        const float w = (float)k * r_rcp_fast(cnt);   /* k / (n0 + k) */
        const float s = n0 * w;
#pragma unroll
        for(int j = 0; j < NS; j += 1)
        {
            m2[j] = fmaf(mean[j] * mean[j], s, m2[j]);
            mean[j] = fmaf(-mean[j], w, mean[j]);
        }
    }
    /* nz paths that contributed nothing and the samples E * r of `bs`, in one pairwise update (Chan et al.): the batch has count
     * n = nz + bs.cnt, sum E S, mean E S / n and M2 = E^2 (Q + nz K^2 - n (S / n - K)^2) (the zeros are samples r = 0).  `e` = this
     * lane's E in the SpdIndex::light_pairs layout.  Without replayed samples this is add_zeros(nz). */
    __device__ __forceinline__ void add_batch(uint32_t nz, const BatchStats<NS> &bs, const float *e, uint32_t lane16)
    {
        if(bs.cnt == 0u) { add_zeros(nz); return; }
        const float nb = (float)(bs.cnt + nz), n0 = cnt, zf = (float)nz;
        cnt += nb; lit = true;
        const float inv_nb = r_rcp_fast(nb);
        const float w = nb * r_rcp_fast(cnt);   /* n / (n0 + n) */
        const float s = n0 * w;
#pragma unroll
        for(int j = 0; j < NS; j += 1)
        {
            float S, Q, K, t;
            if(j + 1 < NS || !(NS & 1))
            {
                if(j & 1) { upk2(bs.s2[j >> 1], t, S); upk2(bs.q2[j >> 1], t, Q); upk2(bs.k2[j >> 1], t, K); }
                else      { upk2(bs.s2[j >> 1], S, t); upk2(bs.q2[j >> 1], Q, t); upk2(bs.k2[j >> 1], K, t); }
            }
            else { S = bs.s1; Q = bs.q1; K = bs.k1; }
            const float E = e[2 * ((j >> 1) * DRT_HALF + lane16) + (j & 1)];
            const float m = S * inv_nb, dk = m - K;
            const float m2b = fmaxf(fmaf(-nb * dk, dk, fmaf(zf * K, K, Q)), 0.f);   /* the batch's M2 over r */
            const float delta = fmaf(E, m, -mean[j]);
            sum[j] = fmaf(E, S, sum[j]);
            m2[j] = fmaf(delta * delta, s, fmaf(E * E, m2b, m2[j]));
            mean[j] = fmaf(delta, w, mean[j]);
        }
    }
    /* this half <- this half (+) the other half: count, mean, M2 by the pairwise update, sums added */
    __device__ __forceinline__ void merge_halves()
    {
        float nb = __shfl_xor_sync(0xffffffffu, cnt, DRT_HALF);
        bool  lb = __shfl_xor_sync(0xffffffffu, (int)lit, DRT_HALF) != 0;
        float nab = cnt + nb;
        float wb = (nab > 0.f) ? nb / nab : 0.f;
#pragma unroll
        for(int k = 0; k < NS; k += 1)
        {
            float mb = __shfl_xor_sync(0xffffffffu, mean[k], DRT_HALF);
            float vb = __shfl_xor_sync(0xffffffffu, m2[k], DRT_HALF);
            float sb = __shfl_xor_sync(0xffffffffu, sum[k], DRT_HALF);
            float delta = mb - mean[k];
            m2[k] = m2[k] + vb + delta * delta * cnt * wb;
            mean[k] = fmaf(delta, wb, mean[k]);
            sum[k] += sb;
        }
        cnt = nab; lit = lit || lb;
    }
};

/* Adaptive sampling's stopping rule, taken at the end of a batch of a pixel (render_kernel_adaptive).  With n the pixel's count, w_l
 * the luminance weights cmf_y * ref_white of the .bmp conversion (RenderLaunch::luminance_w), Y = sum_l w_l mean_l and
 * err = sum_l w_l sqrt(M2_l / (n (n - 1))) -- an upper bound on the standard error of Y, since the sd of a sum is at most the sum of the
 * sds -- the pixel stops when n >= min_samples and err <= rel_error * Y.  A NaN never stops a pixel, nor does Y = 0 with noise; a
 * film without variance (all samples zero, or all equal) stops as soon as n >= min_samples.
 * The two half warps' partial films are merged into temporaries with merge_halves' arithmetic and stay as they are.  The halves'
 * merged values can differ by rounding, so lane 0's decision is the warp's.  The weights are read from global memory (L1) here
 * only: kept in registers through the batch loop they would cost the plastic-only kernel its register budget. */
template <int NS>
static __device__ __forceinline__ bool pixel_converged(const PixelFilm<NS> &f, const RenderLaunch &L, uint32_t n, uint32_t lane16)
{
    const float nb = __shfl_xor_sync(0xffffffffu, f.cnt, DRT_HALF);
    const float nab = f.cnt + nb;
    const float wb = (nab > 0.f) ? nb / nab : 0.f;
    const float inv = 1.f / (nab * (nab - 1.f));
    float y = 0.f, e = 0.f;
#pragma unroll
    for(int k = 0; k < NS; k += 1)
    {
        const float mb = __shfl_xor_sync(0xffffffffu, f.mean[k], DRT_HALF);
        const float vb = __shfl_xor_sync(0xffffffffu, f.m2[k], DRT_HALF);
        const float delta = mb - f.mean[k];
        const float m2 = f.m2[k] + vb + delta * delta * f.cnt * wb;
        const float mean = fmaf(delta, wb, f.mean[k]);
        const uint32_t wl = lane16 + k * DRT_HALF;
        if(wl < n)
        {
            const float w = __ldg(L.luminance_w + wl);
            y = fmaf(w, mean, y);
            e = fmaf(w, sqrtf(fmaxf(m2, 0.f) * inv), e);
        }
    }
#pragma unroll
    for(int o = DRT_HALF / 2; o > 0; o >>= 1) { y += __shfl_xor_sync(0xffffffffu, y, o); e += __shfl_xor_sync(0xffffffffu, e, o); }
    const bool stop = nab >= (float)L.min_samples && e <= L.rel_error * y;
    return __shfl_sync(0xffffffffu, stop ? 1 : 0, 0) != 0;
}

/* film <-> HBM, once per pixel per render: out of line (cold relative to the per-sample code) and by value.
 * Only the lower half warp (lanes 0-15) touches memory. */
template <int NS>
static __device__ __noinline__ PixelFilm<NS> film_load(FilmPtrs film, uint32_t gpix, uint32_t n, uint32_t lane)
{
    PixelFilm<NS> f;
    f.clear();
    if(lane >= DRT_HALF) return f;
    f.cnt = film.filter[gpix]; f.lit = true;
#pragma unroll
    for(int k = 0; k < NS; k += 1)
    {
        uint32_t wl = lane + k * DRT_HALF;
        size_t at = (size_t)gpix * n + wl;
        f.sum[k] = (wl < n) ? film.sum[at] : 0.f; f.mean[k] = (wl < n) ? film.mean[at] : 0.f; f.m2[k] = (wl < n) ? film.m2[at] : 0.f;
    }
    return f;
}

template <int NS>
static __device__ __noinline__ void film_store(FilmPtrs film, uint32_t gpix, uint32_t n, uint32_t lane, PixelFilm<NS> f)
{
    if(lane >= DRT_HALF) return;
#pragma unroll
    for(int k = 0; k < NS; k += 1)
    {
        uint32_t wl = lane + k * DRT_HALF;
        if(wl < n)
        {
            size_t at = (size_t)gpix * n + wl;
            film.sum[at] = f.sum[k]; film.mean[at] = f.mean[k]; film.m2[at] = f.m2[k];
        }
    }
    if(lane == 0) film.filter[gpix] = f.cnt;
}

/* ------------------------------------------------------------------ the kernel */

/* Diagnostics (drt_cuda_sample_paths / drt_cuda_debug_records): per-path spectrum and raw record to global memory, by the 16
 * lanes of a half warp.  Out of line: never on the path of a film render.  `e` (compact records, whose replay leaves out the light's
 * emission): the SpdIndex::light_pairs row the spectrum c is multiplied by, else null. */
template <int NS>
static __device__ __noinline__ void dump_path(float *record_dump, float *path_dump, uint32_t path_words, const float *rec_slot, const float *c,
                                       const float *e, size_t path_index, uint32_t n, uint32_t lane16)
{
    if(record_dump)
        for(uint32_t wd = lane16; wd < path_words; wd += DRT_HALF) record_dump[path_index * path_words + wd] = rec_slot[wd];
    if(path_dump)
#pragma unroll
        for(int k = 0; k < NS; k += 1)
        {
            uint32_t wl = lane16 + k * DRT_HALF;
            const float ek = e ? e[2 * ((k >> 1) * DRT_HALF + lane16) + (k & 1)] : 1.f;
            if(wl < n) path_dump[path_index * n + wl] = c ? ek * c[k] : 0.f;
        }
}

/* ALLFAST: every surface material of the scene is a two-lobe plastic and there is exactly one light (decided by the
 * host at scene upload: all shipped Cornell boxes except the gold/glass balls of cornell_plane_light).  The kernel then
 * contains neither the general lobe evaluators nor the general shader. */
/* Phase clocks, diagnostic builds only (tools/build_variant.sh NAME -DDRT_PHASE_CLOCKS; tools/phase_split.py reads them through
 * drt_cuda_phase_clocks).  Each warp's timeline after the scene staging is cut at the boundaries of a batch, and the SM-clock cycles
 * since the previous cut go to the part that just ended: TRACE = phase 1 (film parking, the gate in front of it, trace_path), BOOK =
 * the batch bookkeeping (histogram, sort, zero counts, film unpark, add_batch, the phase-2 gate), REPLAY = phase 2 (the replay of the
 * records and BatchStats::add), OTHER = task fetch, film load / store, culled pixels.  Lane 0 adds each piece to a shared-memory
 * counter.  Without the flag the macro is empty and the kernels compile to the same code. */
#define DRT_PHASE_TRACE  0
#define DRT_PHASE_BOOK   1
#define DRT_PHASE_REPLAY 2
#define DRT_PHASE_OTHER  3
#ifdef DRT_PHASE_CLOCKS
#define DRT_PHASE_CUT(k) do { uint32_t t_; asm volatile("mov.u32 %0, %%clock;" : "=r"(t_) :: "memory"); \
                              if(lane == 0) atomicAdd(&s_phase[k], (unsigned long long)(t_ - phase_t)); phase_t = t_; } while(0)
#else
#define DRT_PHASE_CUT(k) do {} while(0)
#endif
/* PAIRED: one pixel per task with all its samples (spp >= 32) against 32/spp whole pixels per task; see the task loop. */
#define DRT_RENDER_BOUNDS(MODE) __launch_bounds__(DRT_RENDER_SHAPE[MODE].warps * DRT_WARP, DRT_RENDER_SHAPE[MODE].min_ctas)
template <typename R, int NS, int MODE, bool PAIRED, bool DEEP>
__global__ void DRT_RENDER_BOUNDS(MODE) render_kernel(const RenderLaunch L)
{
    constexpr bool ADAPTIVE = false;
#include "drt_render_body.cuh"
}

/* Adaptive sampling (drt_cuda_render_*_adaptive): f32 geometry, one pixel per task.  A pixel stops at the end of the first batch after
 * which its film meets the luminance error bound (pixel_converged), or when the launch's samples run out. */
template <typename R, int NS, int MODE, bool DEEP>
__global__ void DRT_RENDER_BOUNDS(MODE) render_kernel_adaptive(const RenderLaunch L)
{
    constexpr bool PAIRED = true, ADAPTIVE = true;
#include "drt_render_body.cuh"
}

} // namespace drt

/* ------------------------------------------------------------------ launch helper of the instantiating translation units */

/* DEEP = the instantiation whose records overflow to global memory (RenderLaunch::deep); the instantiating translation units
 * (drt_kernels_*.cu) build the shallow and the deep kernels of a mode separately so that the hot ones keep their register budget. */
template <typename K>
static cudaError_t drt_launch_one(K kernel, const RenderLaunch &L, int grid, int warps, size_t smem, cudaStream_t stream)
{
    cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if(e != cudaSuccess) return e;
    e = cudaFuncSetAttribute(kernel, cudaFuncAttributePreferredSharedMemoryCarveout, 100);
    if(e != cudaSuccess) return e;
    kernel<<<grid, warps * DRT_WARP, smem, stream>>>(L);
    return cudaGetLastError();
}

template <typename R, int MODE, bool PAIRED, bool DEEP>
static cudaError_t drt_launch_render_ns(const RenderLaunch &L, int nslots, int grid, int warps, size_t smem, cudaStream_t stream)
{
    switch(nslots)   /* wavelength slots per lane of a half warp: N <= 32, 48, 80, 128 */
    {
        case 2: return drt_launch_one(drt::render_kernel<R, 2, MODE, PAIRED, DEEP>, L, grid, warps, smem, stream);
        case 3: return drt_launch_one(drt::render_kernel<R, 3, MODE, PAIRED, DEEP>, L, grid, warps, smem, stream);
        case 5: return drt_launch_one(drt::render_kernel<R, 5, MODE, PAIRED, DEEP>, L, grid, warps, smem, stream);
        default: return drt_launch_one(drt::render_kernel<R, 8, MODE, PAIRED, DEEP>, L, grid, warps, smem, stream);
    }
}

template <int MODE, bool DEEP>
static cudaError_t drt_launch_adaptive_ns(const RenderLaunch &L, int nslots, int grid, int warps, size_t smem, cudaStream_t stream)
{
    switch(nslots)
    {
        case 2: return drt_launch_one(drt::render_kernel_adaptive<float, 2, MODE, DEEP>, L, grid, warps, smem, stream);
        case 3: return drt_launch_one(drt::render_kernel_adaptive<float, 3, MODE, DEEP>, L, grid, warps, smem, stream);
        case 5: return drt_launch_one(drt::render_kernel_adaptive<float, 5, MODE, DEEP>, L, grid, warps, smem, stream);
        default: return drt_launch_one(drt::render_kernel_adaptive<float, 8, MODE, DEEP>, L, grid, warps, smem, stream);
    }
}

/* one translation unit = one mode of the adaptive kernel (f32 geometry, one pixel per task), shallow and deep */
#define DRT_DEFINE_ADAPTIVE_LAUNCHERS(NAME, MODE) \
    cudaError_t NAME(const RenderLaunch &L, int nslots, int grid, int warps, size_t smem, cudaStream_t stream) \
    { \
        return drt_launch_adaptive_ns<MODE, false>(L, nslots, grid, warps, smem, stream); \
    } \
    cudaError_t NAME##_deep(const RenderLaunch &L, int nslots, int grid, int warps, size_t smem, cudaStream_t stream) \
    { \
        return drt_launch_adaptive_ns<MODE, true>(L, nslots, grid, warps, smem, stream); \
    }

/* one translation unit = one (arithmetic type, mode, deep) combination, both task shapes */
#define DRT_DEFINE_LAUNCHER(NAME, R, MODE, DEEP) \
    cudaError_t NAME(const RenderLaunch &L, bool paired, int nslots, int grid, int warps, size_t smem, cudaStream_t stream) \
    { \
        return paired ? drt_launch_render_ns<R, MODE, true, DEEP>(L, nslots, grid, warps, smem, stream) \
                      : drt_launch_render_ns<R, MODE, false, DEEP>(L, nslots, grid, warps, smem, stream); \
    }
