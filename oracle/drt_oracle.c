/*
 * oracle/drt_oracle.c -- TEST INFRASTRUCTURE: CPU restatement of the reference's render hot path.
 *
 * Plain C, f64, single-threaded, over the flattened drt_scene / drt_camera of include/drt_scene.h and the
 * per-path random streams of include/drt_rng.h.  It exists to CHECK the CUDA path (tests/, __graft_entry__.smoke,
 * bench.py's cpu_baseline leg); nothing in the product may call it.  Every function names the reference lines
 * it follows; operation order and the long-double PI of types.h:1 are kept so that results are bit-identical
 * to the reference compiled in oracle/_ref (pinned by tests/test_oracle_vs_ref.py and tests/golden/).
 * Quirk numbers (Qn) refer to SURVEY.md Appendix A.
 */
#include <math.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>
#include "drt_scene.h"
#include "drt_rng.h"

#define PI_L 3.1415926535897932385L   /* types.h:1 */

typedef struct { double x, y, z; } v3;
typedef struct { v3 col[3]; } m3;      /* geometry.h:32-35 */

typedef struct
{
    uint64_t paths, closest_rays, shadow_rays, shaded_bounces, rng_draws;
    uint64_t terminated_at_depth[8];   /* paths that left the loop by escape/emitter at depth d (d>=7 pooled) */
    uint64_t reached_depth_cap;
} drt_oracle_counters;

typedef struct
{
    const drt_scene  *scene;
    const drt_camera *cam;
    int               n;
    drt_rng_stream    rng;
    drt_oracle_counters *count;
} ctx;

/* scene_point, daily_ray_trace.h:113-125 */
typedef struct
{
    v3 position, normal, out;
    double on_dot, trans_wl;
    const drt_material *surface_material, *incident_material, *transmit_material;
} hit_point;

/* ---- geometry.c:6-106 ---- */
static v3 v3_make(const double *p) { v3 r = { p[0], p[1], p[2] }; return r; }
static int v3_equal(v3 a, v3 b) { return a.x == b.x && a.y == b.y && a.z == b.z; }
static v3 v3_sum(v3 a, v3 b) { v3 r = { a.x + b.x, a.y + b.y, a.z + b.z }; return r; }
static v3 v3_sub(v3 a, v3 b) { v3 r = { a.x - b.x, a.y - b.y, a.z - b.z }; return r; }
static double v3_dot(v3 a, v3 b) { return a.x * b.x + a.y * b.y + a.z * b.z; }
static v3 v3_cross(v3 a, v3 b) { v3 n = { a.y * b.z - a.z * b.y, a.z * b.x - a.x * b.z, a.x * b.y - a.y * b.x }; return n; }
static v3 v3_scale(v3 v, double f) { v3 r = { f * v.x, f * v.y, f * v.z }; return r; }
static v3 v3_div(v3 v, double f) { v3 r = { v.x / f, v.y / f, v.z / f }; return r; }
static double v3_length(v3 v) { return sqrt(v3_dot(v, v)); }
static v3 v3_normalise(v3 v) { return v3_div(v, v3_length(v)); }
static v3 v3_reverse(v3 v) { v3 r = { -v.x, -v.y, -v.z }; return r; }

static v3 v3_reflect(v3 v, v3 n)   /* geometry.c:85-90 */
{
    double f = 2.0 * v3_dot(v, n);
    return v3_sub(v, v3_scale(n, f));
}

static v3 v3_transmit(v3 v, v3 n, double ir, double tr)   /* geometry.c:92-106; NaN under total internal reflection */
{
    double vn = v3_dot(v, n);
    double rel = ir / tr;
    v3 m = v3_scale(n, vn);
    v = v3_sub(m, v);
    v3 perpend = v3_reverse(v3_scale(v, rel));
    double pd = -sqrt(1.0 - v3_dot(perpend, perpend));
    v3 parallel = v3_scale(n, pd);
    return v3_sum(perpend, parallel);
}

static double ray_sphere(v3 o, v3 d, v3 c, double r)   /* line_sphere_intersection, geometry.c:123-146 */
{
    v3 co = v3_sub(o, c);
    double a = 1.0;
    double b = -2.0 * v3_dot(co, d);
    double cc = v3_dot(co, co) - r * r;
    double disc = b * b - 4.0 * a * cc;
    if(disc < 0.0) return INFINITY;
    double sq = sqrt(disc);
    double a2 = 2.0 * a;
    double s0 = (b + sq) / a2;
    double s1 = (b - sq) / a2;
    if(s0 < 0.0 && s1 < 0.0) return INFINITY;
    else if(s0 >= 0.0 && s1 < 0.0) return s0;
    else if(s1 >= 0.0 && s0 < 0.0) return s1;
    else if(s0 <= s1) return s0;
    else return s1;
}

static double ray_plane(v3 o, v3 d, v3 p, v3 n, v3 u, v3 v)   /* line_plane_intersection, geometry.c:157-182 */
{
    if(v3_dot(d, n) == 0.0) return INFINITY;
    v3 op = v3_sub(p, o);
    double l = v3_dot(op, n) / v3_dot(d, n);
    v3 i = v3_sum(o, v3_scale(d, l));
    v3 j = v3_sub(i, p);
    double ul = v3_length(u), vl = v3_length(v);
    v3 un = v3_normalise(u), vn = v3_normalise(v);
    double ju = v3_dot(j, un), jv = v3_dot(j, vn);
    if(l >= 0.0 && 0.0 <= ju && ju <= ul && 0.0 <= jv && jv <= vl) return l;
    return INFINITY;
}

static v3 m3_row(m3 m, int r)
{
    const double *c0 = &m.col[0].x, *c1 = &m.col[1].x, *c2 = &m.col[2].x;
    v3 v = { c0[r], c1[r], c2[r] };
    return v;
}
static v3 m3_apply(m3 m, v3 v) { v3 w = { v3_dot(m3_row(m, 0), v), v3_dot(m3_row(m, 1), v), v3_dot(m3_row(m, 2), v) }; return w; }

static m3 rotation_between(v3 v, v3 w)   /* find_rotation_between_vectors, geometry.c:263-295 (Q14: -I when antiparallel) */
{
    v3 n = v3_cross(v, w);
    double c = v3_dot(v, w);
    m3 r = {{{1.0, 0.0, 0.0}, {0.0, 1.0, 0.0}, {0.0, 0.0, 1.0}}};
    if(v3_dot(n, n) == 0.0 && c <= 0.0)
    {
        r.col[0].x = -1.0; r.col[1].y = -1.0; r.col[2].z = -1.0;
        return r;
    }
    m3 m = {{{0.0, n.z, -n.y}, {-n.z, 0.0, n.x}, {n.y, -n.x, 0.0}}};
    m3 mm;
    for(int i = 0; i < 3; i += 1)
    {
        v3 row = m3_row(m, i);
        double *dst = &mm.col[i].x;      /* mat3x3_mul stores (row i).(column j) at columns[i].xyz[j], geometry.c:243-256 */
        for(int j = 0; j < 3; j += 1) dst[j] = v3_dot(row, m.col[j]);
    }
    double f = (1.0 / (1.0 + c));
    m3 id = {{{1.0, 0.0, 0.0}, {0.0, 1.0, 0.0}, {0.0, 0.0, 1.0}}};
    for(int i = 0; i < 3; i += 1) r.col[i] = v3_sum(v3_sum(id.col[i], m.col[i]), v3_scale(mm.col[i], f));
    return r;
}

/* ---- rng.c:2-51 on the per-path stream ---- */
static double rng(ctx *c) { c->count->rng_draws += 1; return drt_rng_f64(&c->rng); }

static v3 uniform_sample_sphere(ctx *c)   /* rng.c:14-23: z = u >= 0, i.e. a hemisphere */
{
    double u = rng(c);
    double v = rng(c);
    double r = sqrt(1.0 - u * u);
    double t = 2.0 * PI_L * v;
    v3 s = { r * cos(t), r * sin(t), u };
    return s;
}

static v3 uniform_sample_disc(ctx *c)   /* rng.c:25-51: concentric map with signed radius (Q16) */
{
    v3 v = { 0.0, 0.0, 0.0 };
    double rx = rng(c);
    double ry = rng(c);
    double ox = 2.0 * rx - 1.0;
    double oy = 2.0 * ry - 1.0;
    if(ox == 0.0 && oy == 0.0) return v;
    double r, t;
    if(fabs(ox) > fabs(oy)) { r = ox; t = (PI_L / 4.0) * (oy / ox); }
    else                    { r = oy; t = (PI_L / 2.0) - (PI_L / 4.0) * (ox / oy); }
    v.x = r * cos(t);
    v.y = r * sin(t);
    return v;
}

/* ---- spectrum.c:150-243 ---- */
static double value_at_wl(const ctx *c, const double *spd, double wl)   /* spectrum.c:150-162 */
{
    uint32_t i0 = (uint32_t)((wl - c->scene->min_wl) / c->scene->wl_interval);
    uint32_t i1 = i0 + 1;
    double w0 = c->scene->min_wl + i0 * c->scene->wl_interval;
    double w1 = c->scene->min_wl + i1 * c->scene->wl_interval;
    double s0 = spd[i0], s1 = spd[i1];
    return s0 + ((wl - w0) * ((s1 - s0) / (w1 - w0)));
}

/* ---- bdsf.c:3-101 helpers ---- */
static double ggx(v3 sn, v3 mn, double r)   /* bdsf.c:3-20 */
{
    double d = v3_dot(sn, mn);
    double r2 = r * r;
    if(d <= 0.0) return 0.0;
    double d2 = d * d;
    double d4 = d2 * d2;
    double tan_sq = (1.0 / d2) - 1.0;
    return r2 / (PI_L * d4 * (r2 + tan_sq) * (r2 + tan_sq));
}

static double ggx_att(v3 v, v3 sn, v3 mn, double r)   /* bdsf.c:22-42: D * G1(out) only */
{
    double att;
    double g = ggx(sn, mn, r);
    double v_mn = v3_dot(v, mn);
    double v_sn = v3_dot(v, sn);
    double quot = fabs(v_mn / v_sn);
    double r2 = r * r;
    if(quot <= 0.0) att = 0.0;
    else
    {
        double tan_sq = (1.0 / (v_sn * v_sn)) - 1.0;
        att = 2.0 / (1.0 + sqrt(1.0 + r2 * tan_sq));
    }
    return g * att;
}

static void dielectric_reflectance(const ctx *c, double *out, const double *ir, const double *tr, double inc_cos)   /* bdsf.c:44-66 */
{
    double inc_sin_sq = 1.0 - inc_cos * inc_cos;
    for(int i = 0; i < c->n; i += 1)
    {
        double rel = ir[i] / tr[i];
        double ts_sin_sq = rel * rel * inc_sin_sq;
        if(ts_sin_sq >= 1.0) { out[i] = 1.0; continue; }
        double ts_cos = sqrt(1.0 - ts_sin_sq * ts_sin_sq);   /* Q9: sin^2 is squared again */
        double tr_on = tr[i] * inc_cos, tr_ts = tr[i] * ts_cos;
        double ir_on = ir[i] * inc_cos, ir_ts = ir[i] * ts_cos;
        double par = (tr_on - ir_ts) / (tr_on + ir_ts);
        double per = (ir_on - tr_ts) / (ir_on + tr_ts);
        par *= par;
        per *= per;
        out[i] = 0.5 * (par + per);
    }
}

static void conductor_reflectance(const ctx *c, double *out, const double *ir, const double *tr, const double *te, double inc_cos)   /* bdsf.c:78-101 */
{
    double cos_sq = inc_cos * inc_cos;
    double sin_sq = 1.0 - cos_sq;
    for(int i = 0; i < c->n; i += 1)
    {
        double eta = tr[i] / ir[i];
        double kap = te[i] / ir[i];
        double eta_sq = eta * eta;
        double kap_sq = kap * kap;
        double r = eta_sq - kap_sq - sin_sq;
        double apb_sq = sqrt(r * r + 4.0 * eta_sq * kap_sq);
        double a = sqrt(0.5 * (apb_sq + r));
        double s = apb_sq + cos_sq;
        double t = 2.0 * a * inc_cos;
        double u = cos_sq * apb_sq + sin_sq * sin_sq;
        double v = t * sin_sq;
        double par = (s - t) / (s + t);
        double per = par * (u - v) / (u + v);
        out[i] = 0.5 * (par + per);
    }
}

/* ---- the seven lobes, bdsf.c:105-186; `res` is the shared scratch of bdsf() (Q7) ---- */
static void eval_lobe(const ctx *c, int lobe, double *res, const hit_point *p, v3 in)
{
    int n = c->n;
    const drt_material *sm = p->surface_material;
    switch(lobe)
    {
        case DRT_LOBE_BP_DIFFUSE:   /* :105-109 */
        {
            double inv_pi = 1.0 / PI_L;
            double w = fabs(v3_dot(p->normal, in));
            for(int i = 0; i < n; i += 1) res[i] = sm->spd[DRT_SPD_DIFFUSE][i] * inv_pi;
            for(int i = 0; i < n; i += 1) res[i] = res[i] * w;
            break;
        }
        case DRT_LOBE_BP_GLOSSY:   /* :111-119 */
        {
            v3 bis = v3_normalise(v3_sum(p->out, in));
            double nb = v3_dot(p->normal, bis);
            double coef = pow((0.0 > nb) ? 0.0 : nb, sm->shininess);
            double w = fabs(v3_dot(p->normal, in));
            for(int i = 0; i < n; i += 1) res[i] = sm->spd[DRT_SPD_GLOSSY][i] * coef;
            for(int i = 0; i < n; i += 1) res[i] = res[i] * w;
            break;
        }
        case DRT_LOBE_MIRROR:   /* :121-132: the one specular lobe that zeroes on mismatch */
        {
            if(v3_equal(in, v3_reflect(v3_reverse(p->out), p->normal))) memcpy(res, sm->spd[DRT_SPD_MIRROR], sizeof(double) * (size_t)n);
            else memset(res, 0, sizeof(double) * (size_t)n);
            break;
        }
        case DRT_LOBE_FS_CONDUCTOR:   /* :134-146: no write on mismatch */
        {
            if(v3_equal(in, v3_reflect(v3_reverse(p->out), p->normal)))
                conductor_reflectance(c, res, p->incident_material->spd[DRT_SPD_REFRACT], p->transmit_material->spd[DRT_SPD_REFRACT],
                                      p->transmit_material->spd[DRT_SPD_EXTINCT], p->on_dot);
            break;
        }
        case DRT_LOBE_FS_DIELECTRIC_REFLECTANCE:   /* :148-159: no write on mismatch */
        {
            if(v3_equal(in, v3_reflect(v3_reverse(p->out), p->normal)))
                dielectric_reflectance(c, res, p->incident_material->spd[DRT_SPD_REFRACT], p->transmit_material->spd[DRT_SPD_REFRACT], p->on_dot);
            break;
        }
        case DRT_LOBE_FS_DIELECTRIC_TRANSMITTANCE:   /* :161-172: no write on mismatch */
        {
            const double *ir_spd = p->incident_material->spd[DRT_SPD_REFRACT], *tr_spd = p->transmit_material->spd[DRT_SPD_REFRACT];
            double ir = value_at_wl(c, ir_spd, p->trans_wl);
            double tr = value_at_wl(c, tr_spd, p->trans_wl);
            if(v3_equal(in, v3_transmit(v3_reverse(p->out), p->normal, ir, tr)))
            {
                dielectric_reflectance(c, res, ir_spd, tr_spd, p->on_dot);
                for(int i = 0; i < n; i += 1) res[i] = 1.0 - res[i];
            }
            break;
        }
        case DRT_LOBE_CT_CONDUCTOR:   /* :174-186 */
        {
            v3 mn = v3_normalise(v3_sum(p->out, in));
            double mn_dot = fabs(v3_dot(p->normal, mn));
            conductor_reflectance(c, res, p->incident_material->spd[DRT_SPD_REFRACT], p->transmit_material->spd[DRT_SPD_REFRACT],
                                  p->transmit_material->spd[DRT_SPD_EXTINCT], mn_dot);
            double coef = ggx_att(p->out, p->normal, mn, sm->roughness) * (1.0 / (4.0 * p->on_dot));
            for(int i = 0; i < n; i += 1) res[i] = res[i] * coef;
            break;
        }
        default: break;
    }
}

static void bdsf(const ctx *c, double *reflectance, const hit_point *p, v3 in)   /* daily_ray_trace.c:215-229 */
{
    double res[DRT_MAX_WAVELENGTHS];
    int n = c->n;
    memset(res, 0, sizeof(double) * (size_t)n);
    memset(reflectance, 0, sizeof(double) * (size_t)n);
    const drt_material *m = p->surface_material;
    for(int k = 0; k < m->num_lobes; k += 1)
    {
        eval_lobe(c, m->lobes[k], res, p, in);
        for(int i = 0; i < n; i += 1) reflectance[i] = reflectance[i] + res[i];
    }
}

/* ---- the six direction samplers, bdsf.c:191-292; *inv_pdf is the RECIPROCAL pdf (Q12) ---- */
static void sample_direction(ctx *c, int which, v3 *v, double *inv_pdf, const hit_point *p)
{
    const v3 plus_z = { 0.0, 0.0, 1.0 };
    switch(which)
    {
        case DRT_DIR_UNIFORM_HEMISPHERE:   /* :191-198 */
        {
            *v = uniform_sample_sphere(c);
            m3 r = rotation_between(plus_z, p->normal);
            *v = m3_apply(r, *v);
            *inv_pdf = (2.0 * PI_L);
            break;
        }
        case DRT_DIR_COS_WEIGHTED_HEMISPHERE:   /* :200-213 */
        {
            v3 q;
            for(;;)
            {
                q = uniform_sample_disc(c);
                if(v3_dot(q, q) < 1.0) break;
            }
            q.z = sqrt(1.0 - v3_dot(q, q));
            m3 r = rotation_between(plus_z, p->normal);
            *v = m3_apply(r, q);
            *inv_pdf = PI_L / v3_dot(p->normal, *v);
            break;
        }
        case DRT_DIR_SPECULAR:   /* :215-220 */
        {
            *v = v3_reflect(v3_reverse(p->out), p->normal);
            *inv_pdf = 1.0;
            break;
        }
        case DRT_DIR_TRANSMIT:   /* :222-234 */
        {
            double ir = value_at_wl(c, p->incident_material->spd[DRT_SPD_REFRACT], p->trans_wl);
            double tr = value_at_wl(c, p->transmit_material->spd[DRT_SPD_REFRACT], p->trans_wl);
            *v = v3_transmit(v3_reverse(p->out), p->normal, ir, tr);
            *inv_pdf = 1.0;
            break;
        }
        case DRT_DIR_REFLECT_OR_TRANSMIT:   /* :236-259 */
        {
            double refl[DRT_MAX_WAVELENGTHS];
            const double *ir_spd = p->incident_material->spd[DRT_SPD_REFRACT], *tr_spd = p->transmit_material->spd[DRT_SPD_REFRACT];
            dielectric_reflectance(c, refl, ir_spd, tr_spd, p->on_dot);
            double rd = value_at_wl(c, refl, p->trans_wl);
            double ir = value_at_wl(c, ir_spd, p->trans_wl);
            double tr = value_at_wl(c, tr_spd, p->trans_wl);
            double f = rng(c);
            v3 w = v3_reverse(p->out);
            if(f < rd) { *v = v3_reflect(w, p->normal); *inv_pdf = 1.0 / rd; }
            else       { *v = v3_transmit(w, p->normal, ir, tr); *inv_pdf = 1.0 / (1.0 - rd); }
            break;
        }
        case DRT_DIR_CT:   /* :261-292 */
        {
            double rough = p->surface_material->roughness;
            do
            {
                double f = rng(c);
                double g = rng(c);
                double phi = 2.0 * PI_L * g;
                double tan_mn = (rough * sqrt(f)) / sqrt(1.0 - f);
                double cos_mn = 1.0 / sqrt(1.0 + tan_mn * tan_mn);
                double sin_mn = sqrt(1.0 - cos_mn * cos_mn);
                v3 mn = { sin_mn * cos(phi), sin_mn * sin(phi), cos_mn };
                m3 r = rotation_between(plus_z, p->normal);
                mn = m3_apply(r, mn);
                double sn_mn = v3_dot(p->normal, mn);
                if(sn_mn < 0.0) { mn = v3_reverse(mn); sn_mn = -sn_mn; }
                double o_mn = v3_dot(p->out, mn);
                *v = v3_reflect(v3_reverse(p->out), mn);
                double d = ggx(p->normal, mn, rough) * sn_mn;
                *inv_pdf = ((4.0 * o_mn) / d);
            }
            while(v3_dot(*v, p->normal) < 0.0);
            break;
        }
        default: break;
    }
}

/* ---- daily_ray_trace.c:238-403 ---- */
static double intersect_surface(const drt_surface *s, v3 o, v3 d)
{
    if(s->type == DRT_GEO_SPHERE) return ray_sphere(o, d, v3_make(s->position), s->radius);
    return ray_plane(o, d, v3_make(s->position), v3_make(s->normal), v3_make(s->u), v3_make(s->v));
}

static int mutually_visible(ctx *c, v3 p0, v3 p1)   /* points_mutually_visible, :238-270 */
{
    c->count->shadow_rays += 1;
    v3 dir = v3_normalise(v3_sub(p1, p0));
    v3 origin = v3_sum(p0, v3_scale(dir, DRT_RAY_FUDGE));
    double vis_dist = v3_length(v3_sub(p1, origin)) - DRT_RAY_FUDGE;
    for(int i = 0; i < c->scene->num_surfaces; i += 1)
    {
        const drt_surface *s = &c->scene->surfaces[i];
        if(s->type == DRT_GEO_POINT) continue;
        if(s->type != DRT_GEO_SPHERE && s->type != DRT_GEO_PLANE) continue;
        if(intersect_surface(s, origin, dir) < vis_dist) return 0;
    }
    return 1;
}

static void find_intersection(ctx *c, hit_point *hit, v3 origin, v3 dir)   /* find_ray_intersection, :334-403 */
{
    const drt_scene *sc = c->scene;
    c->count->closest_rays += 1;
    double min_dist = INFINITY;
    int found = -1;
    origin = v3_sum(origin, v3_scale(dir, DRT_RAY_FUDGE));   /* Q2 */
    for(int i = 0; i < sc->num_surfaces; i += 1)
    {
        const drt_surface *s = &sc->surfaces[i];
        if(s->type != DRT_GEO_SPHERE && s->type != DRT_GEO_PLANE) continue;
        double dist = intersect_surface(s, origin, dir);
        if(dist < min_dist) { min_dist = dist; found = i; }   /* strict <: lowest index wins ties (Q21) */
    }
    if(found < 0) { hit->surface_material = &sc->materials[sc->escape_material]; return; }
    const drt_surface *s = &sc->surfaces[found];
    const drt_material *sm = &sc->materials[s->material], *base = &sc->materials[sc->base_material];
    hit->position = v3_sum(origin, v3_scale(dir, min_dist));
    hit->normal = (s->type == DRT_GEO_SPHERE) ? v3_normalise(v3_sub(hit->position, v3_make(s->position))) : v3_make(s->normal);
    hit->trans_wl = DRT_TRANS_WL;
    hit->out = v3_reverse(dir);
    hit->on_dot = v3_dot(hit->normal, hit->out);
    hit->transmit_material = sm;
    hit->incident_material = base;
    if(hit->on_dot < 0.0)
    {
        if(s->type != DRT_GEO_PLANE) { hit->transmit_material = base; hit->incident_material = sm; }   /* Q11 */
        hit->normal = v3_reverse(hit->normal);
        hit->on_dot = v3_dot(hit->normal, hit->out);
    }
    hit->surface_material = sm;
}

static void direct_light(ctx *c, double *contribution, const hit_point *hit)   /* direct_light_contribution, :272-332 */
{
    const drt_scene *sc = c->scene;
    int n = c->n;
    double refl[DRT_MAX_WAVELENGTHS];
    memset(refl, 0, sizeof(double) * (size_t)n);
    memset(contribution, 0, sizeof(double) * (size_t)n);
    for(int i = 0; i < sc->num_surfaces; i += 1)
    {
        const drt_surface *ls = &sc->surfaces[i];
        const drt_material *lm = &sc->materials[ls->material];
        if(!lm->is_emissive) continue;
        double light_pdf = 0.0, attenuation = 1.0;
        v3 lp = { 0.0, 0.0, 0.0 };
        switch(ls->type)
        {
            case DRT_GEO_POINT:
            {
                lp = v3_make(ls->position);
                double dist = v3_length(v3_sub(lp, hit->position));
                light_pdf = 1.0;
                attenuation = (4.0 * PI_L * dist * dist);   /* Q3: multiplied, not divided */
                break;
            }
            case DRT_GEO_SPHERE:
            {
                double u = rng(c);
                double v = rng(c);
                double r = sqrt(1.0 - u * u);
                double t = 2.0 * PI_L * v;
                v3 sp = { r * cos(t), r * sin(t), u };   /* Q5: z >= 0 half only */
                lp = v3_sum(v3_make(ls->position), v3_scale(sp, ls->radius));
                light_pdf = (4.0 * PI_L * ls->radius * ls->radius);
                break;
            }
            case DRT_GEO_PLANE:
            {
                double u = rng(c);
                double v = rng(c);
                v3 up = v3_scale(v3_make(ls->u), u);
                v3 vp = v3_scale(v3_make(ls->v), v);
                lp = v3_sum(v3_sum(v3_make(ls->position), up), vp);
                light_pdf = v3_length(v3_cross(v3_make(ls->u), v3_make(ls->v)));
                break;
            }
            default: break;
        }
        if(mutually_visible(c, hit->position, lp))
        {
            v3 incoming = v3_normalise(v3_sub(lp, hit->position));
            bdsf(c, refl, hit, incoming);
            double k = attenuation * (light_pdf);
            for(int w = 0; w < n; w += 1) contribution[w] = contribution[w] + refl[w];            /* Q4: running sum ... */
            for(int w = 0; w < n; w += 1) contribution[w] = contribution[w] * lm->spd[DRT_SPD_EMISSION][w];
            for(int w = 0; w < n; w += 1) contribution[w] = contribution[w] * k;                  /* ... rescaled by every later light */
        }
    }
}

static void cast_ray(ctx *c, double *dst, v3 origin, v3 dir, uint32_t max_depth)   /* :432-479 */
{
    int n = c->n;
    double contribution[DRT_MAX_WAVELENGTHS], throughput[DRT_MAX_WAVELENGTHS], refl[DRT_MAX_WAVELENGTHS];
    memset(contribution, 0, sizeof(double) * (size_t)n);
    memset(refl, 0, sizeof(double) * (size_t)n);
    for(int i = 0; i < n; i += 1) throughput[i] = 1.0;
    hit_point hit;
    memset(&hit, 0, sizeof(hit));
    uint32_t depth;
    for(depth = 0; depth < max_depth; depth += 1)
    {
        find_intersection(c, &hit, origin, dir);
        const drt_material *mat = hit.surface_material;
        if(mat->is_black_body && !mat->is_emissive) break;
        else if(mat->is_black_body && mat->is_emissive)
        {
            for(int i = 0; i < n; i += 1) dst[i] = dst[i] + (throughput[i] * mat->spd[DRT_SPD_EMISSION][i]);   /* Q6 */
            break;
        }
        else
        {
            c->count->shaded_bounces += 1;
            direct_light(c, contribution, &hit);
            for(int i = 0; i < n; i += 1) dst[i] = dst[i] + (throughput[i] * contribution[i]);
            v3 in = { 0.0, 0.0, 0.0 };
            double inv_pdf = 0.0;
            sample_direction(c, mat->dir_func, &in, &inv_pdf, &hit);
            bdsf(c, refl, &hit, in);
            for(int i = 0; i < n; i += 1) refl[i] = refl[i] * inv_pdf;
            for(int i = 0; i < n; i += 1) throughput[i] = throughput[i] * refl[i];
            dir = in;
            origin = hit.position;
        }
    }
    if(depth < max_depth) c->count->terminated_at_depth[depth < 7 ? depth : 7] += 1;
    else c->count->reached_depth_cap += 1;
}

/* the camera ray of sample_scene, daily_ray_trace.c:571-612 (sample_pixel_point :550-569) */
static void camera_ray(ctx *c, uint32_t x, uint32_t y, int scheme, v3 *origin_out, v3 *dir_out)
{
    const drt_camera *cam = c->cam;
    double px = 0.0, py = 0.0;
    if(scheme == DRT_PIXEL_CENTER) { px = 0.5; py = 0.5; }
    else if(scheme == DRT_PIXEL_RANDOM) { px = rng(c); py = rng(c); }
    double film_x = ((double)x + px) * cam->pixel_width;
    double film_y = ((double)y + py) * cam->pixel_height;
    v3 up = v3_make(cam->up), right = v3_make(cam->right), forward = v3_make(cam->forward);
    v3 bottom = v3_scale(up, film_y);
    v3 left = v3_scale(right, film_x);
    v3 point = v3_sum(v3_sum(left, bottom), v3_make(cam->film_bottom_left));

    v3 origin, dir;
    v3 aperture = v3_make(cam->aperture_position);
    if(cam->aperture_radius > 0.0)
    {
        const v3 plus_z = { 0.0, 0.0, 1.0 };
        v3 focus_dir = v3_normalise(v3_sub(aperture, point));
        focus_dir = v3_scale(focus_dir, cam->focal_depth / v3_dot(focus_dir, forward));
        v3 focus_point = v3_sum(point, focus_dir);
        m3 r = rotation_between(plus_z, forward);
        v3 disc = v3_scale(uniform_sample_disc(c), cam->aperture_radius);
        v3 lens = m3_apply(r, disc);
        origin = v3_sum(aperture, lens);
        dir = v3_normalise(v3_sub(focus_point, origin));
    }
    else
    {
        origin = point;
        dir = v3_normalise(v3_sub(aperture, origin));   /* Q1: film sits behind the pinhole, image comes out rotated */
    }
    *origin_out = origin;
    *dir_out = dir;
}

/* sample_scene, daily_ray_trace.c:571-618 */
static void sample_scene(ctx *c, double *contribution, double *filter, uint32_t x, uint32_t y, uint32_t max_depth, int scheme)
{
    int n = c->n;
    memset(contribution, 0, sizeof(double) * (size_t)n);
    c->count->paths += 1;

    v3 origin, dir, forward = v3_make(c->cam->forward);
    camera_ray(c, x, y, scheme, &origin, &dir);
    cast_ray(c, contribution, origin, dir, max_depth);

    double vignette = v3_dot(dir, forward);   /* Q20 */
    for(int i = 0; i < n; i += 1) contribution[i] = contribution[i] * (vignette * 1.0);
    *filter = 1.0;
}

/* ------------------------------------------------------------------ exported checker API */

void drt_oracle_sample(const drt_scene *scene, const drt_camera *camera, const drt_render_params *params,
                       uint32_t x, uint32_t y, uint32_t sample, double *out_spd, double *out_filter, drt_oracle_counters *counters)
{
    drt_oracle_counters local;
    memset(&local, 0, sizeof(local));
    ctx c = { scene, camera, scene->num_wavelengths, {0}, counters ? counters : &local };
    drt_rng_begin(&c.rng, params->seed, y * params->width + x, sample);
    sample_scene(&c, out_spd, out_filter, x, y, params->max_depth, params->pixel_scheme);
}

/* Pixels [x0,x1)x[y0,y1), samples [params->sample_begin, sample_end), accumulated as render_image does
 * (daily_ray_trace.c:720-743).  Tile-local row-major buffers, zeroed by the caller:
 *   sum (N+1 per pixel: SPD sum, filter sum), avg, m2 (N per pixel), paths (optional, [pixel][sample][N]). */
void drt_oracle_render_tile(const drt_scene *scene, const drt_camera *camera, const drt_render_params *params,
                            uint32_t x0, uint32_t y0, uint32_t x1, uint32_t y1,
                            double *sum, double *avg, double *m2, double *paths, drt_oracle_counters *counters)
{
    drt_oracle_counters local;
    memset(&local, 0, sizeof(local));
    ctx c = { scene, camera, scene->num_wavelengths, {0}, counters ? counters : &local };
    size_t n = (size_t)c.n;
    uint32_t tw = x1 - x0, s0 = params->sample_begin, s1 = params->sample_end;
    double contribution[DRT_MAX_WAVELENGTHS], filter;
    for(uint32_t s = s0; s < s1; s += 1)
    for(uint32_t y = y0; y < y1; y += 1)
    for(uint32_t x = x0; x < x1; x += 1)
    {
        size_t p = (size_t)(y - y0) * tw + (x - x0);
        double *d_sum = sum + (n + 1) * p, *d_avg = avg + n * p, *d_m2 = m2 + n * p;
        drt_rng_begin(&c.rng, params->seed, y * params->width + x, s);
        sample_scene(&c, contribution, &filter, x, y, params->max_depth, params->pixel_scheme);
        if(paths) memcpy(paths + (p * (s1 - s0) + (s - s0)) * n, contribution, n * sizeof(double));
        for(size_t i = 0; i < n; i += 1) d_sum[i] = d_sum[i] + contribution[i];
        d_sum[n] += filter;
        for(size_t i = 0; i < n; i += 1)   /* Welford, :736-743 */
        {
            double delta = contribution[i] - d_avg[i];
            double step = delta / (double)(s + 1);
            d_avg[i] = d_avg[i] + step;
            d_m2[i] = d_m2[i] + (delta * (contribution[i] - d_avg[i]));
        }
    }
}

/* The material the camera ray of sample `sample` of pixel (x, y) hits first (the escape material when it hits nothing). */
int drt_oracle_primary_material(const drt_scene *scene, const drt_camera *camera, const drt_render_params *params,
                                uint32_t x, uint32_t y, uint32_t sample)
{
    drt_oracle_counters local;
    memset(&local, 0, sizeof(local));
    ctx c = { scene, camera, scene->num_wavelengths, {0}, &local };
    drt_rng_begin(&c.rng, params->seed, y * params->width + x, sample);
    v3 origin, dir;
    camera_ray(&c, x, y, params->pixel_scheme, &origin, &dir);
    hit_point hit;
    memset(&hit, 0, sizeof(hit));
    find_intersection(&c, &hit, origin, dir);
    return (int)(hit.surface_material - scene->materials);
}

/* bdsf() at a hand-built hit point, set up as oracle/ref_perpath.c's ref_bdsf does (on_dot = n.out, trans_wl 630 nm):
 * the CPU-tier check of the classed kernel's factorisation where the reference build is absent. */
void drt_oracle_bdsf(const drt_scene *scene, uint32_t surface_material, uint32_t incident_material, uint32_t transmit_material,
                     const double *normal, const double *out_dir, const double *in_dir, double *result)
{
    ctx c = { scene, NULL, scene->num_wavelengths, {0}, NULL };
    hit_point p;
    memset(&p, 0, sizeof(p));
    p.normal = v3_make(normal);
    p.out = v3_make(out_dir);
    p.on_dot = v3_dot(p.normal, p.out);
    p.trans_wl = 630.0;
    p.surface_material = &scene->materials[surface_material];
    p.incident_material = &scene->materials[incident_material];
    p.transmit_material = &scene->materials[transmit_material];
    bdsf(&c, result, &p, v3_make(in_dir));
}

/* The hemisphere samplers' frame: q (a sample about +z) rotated onto the normal n, as sample_direction does it. */
void drt_oracle_rotate_from_z(const double *normal, const double *q, double *result)
{
    const v3 plus_z = { 0.0, 0.0, 1.0 };
    v3 v = m3_apply(rotation_between(plus_z, v3_make(normal)), v3_make(q));
    result[0] = v.x; result[1] = v.y; result[2] = v.z;
}
