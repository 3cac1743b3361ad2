/*
 * csrc/drt_capi.cu -- the C ABI of include/drt_cuda.h over the kernels in this directory.
 *
 * Host-side work here is only: narrowing the f64 scene into the device layout (precomputing what the reference
 * recomputes per call, e.g. the normalised plane frame of line_plane_intersection, geometry.c:166-170), owning
 * device buffers, sizing the persistent grid, and launching.  There is no CPU implementation of any render step.
 */
#include <cuda_runtime.h>
#include <math.h>
#include <stdarg.h>
#include <stdio.h>
#include <string.h>
#include <vector>
#include "drt_context.cuh"

static thread_local char g_err[512];

int drt_fail(int code, const char *fmt, ...)
{
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
    return code;
}

extern "C" const char *drt_cuda_last_error(void) { return g_err; }

extern "C" int drt_cuda_device_count(void)
{
    int n = 0;
    if(cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
    return n;
}

extern "C" int drt_cuda_create(int device, drt_cuda_context **out)
{
    if(!out) return fail(DRT_CUDA_E_ARG, "out is NULL");
    int count = drt_cuda_device_count();
    if(count <= 0) return fail(DRT_CUDA_E_NO_DEVICE, "no CUDA device is visible; this library has no CPU path");
    if(device < 0 || device >= count) return fail(DRT_CUDA_E_ARG, "device %d out of range (%d visible)", device, count);
    CU(cudaSetDevice(device));
    cudaDeviceProp prop;
    CU(cudaGetDeviceProperties(&prop, device));
    drt_cuda_context *ctx = new drt_cuda_context();
    ctx->device = device;
    ctx->num_sms = prop.multiProcessorCount;
    ctx->smem_optin = prop.sharedMemPerBlockOptin;
    cudaError_t e = cudaMalloc(&ctx->d_stats_ring, DRT_RING * sizeof(DeviceStats));
    if(e == cudaSuccess) e = cudaMalloc(&ctx->d_counter_ring, DRT_RING * sizeof(unsigned int));
    if(e == cudaSuccess) e = cudaMemset(ctx->d_stats_ring, 0, DRT_RING * sizeof(DeviceStats));
    if(e != cudaSuccess)
    {
        cudaFree(ctx->d_stats_ring); cudaFree(ctx->d_counter_ring);
        delete ctx;
        return fail(DRT_CUDA_E_CUDA, "drt_cuda_create: %s", cudaGetErrorString(e));
    }
    ctx->d_stats = ctx->d_stats_ring;
    *out = ctx;
    return DRT_CUDA_OK;
}

extern "C" void drt_cuda_destroy(drt_cuda_context *ctx)
{
    if(!ctx) return;
    cudaSetDevice(ctx->device);
    cudaFree(ctx->d_geom32); cudaFree(ctx->d_geom64); cudaFree(ctx->d_index); cudaFree(ctx->d_pool);
    cudaFree(ctx->d_rgb_tables); cudaFree(ctx->d_stats_ring); cudaFree(ctx->d_counter_ring); cudaFree(ctx->d_film); cudaFree(ctx->d_dump); cudaFree(ctx->d_slice); cudaFree(ctx->d_deep);
    cudaFree(ctx->d_denoise);
    if(ctx->denoise_done) cudaEventDestroy(ctx->denoise_done);
    drt_exchange_release(ctx);
    if(ctx->band_render) cudaStreamDestroy(ctx->band_render);
    if(ctx->band_copy) cudaStreamDestroy(ctx->band_copy);
    for(int i = 0; i < 16; i += 1) if(ctx->band_done[i]) cudaEventDestroy(ctx->band_done[i]);
    delete ctx;
}

/* value_at_wl, spectrum.c:150-162, in f64 on the host */
static double value_at_wl(const drt_scene *s, const double *spd, double wl)
{
    uint32_t i0 = (uint32_t)((wl - s->min_wl) / s->wl_interval), i1 = i0 + 1;
    double w0 = s->min_wl + i0 * s->wl_interval, w1 = s->min_wl + i1 * s->wl_interval;
    return spd[i0] + ((wl - w0) * ((spd[i1] - spd[i0]) / (w1 - w0)));
}

/* Screen-space bound of the scene for a pinhole camera: the film point whose ray passes through a world point Q is
 * P = ap + (ap - Q) * f / depth(Q) (sample_scene :602-607: the ray starts on the film and runs through the aperture), so the
 * projection of a convex surface is the hull of its projected corners as long as every corner is in front of the aperture.
 * Returns false (no bound) for a thin lens, when a surface reaches behind the aperture, or when the escape material is
 * EMISSIVE (an environment light, Q19: init_scene forces the escape material black-body, daily_ray_trace.c:148, and cast_ray
 * :452-456 adds throughput * emission for a ray that leaves the scene -- such a pixel is lit although it sees no surface).
 * Pure host arithmetic. */
static bool scene_hit_bound(const drt_scene *scene, const drt_camera *camera, double *out_u0, double *out_u1, double *out_v0, double *out_v1)
{
    if(camera->aperture_radius != 0.0) return false;
    if(scene->escape_material >= 0 && scene->escape_material < scene->num_materials && scene->materials[scene->escape_material].is_emissive) return false;
    const double *ap = camera->aperture_position, *fw = camera->forward;
    double fd = 0.0;
    for(int k = 0; k < 3; k += 1) fd += (ap[k] - camera->film_bottom_left[k]) * fw[k];
    double g_rr = 0.0, g_uu = 0.0, g_ru = 0.0;
    for(int k = 0; k < 3; k += 1) { g_rr += camera->right[k] * camera->right[k]; g_uu += camera->up[k] * camera->up[k]; g_ru += camera->right[k] * camera->up[k]; }
    const double g_det = g_rr * g_uu - g_ru * g_ru;
    bool ok = fd > 0.0 && camera->pixel_width > 0.0 && camera->pixel_height > 0.0 && g_det > 1e-12;
    double u0 = 1e300, u1 = -1e300, v0 = 1e300, v1 = -1e300;
    auto project = [&](const double *q) {
        double depth = 0.0;
        for(int k = 0; k < 3; k += 1) depth += (q[k] - ap[k]) * fw[k];
        if(!(depth > 1e-9)) { ok = false; return; }
        double dr = 0.0, du = 0.0;   /* (P - film_bottom_left) = a * right + b * up: solve for a, b (no orthonormality assumed) */
        for(int k = 0; k < 3; k += 1)
        {
            double pk = ap[k] + (ap[k] - q[k]) * (fd / depth) - camera->film_bottom_left[k];
            dr += pk * camera->right[k]; du += pk * camera->up[k];
        }
        double u = (dr * g_uu - du * g_ru) / g_det / camera->pixel_width, v = (du * g_rr - dr * g_ru) / g_det / camera->pixel_height;
        if(u < u0) u0 = u; if(u > u1) u1 = u; if(v < v0) v0 = v; if(v > v1) v1 = v;
    };
    for(int i = 0; i < scene->num_surfaces && ok; i += 1)
    {
        const drt_surface *f = &scene->surfaces[i];
        if(f->type == DRT_GEO_PLANE)
            for(int c = 0; c < 4; c += 1)
            {
                double q[3];
                for(int k = 0; k < 3; k += 1) q[k] = f->position[k] + ((c & 1) ? f->u[k] : 0.0) + ((c & 2) ? f->v[k] : 0.0);
                project(q);
            }
        else if(f->type == DRT_GEO_SPHERE)
            for(int c = 0; c < 8; c += 1)   /* corners of the sphere's bounding cube */
            {
                double q[3];
                for(int k = 0; k < 3; k += 1) q[k] = f->position[k] + (((c >> k) & 1) ? f->radius : -f->radius);
                project(q);
            }
    }
    if(!(ok && u0 <= u1)) return false;
    *out_u0 = u0; *out_u1 = u1; *out_v0 = v0; *out_v1 = v1;
    return true;
}

/* the pixel rectangle of a bound, with one pixel of slack on every side (f32 camera arithmetic of the kernel against the f64 projection) */
static void hit_rect(bool have, double u0, double u1, double v0, double v1, uint32_t width, uint32_t height, uint32_t rect[4])
{
    rect[0] = 0; rect[1] = 0; rect[2] = width; rect[3] = height;
    if(!have) return;
    auto clampi = [](double v, uint32_t hi) -> uint32_t { return v <= 0.0 ? 0u : v >= (double)hi ? hi : (uint32_t)v; };
    rect[0] = clampi(floor(u0) - 1.0, width);  rect[2] = clampi(ceil(u1) + 1.0, width);
    rect[1] = clampi(floor(v0) - 1.0, height); rect[3] = clampi(ceil(v1) + 1.0, height);
}

/* boundary plane: every other surface (rectangle corners, sphere extents, points) lies in one closed half-space of it, so a segment
 * between two points of the scene can meet it only at its end points (GeomT::nax_b) */
static bool surface_is_boundary(const drt_scene *s, int i)
{
    const drt_surface *f = &s->surfaces[i];
    if(f->type != DRT_GEO_PLANE) return false;
    const double eps = 1e-6;   /* two orders below the reference's 1e-4 ray offset */
    double lo = 0.0, hi = 0.0;
    auto side = [&](const double *q, double r) {
        double d = (q[0] - f->position[0]) * f->normal[0] + (q[1] - f->position[1]) * f->normal[1] + (q[2] - f->position[2]) * f->normal[2];
        if(d - r < lo) lo = d - r;
        if(d + r > hi) hi = d + r;
    };
    for(int j = 0; j < s->num_surfaces; j += 1)
    {
        if(j == i) continue;
        const drt_surface *o = &s->surfaces[j];
        if(o->type == DRT_GEO_PLANE)
            for(int c = 0; c < 4; c += 1)
            {
                double q[3];
                for(int k = 0; k < 3; k += 1) q[k] = o->position[k] + ((c & 1) ? o->u[k] : 0.0) + ((c & 2) ? o->v[k] : 0.0);
                side(q, 0.0);
            }
        else side(o->position, o->type == DRT_GEO_SPHERE ? o->radius : 0.0);
    }
    return lo >= -eps || hi <= eps;
}

extern "C" int drt_cuda_analyse_scene(const drt_scene *scene, const drt_camera *camera, uint32_t width, uint32_t height,
                                      uint32_t hit_rect_out[4], int32_t *boundary_out)
{
    if(!scene || !camera || !hit_rect_out || !boundary_out) return fail(DRT_CUDA_E_ARG, "NULL argument");
    if(scene->num_surfaces < 0 || scene->num_surfaces > DRT_MAX_SURFACES) return fail(DRT_CUDA_E_ARG, "%d surfaces out of range", scene->num_surfaces);
    double u0 = 0, u1 = 0, v0 = 0, v1 = 0;
    bool have = scene_hit_bound(scene, camera, &u0, &u1, &v0, &v1);
    hit_rect(have, u0, u1, v0, v1, width, height, hit_rect_out);
    for(int i = 0; i < scene->num_surfaces; i += 1) boundary_out[i] = surface_is_boundary(scene, i) ? 1 : 0;
    return DRT_CUDA_OK;
}

/* Shading class of a material for the compact-record kernels (GeomT::mclass), with the lobe multiplicities of a plastic and the
 * spectral basis of a specular material.  Every lobe of bdsf.c either always writes (bp_diffuse, bp_glossy, mirror -- which writes
 * zero on a mismatch --, ct_conductor) or writes only when `in` is the exact reflection / refraction direction (fs_*: Q7, Q8). */
static int classify_material(const drt_scene *s, int m, int *nd_out, int *ng_out, int *basis_out)
{
    const drt_material *mm = &s->materials[m];
    int nd = 0, ng = 0, nmirror = 0, ncond = 0, ndiel = 0, nct = 0, nother = 0;
    for(int k = 0; k < mm->num_lobes; k += 1)
        switch(mm->lobes[k])
        {
            case DRT_LOBE_BP_DIFFUSE: nd += 1; break;
            case DRT_LOBE_BP_GLOSSY: ng += 1; break;
            case DRT_LOBE_MIRROR: nmirror += 1; break;
            case DRT_LOBE_FS_CONDUCTOR: ncond += 1; break;
            case DRT_LOBE_FS_DIELECTRIC_REFLECTANCE: case DRT_LOBE_FS_DIELECTRIC_TRANSMITTANCE: ndiel += 1; break;
            case DRT_LOBE_CT_CONDUCTOR: nct += 1; break;
            default: nother += 1; break;
        }
    if(nd_out) *nd_out = nd;
    if(ng_out) *ng_out = ng;
    if(basis_out) *basis_out = 0;
    if(mm->num_lobes < 1 || nother) return DRT_CLASS_GENERAL;
    const bool base_n = s->base_material >= 0 && (s->materials[s->base_material].spd_mask & (1 << DRT_SPD_REFRACT));
    const bool own_n = (mm->spd_mask & (1 << DRT_SPD_REFRACT)) != 0;
    if(nd + ng == mm->num_lobes) return DRT_CLASS_PLASTIC;
    if(nct == mm->num_lobes) return (base_n && own_n) ? DRT_CLASS_ROUGH : DRT_CLASS_GENERAL;
    if(nmirror + ncond + ndiel == mm->num_lobes && (nmirror != 0) + (ncond != 0) + (ndiel != 0) == 1)
    {
        if(basis_out) *basis_out = nmirror ? 0 : ndiel ? 1 : 2;
        return (nmirror || (base_n && own_n)) ? DRT_CLASS_SPECULAR : DRT_CLASS_GENERAL;
    }
    return DRT_CLASS_GENERAL;
}

/* Which render kernel a scene gets (drt_render.cuh): 1 plastic-only, 2 classed, 0 general.  The compact-record kernels (1, 2) carry
 * throughput * E(light): the only emitter a path can run into must then be that light, so an emissive escape material (a sky, Q19) or
 * a second light sends the scene to the general kernel. */
static int scene_kernel_mode(const drt_scene *scene)
{
    int nlights = 0;
    for(int i = 0; i < scene->num_surfaces; i += 1) nlights += scene->materials[scene->surfaces[i].material].is_emissive ? 1 : 0;
    bool all_fast = nlights == 1 && !scene->materials[scene->escape_material].is_emissive, classed = all_fast;
    for(int i = 0; i < scene->num_surfaces; i += 1)
    {
        const int m = scene->surfaces[i].material;
        if(scene->materials[m].is_black_body || scene->surfaces[i].type == DRT_GEO_POINT || scene->surfaces[i].type == DRT_GEO_NONE) continue;
        const int cls = classify_material(scene, m, nullptr, nullptr, nullptr);
        if(cls != DRT_CLASS_PLASTIC) all_fast = false;
        if(cls == DRT_CLASS_GENERAL) classed = false;
    }
    return all_fast ? 1 : classed ? 2 : 0;
}

template <typename R>
static void fill_geom(GeomT<R> *g, const drt_scene *s, const drt_camera *c);

extern "C" int drt_cuda_plan_scene(const drt_scene *scene, const drt_camera *camera, int32_t *kernel_mode_out, int32_t *material_class, float *specular_constants)
{
    if(!scene || !camera || !kernel_mode_out) return fail(DRT_CUDA_E_ARG, "NULL argument");
    int rc = drt_cuda_validate_scene(scene);
    if(rc != DRT_CUDA_OK) return rc;
    *kernel_mode_out = scene_kernel_mode(scene);
    if(material_class || specular_constants)
    {
        GeomT<float> *g = new GeomT<float>();
        fill_geom(g, scene, camera);
        for(int m = 0; m < scene->num_materials; m += 1)
        {
            if(material_class) material_class[m] = g->mclass[m];
            if(specular_constants) memcpy(specular_constants + (size_t)m * 6, g->spec_c[m], 6 * sizeof(float));
        }
        delete g;
    }
    return DRT_CUDA_OK;
}

template <typename R>
static void fill_geom(GeomT<R> *g, const drt_scene *s, const drt_camera *c)
{
    memset(g, 0, sizeof(*g));
    g->nsurf = s->num_surfaces; g->nmat = s->num_materials; g->n = s->num_wavelengths;
    g->base_mat = s->base_material; g->escape_mat = s->escape_material;
    uint32_t i0 = (uint32_t)((DRT_TRANS_WL - s->min_wl) / s->wl_interval);
    double w0 = s->min_wl + i0 * s->wl_interval, w1 = s->min_wl + (i0 + 1) * s->wl_interval;
    g->trans_num = (R)(DRT_TRANS_WL - w0);
    g->trans_den = (R)(w1 - w0);
    int nl = 0;
    for(int i = 0; i < s->num_surfaces; i += 1)
    {
        const drt_surface *f = &s->surfaces[i];
        g->type[i] = f->type; g->mat[i] = f->material;
        g->px[i] = (R)f->position[0]; g->py[i] = (R)f->position[1]; g->pz[i] = (R)f->position[2];
        g->rad[i] = (R)f->radius;
        g->nx[i] = (R)f->normal[0]; g->ny[i] = (R)f->normal[1]; g->nz[i] = (R)f->normal[2];
        g->ux[i] = (R)f->u[0]; g->uy[i] = (R)f->u[1]; g->uz[i] = (R)f->u[2];
        g->vx[i] = (R)f->v[0]; g->vy[i] = (R)f->v[1]; g->vz[i] = (R)f->v[2];
        double pdf = 1.0;
        if(f->type == DRT_GEO_PLANE)
        {
            double ul = sqrt(f->u[0] * f->u[0] + f->u[1] * f->u[1] + f->u[2] * f->u[2]);
            double vl = sqrt(f->v[0] * f->v[0] + f->v[1] * f->v[1] + f->v[2] * f->v[2]);
            g->ulen[i] = (R)ul; g->vlen[i] = (R)vl;
            g->unx[i] = (R)(f->u[0] / ul); g->uny[i] = (R)(f->u[1] / ul); g->unz[i] = (R)(f->u[2] / ul);
            g->vnx[i] = (R)(f->v[0] / vl); g->vny[i] = (R)(f->v[1] / vl); g->vnz[i] = (R)(f->v[2] / vl);
            double cx = f->u[1] * f->v[2] - f->u[2] * f->v[1], cy = f->u[2] * f->v[0] - f->u[0] * f->v[2], cz = f->u[0] * f->v[1] - f->u[1] * f->v[0];
            pdf = sqrt(cx * cx + cy * cy + cz * cz);                       /* daily_ray_trace.c:314 */
        }
        else if(f->type == DRT_GEO_SPHERE) pdf = (double)(4.0 * 3.1415926535897932385L * f->radius * f->radius);   /* :304 */
        g->light_pdf[i] = (R)pdf;
        if(s->materials[f->material].is_emissive) g->light_surf[nl++] = i;
    }
    g->nlights = nl;
    /* packed copies regrouped by type for the intersection loops: x-, y-, z-aligned rectangles, other planes, spheres */
    auto plane_axis = [&](const drt_surface *f) -> int {
        auto single = [](const double *v) -> int {
            int axis = -1;
            for(int k = 0; k < 3; k += 1) if(v[k] != 0.0) { if(axis >= 0) return -1; axis = k; }
            return axis;
        };
        int a = single(f->normal), b = single(f->u), c = single(f->v);
        if(a < 0 || b < 0 || c < 0 || a == b || a == c || b == c) return -1;
        if(f->normal[a] != 1.0 && f->normal[a] != -1.0) return -1;
        return a;
    };
    int slot = 0;
    for(int pass = 0; pass < 9; pass += 1)   /* passes 0-7: plane group (pass / 2), boundary planes first; pass 8: spheres */
        for(int i = 0; i < s->num_surfaces; i += 1)
        {
            const drt_surface *f = &s->surfaces[i];
            const int group = pass / 2;
            if(pass < 8)
            {
                if(f->type != DRT_GEO_PLANE || plane_axis(f) != (group < 3 ? group : -1)) continue;
                if(surface_is_boundary(s, i) != ((pass & 1) == 0)) continue;
                if((pass & 1) == 0) g->nax_b[group] += 1;
            }
            else if(f->type != DRT_GEO_SPHERE) continue;
            g->sid[slot] = i;
            g->N4[slot] = R4<R>{ g->nx[i], g->ny[i], g->nz[i], (R)0 };
            g->P4[slot] = R4<R>{ g->px[i], g->py[i], g->pz[i], g->rad[i] };
            g->U4[slot] = R4<R>{ g->unx[i], g->uny[i], g->unz[i], g->ulen[i] };
            g->V4[slot] = R4<R>{ g->vnx[i], g->vny[i], g->vnz[i], g->vlen[i] };
            if(group < 3)
            {
                const int a = group, b = (a == 0) ? 1 : 0, c = (a == 2) ? 1 : 2;   /* in-plane axes b < c */
                double lo[2], hi[2];
                const int bc[2] = { b, c };
                for(int k = 0; k < 2; k += 1)
                {
                    double p0 = f->position[bc[k]], p1 = p0 + f->u[bc[k]] + f->v[bc[k]];   /* one of u, v lies along this axis */
                    lo[k] = p0 < p1 ? p0 : p1; hi[k] = p0 < p1 ? p1 : p0;
                }
                g->AX4[slot] = R4<R>{ (R)f->position[a], (R)(0.5 * (lo[0] + hi[0])), (R)(0.5 * (hi[0] - lo[0])), (R)(0.5 * (lo[1] + hi[1])) };
                g->AXH[slot] = R2<R>{ (R)(0.5 * (hi[1] - lo[1])), (R)i };
                g->nax[a] += 1;
            }
            slot += 1;
            if(pass < 8) g->nplanes += 1; else g->nspheres += 1;
        }
    for(int m = 0; m < s->num_materials; m += 1)
    {
        const drt_material *mm = &s->materials[m];
        g->mflags[m] = (mm->is_black_body ? 1 : 0) | (mm->is_emissive ? 2 : 0);
        g->nlobes[m] = mm->num_lobes; g->dirf[m] = mm->dir_func;
        for(int k = 0; k < mm->num_lobes && k < DRT_MAX_LOBES; k += 1) g->lobes[m][k] = (unsigned char)mm->lobes[k];
        g->shin[m] = (R)mm->shininess; g->rough[m] = (R)mm->roughness;
        /* which spectral bases this lobe list can produce, and how many record words one evaluation needs */
        int mask = 0;
        for(int k = 0; k < mm->num_lobes && k < DRT_MAX_LOBES; k += 1)
            switch(mm->lobes[k])
            {
                case DRT_LOBE_BP_DIFFUSE: mask |= 1 << BK_DIFFUSE; break;
                case DRT_LOBE_BP_GLOSSY: mask |= 1 << BK_GLOSSY; break;
                case DRT_LOBE_MIRROR: mask |= 1 << BK_MIRROR; break;
                case DRT_LOBE_FS_CONDUCTOR: mask |= 1 << BK_COND_ON; break;
                case DRT_LOBE_FS_DIELECTRIC_REFLECTANCE: mask |= 1 << BK_DIEL_R; break;
                case DRT_LOBE_FS_DIELECTRIC_TRANSMITTANCE: mask |= (1 << BK_DIEL_R) | (1 << BK_CONST); break;
                case DRT_LOBE_CT_CONDUCTOR: mask |= 1 << BK_COND_MN; break;
                default: break;
            }
        g->bmask[m] = mask;
        g->mclass[m] = classify_material(s, m, nullptr, nullptr, nullptr);
        if(g->mclass[m] == DRT_CLASS_SPECULAR)
            for(int match = 0; match < 3; match += 1)
            {
                /* the lobe walk of bdsf() (daily_ray_trace.c:215-229) over the match-gated lobes: a lobe that does not write leaves
                 * the previous lobe's value in the scratch spectrum, which is added again (Q7) */
                const bool refl = match == 1, trans = match == 2;
                double cur_c = 0.0, cur_x = 0.0, acc_c = 0.0, acc_x = 0.0;
                for(int k = 0; k < mm->num_lobes; k += 1)
                {
                    bool wrote = false; double val = 0.0, val_c = 0.0;
                    switch(mm->lobes[k])
                    {
                        case DRT_LOBE_MIRROR: wrote = true; val = refl ? 1.0 : 0.0; break;
                        case DRT_LOBE_FS_CONDUCTOR: case DRT_LOBE_FS_DIELECTRIC_REFLECTANCE: wrote = refl; val = 1.0; break;
                        case DRT_LOBE_FS_DIELECTRIC_TRANSMITTANCE: wrote = trans; val = -1.0; val_c = 1.0; break;
                        default: break;
                    }
                    if(wrote) { cur_x = val; cur_c = val_c; }
                    acc_c += cur_c; acc_x += cur_x;
                }
                g->spec_c[m][match][0] = (float)acc_c; g->spec_c[m][match][1] = (float)acc_x;
            }
        int nct = 0;
        for(int k = 0; k < mm->num_lobes && k < DRT_MAX_LOBES; k += 1) nct += mm->lobes[k] == DRT_LOBE_CT_CONDUCTOR;
        g->ct_mult[m] = (float)nct;
        int words = __builtin_popcount((unsigned)mask) + ((mask >> BK_COND_MN) & 1);
        if(!mm->is_black_body && words > g->eval_words) g->eval_words = words;
        if(mm->spd_mask & (1 << DRT_SPD_REFRACT))
        {
            g->n630[m] = (R)value_at_wl(s, mm->spd[DRT_SPD_REFRACT], DRT_TRANS_WL);
            g->refr_a[m] = (R)mm->spd[DRT_SPD_REFRACT][i0];
            g->refr_b[m] = (R)mm->spd[DRT_SPD_REFRACT][i0 + 1];
        }
    }
    for(int k = 0; k < 3; k += 1)
    {
        g->fwd[k] = (R)c->forward[k]; g->right[k] = (R)c->right[k]; g->up[k] = (R)c->up[k];
        g->ap_pos[k] = (R)c->aperture_position[k]; g->film_bl[k] = (R)c->film_bottom_left[k];
    }
    g->ap_radius = (R)c->aperture_radius; g->focal_depth = (R)c->focal_depth;
    g->pixel_w = (R)c->pixel_width; g->pixel_h = (R)c->pixel_height;
    for(int k = 0; k < 9; k += 1) g->lens_rot[k] = (R)c->lens_rotation[k];
}

/* Everything the kernels index device tables with, checked on the host (no device needed): a caller other than the in-repo
 * parser gets an error code, not a wild shared-memory read. */
extern "C" int drt_cuda_validate_scene(const drt_scene *scene)
{
    if(!scene) return fail(DRT_CUDA_E_ARG, "NULL argument");
    int n = scene->num_wavelengths;
    if(n < 2 || n > DRT_MAX_WAVELENGTHS) return fail(DRT_CUDA_E_ARG, "%d wavelengths (need 2..%d)", n, DRT_MAX_WAVELENGTHS);
    if(scene->num_surfaces < 0 || scene->num_surfaces > DRT_MAX_SURFACES || scene->num_materials < 1 || scene->num_materials > DRT_MAX_MATERIALS)
        return fail(DRT_CUDA_E_ARG, "%d surfaces / %d materials out of range", scene->num_surfaces, scene->num_materials);
    if(scene->base_material < 0 || scene->escape_material < 0) return fail(DRT_CUDA_E_UNSUPPORTED, "scene needs a base_material and an escape_material");
    if(scene->base_material >= scene->num_materials || scene->escape_material >= scene->num_materials)
        return fail(DRT_CUDA_E_ARG, "base_material %d / escape_material %d out of range (%d materials)", scene->base_material, scene->escape_material, scene->num_materials);
    if(!(scene->wl_interval > 0.0)) return fail(DRT_CUDA_E_ARG, "wl_interval must be positive");
    uint32_t i0 = (uint32_t)((DRT_TRANS_WL - scene->min_wl) / scene->wl_interval);
    if(DRT_TRANS_WL < scene->min_wl || (int)i0 + 1 >= n) return fail(DRT_CUDA_E_UNSUPPORTED, "630 nm (trans_wl, daily_ray_trace.c:381) lies outside the wavelength grid");
    for(int i = 0; i < scene->num_surfaces; i += 1)
    {
        if(scene->surfaces[i].material < 0 || scene->surfaces[i].material >= scene->num_materials) return fail(DRT_CUDA_E_ARG, "surface %d: bad material index", i);
        if(scene->surfaces[i].type < DRT_GEO_NONE || scene->surfaces[i].type > DRT_GEO_PLANE) return fail(DRT_CUDA_E_ARG, "surface %d: bad type %d", i, scene->surfaces[i].type);
    }
    for(int m = 0; m < scene->num_materials; m += 1)
    {
        const drt_material *mm = &scene->materials[m];
        if(mm->num_lobes < 0 || mm->num_lobes > DRT_MAX_LOBES) return fail(DRT_CUDA_E_ARG, "material %d: %d lobes (0..%d)", m, mm->num_lobes, DRT_MAX_LOBES);
        if(mm->dir_func < DRT_DIR_NONE || mm->dir_func >= DRT_DIR_COUNT) return fail(DRT_CUDA_E_ARG, "material %d: bad dir_func %d", m, mm->dir_func);
        for(int k = 0; k < mm->num_lobes; k += 1)
            if(mm->lobes[k] < -1 || mm->lobes[k] >= DRT_LOBE_COUNT) return fail(DRT_CUDA_E_ARG, "material %d: bad lobe id %d", m, mm->lobes[k]);
    }
    /* a surface that can be hit and shaded needs a direction sampler (the reference calls a NULL pointer there, daily_ray_trace.c:465) */
    for(int i = 0; i < scene->num_surfaces; i += 1)
    {
        const drt_material *mm = &scene->materials[scene->surfaces[i].material];
        if(scene->surfaces[i].type != DRT_GEO_POINT && scene->surfaces[i].type != DRT_GEO_NONE && !mm->is_black_body && mm->dir_func == DRT_DIR_NONE)
            return fail(DRT_CUDA_E_ARG, "surface %d: its material has no dir_func", i);
    }
    return DRT_CUDA_OK;
}

/* The compact records address the D, G blocks with 16-bit word offsets.  The pool of a scene that passes drt_cuda_validate_scene, with
 * rows of npad <= DRT_MAX_HALF_SLOTS * 16 words, holds at most row 0 and one row per material SPD, a D, G block per material and the
 * light's emission in slot pairs (each 16-byte aligned), and three Fresnel rows per orientation of every material but the base one. */
static_assert((1 + DRT_MAX_MATERIALS * DRT_SPD_COUNT) * DRT_MAX_HALF_SLOTS * DRT_HALF
                  + DRT_MAX_MATERIALS * ((DRT_MAX_HALF_SLOTS + 1) / 2 * 4 * DRT_HALF + 3)
                  + ((DRT_MAX_HALF_SLOTS + 1) / 2 * 2 * DRT_HALF + 3)
                  + (DRT_MAX_MATERIALS - 1) * 2 * 3 * DRT_MAX_HALF_SLOTS * DRT_HALF <= 65535,
              "the spectrum pool can outgrow the 16-bit offsets of the compact records");

extern "C" int drt_cuda_upload_scene(drt_cuda_context *ctx, const drt_scene *scene, const drt_camera *camera, const drt_tables *tables)
{
    if(!ctx || !scene || !camera || !tables) return fail(DRT_CUDA_E_ARG, "NULL argument");
    int vrc = drt_cuda_validate_scene(scene);
    if(vrc != DRT_CUDA_OK) return vrc;
    CU(cudaSetDevice(ctx->device));
    const int n = scene->num_wavelengths;

    GeomT<float> *g32 = new GeomT<float>();
    GeomT<double> *g64 = new GeomT<double>();
    fill_geom(g32, scene, camera);
    fill_geom(g64, scene, camera);

    ctx->hit_bound = scene_hit_bound(scene, camera, &ctx->hit_u0, &ctx->hit_u1, &ctx->hit_v0, &ctx->hit_v1);

    /* spectrum pool: row 0 = zeros, then one row per SPD a material was given */
    SpdIndex index;
    memset(&index, 0, sizeof(index));
    /* slots per lane of a half warp (16 lanes): the render kernel is instantiated for 2, 3, 5 and 8 */
    int half_slots = (n + 15) / 16;
    half_slots = half_slots <= 2 ? 2 : half_slots <= 3 ? 3 : half_slots <= 5 ? 5 : 8;
    index.n = n; index.nslots = half_slots; index.npad = ((n + 31) / 32) * 32;
    if(index.npad < half_slots * 16) index.npad = half_slots * 16;
    std::vector<float> pool((size_t)index.npad, 0.f);
    int rows = 1;
    for(int m = 0; m < scene->num_materials; m += 1)
        for(int k = 0; k < DRT_SPD_COUNT; k += 1)
        {
            if(!(scene->materials[m].spd_mask & (1 << k))) continue;
            index.row[m][k] = (rows++) * index.npad;   /* word offset of the row in the pool */
            size_t at = pool.size();
            pool.resize(at + (size_t)index.npad, 0.f);
            for(int i = 0; i < n; i += 1) pool[at + (size_t)i] = (float)scene->materials[m].spd[k][i];
        }
    index.nrows = rows;
    if(g32->nlights == 1)
    {
        /* the D, G blocks of the plastic bounces (SpdIndex::plastic2): every material whose lobes are all bp_diffuse / bp_glossy;
         * a lobe listed k times counts k times (bdsf() sums the lobes, daily_ray_trace.c:215-229) */
        for(int m = 0; m < scene->num_materials; m += 1)
        {
            const drt_material *mm = &scene->materials[m];
            int nd = 0, ng = 0;
            if(mm->is_black_body || classify_material(scene, m, &nd, &ng, nullptr) != DRT_CLASS_PLASTIC) continue;
            auto val = [&](int k, int mult, int slot, int lane) -> float {
                int wl = lane + slot * 16;
                return (wl < n && (mm->spd_mask & (1 << k))) ? (float)((double)mult * mm->spd[k][wl]) : 0.f;
            };
            const int nchunks = (half_slots + 1) / 2;
            size_t at2 = (pool.size() + 3) & ~(size_t)3;
            pool.resize(at2 + (size_t)nchunks * 64, 0.f);
            index.plastic2[m] = (int)at2;
            for(int lane = 0; lane < 16; lane += 1)
                for(int ch = 0; ch < nchunks; ch += 1)
                {
                    float *c = &pool[at2 + ((size_t)ch * 16 + lane) * 4];
                    if(2 * ch + 1 < half_slots)
                    {
                        c[0] = val(DRT_SPD_DIFFUSE, nd, 2 * ch, lane); c[1] = val(DRT_SPD_DIFFUSE, nd, 2 * ch + 1, lane);
                        c[2] = val(DRT_SPD_GLOSSY, ng, 2 * ch, lane);  c[3] = val(DRT_SPD_GLOSSY, ng, 2 * ch + 1, lane);
                    }
                    else { c[0] = val(DRT_SPD_DIFFUSE, nd, 2 * ch, lane); c[1] = val(DRT_SPD_GLOSSY, ng, 2 * ch, lane); }
                }
        }
        /* the light's emission in slot pairs (SpdIndex::light_pairs) */
        const double *emission = scene->materials[scene->surfaces[g32->light_surf[0]].material].spd[DRT_SPD_EMISSION];
        const bool have_e = (scene->materials[scene->surfaces[g32->light_surf[0]].material].spd_mask & (1 << DRT_SPD_EMISSION)) != 0;
        const int nchunks = (half_slots + 1) / 2;
        size_t ate = (pool.size() + 3) & ~(size_t)3;
        pool.resize(ate + (size_t)nchunks * 32, 0.f);
        index.light_pairs = (int)ate;
        for(int lane = 0; lane < 16; lane += 1)
            for(int ch = 0; ch < nchunks; ch += 1)
            {
                float *c = &pool[ate + ((size_t)ch * 16 + lane) * 2];
                int w0 = lane + (2 * ch) * 16, w1 = lane + (2 * ch + 1) * 16;
                c[0] = (w0 < n && have_e) ? (float)emission[w0] : 0.f;
                c[1] = (2 * ch + 1 < half_slots && w1 < n && have_e) ? (float)emission[w1] : 0.f;
            }
    }

    /* Fresnel input rows (SpdIndex::fres) of every material with a refraction spectrum, for both orientations */
    if(scene->materials[scene->base_material].spd_mask & (1 << DRT_SPD_REFRACT))
    {
        const drt_material *bm = &scene->materials[scene->base_material];
        const bool base_k = (bm->spd_mask & (1 << DRT_SPD_EXTINCT)) != 0;
        for(int m = 0; m < scene->num_materials; m += 1)
        {
            const drt_material *mm = &scene->materials[m];
            if(m == scene->base_material || mm->is_black_body || !(mm->spd_mask & (1 << DRT_SPD_REFRACT))) continue;
            const bool own_k = (mm->spd_mask & (1 << DRT_SPD_EXTINCT)) != 0;
            for(int side = 0; side < 2; side += 1)
                for(int k = 0; k < 3; k += 1)
                {
                    size_t at = pool.size();
                    pool.resize(at + (size_t)index.npad, 0.f);
                    index.fres[m][side][k] = (int)at;
                    for(int i = 0; i < n; i += 1)
                    {
                        /* side 0: incident = base medium, transmitting = this material; side 1: the other way round (Q11) */
                        const double ir = side ? mm->spd[DRT_SPD_REFRACT][i] : bm->spd[DRT_SPD_REFRACT][i];
                        const double tr = side ? bm->spd[DRT_SPD_REFRACT][i] : mm->spd[DRT_SPD_REFRACT][i];
                        const double te = side ? (base_k ? bm->spd[DRT_SPD_EXTINCT][i] : 0.0) : (own_k ? mm->spd[DRT_SPD_EXTINCT][i] : 0.0);
                        const double eta = tr / ir, kap = te / ir;
                        pool[at + (size_t)i] = (float)(k == 0 ? ir / tr : k == 1 ? eta * eta - kap * kap : 4.0 * eta * eta * kap * kap);
                    }
                }
        }
    }

    std::vector<unsigned char> rgbt(drt_rgb_tables_bytes());
    drt_fill_rgb_tables(rgbt.data(), tables);

    /* the fixed-size blocks are allocated once per context; the pool only grows (a re-upload per frame costs five small copies) */
    ctx->have_scene = false;
    cudaError_t e = cudaSuccess;
    if(e == cudaSuccess && !ctx->d_geom32) e = cudaMalloc(&ctx->d_geom32, sizeof(GeomT<float>));
    if(e == cudaSuccess && !ctx->d_geom64) e = cudaMalloc(&ctx->d_geom64, sizeof(GeomT<double>));
    if(e == cudaSuccess && !ctx->d_index) e = cudaMalloc(&ctx->d_index, sizeof(SpdIndex));
    if(e == cudaSuccess && !ctx->d_rgb_tables) e = cudaMalloc(&ctx->d_rgb_tables, rgbt.size());
    if(e == cudaSuccess && ctx->pool_capacity < pool.size() * 4)
    {
        cudaFree(ctx->d_pool); ctx->d_pool = nullptr; ctx->pool_capacity = 0;
        e = cudaMalloc(&ctx->d_pool, pool.size() * 4);
        if(e == cudaSuccess) ctx->pool_capacity = pool.size() * 4;
    }
    if(e == cudaSuccess) e = cudaMemcpy(ctx->d_geom32, g32, sizeof(GeomT<float>), cudaMemcpyHostToDevice);
    if(e == cudaSuccess) e = cudaMemcpy(ctx->d_geom64, g64, sizeof(GeomT<double>), cudaMemcpyHostToDevice);
    if(e == cudaSuccess) e = cudaMemcpy(ctx->d_index, &index, sizeof(index), cudaMemcpyHostToDevice);
    if(e == cudaSuccess) e = cudaMemcpy(ctx->d_pool, pool.data(), pool.size() * 4, cudaMemcpyHostToDevice);
    if(e == cudaSuccess) e = cudaMemcpy(ctx->d_rgb_tables, rgbt.data(), rgbt.size(), cudaMemcpyHostToDevice);
    int nlights = g32->nlights;
    int eval_words = g32->eval_words > 0 ? g32->eval_words : 1;
    delete g32; delete g64;
    if(e != cudaSuccess) return fail(DRT_CUDA_E_CUDA, "scene upload: %s", cudaGetErrorString(e));
    ctx->n = n; ctx->nslots = index.nslots; ctx->nlights = nlights; ctx->eval_words = eval_words; ctx->scene_mode = scene_kernel_mode(scene); ctx->pool_words = (uint32_t)pool.size();
    ctx->upload_bytes = sizeof(GeomT<float>) + sizeof(GeomT<double>) + sizeof(SpdIndex) + pool.size() * 4 + rgbt.size();
    ctx->have_scene = true;
    return DRT_CUDA_OK;
}

extern "C" int drt_cuda_scene_upload_bytes(const drt_cuda_context *ctx, size_t *bytes)
{
    if(!ctx || !bytes) return fail(DRT_CUDA_E_ARG, "NULL argument");
    *bytes = ctx->upload_bytes;
    return DRT_CUDA_OK;
}

extern "C" int drt_cuda_set_geometry_precision(drt_cuda_context *ctx, int precision)
{
    if(!ctx || (precision != DRT_GEOMETRY_F32 && precision != DRT_GEOMETRY_F64)) return fail(DRT_CUDA_E_ARG, "bad precision");
    ctx->f64_geometry = precision == DRT_GEOMETRY_F64;
    return DRT_CUDA_OK;
}

extern "C" int drt_cuda_film_sizes(const drt_cuda_context *ctx, uint32_t width, uint32_t height, size_t *spectral, size_t *filter)
{
    if(!ctx || !ctx->have_scene) return fail(DRT_CUDA_E_STATE, "upload a scene first");
    if(spectral) *spectral = (size_t)width * height * (size_t)ctx->n * 4;
    if(filter) *filter = (size_t)width * height * 4;
    return DRT_CUDA_OK;
}

/* which instantiation of the render kernel serves the uploaded scene: 0 general (any lobe list, any number of lights; always for the
 * f64-geometry diagnostic), 1 plastic-only, 2 classed (drt_render.cuh) */
static int kernel_mode(const drt_cuda_context *ctx) { return ctx->f64_geometry ? 0 : ctx->scene_mode; }

/* record layout of a render with `max_depth` bounces (RenderLaunch in drt_device.cuh) */
static void record_layout(const drt_cuda_context *ctx, uint32_t max_depth, uint32_t smem_depth, RenderLaunch &L)
{
    L.eval_words = (uint32_t)ctx->eval_words;
    const bool compact = kernel_mode(ctx) != 0;   /* the plastic-only and the classed kernel and their compact records */
    L.bounce_words = (2 + (uint32_t)ctx->nlights * (L.eval_words + 1) + L.eval_words + 3u) & ~3u;
    if(L.bounce_words < 8) L.bounce_words = 8;
    L.head_words = 4;
    if(smem_depth > max_depth) smem_depth = max_depth;
    if(compact) { L.bounce_words = 4; L.head_words = (2 + (smem_depth + 1) / 2 + 3u) & ~3u; }
    L.smem_depth = smem_depth;
    L.path_words = L.head_words + smem_depth * L.bounce_words;      /* the shared-memory part of a record */
    L.path_stride = ((L.path_words / 4) & 1u) ? L.path_words : L.path_words + 4;
    /* bounces past smem_depth: the slot's overflow row in global memory (RenderLaunch::deep) */
    const uint32_t over = max_depth - smem_depth;
    L.deep_hdr_off = over * L.bounce_words;
    L.deep_stride = over ? ((L.deep_hdr_off + (compact ? (over + 1) / 2 : 0u) + 4u + 3u) & ~3u) : 0u;
}

/* Path records live in shared memory.  A record holds as many bounces as fit with the kernel's full number of warps and CTAs per SM
 * (smem_depth); deeper bounces overflow to global memory, so neither max_cast_depth nor the number of lights limits a render
 * (cast_ray loops `depth < max_depth` without a bound, daily_ray_trace.c:446).  whole = true (record dumps): the whole record must
 * sit in shared memory, with fewer warps per CTA if need be.  Fills in L's pool size and record layout (path_words and the rest). */
static bool launch_shape(const drt_cuda_context *ctx, uint32_t max_depth, bool whole, RenderLaunch &L, int *warps_out, int *ctas_out, size_t *smem_out)
{
    const RenderShape &shape = DRT_RENDER_SHAPE[kernel_mode(ctx)];
    const int full_warps = shape.warps, want_ctas = shape.min_ctas;
    L.pool_words = ctx->pool_words;
    auto bytes = [&](uint32_t depth, int warps) { record_layout(ctx, max_depth, depth, L); return drt_render_smem_bytes(L, ctx->f64_geometry, warps, ctx->nslots); };
    int warps = full_warps;
    uint32_t depth = max_depth;
    const size_t per_cta = (size_t)(227 * 1024) / (size_t)want_ctas - 1024;
    if(!whole && max_depth > 1 && bytes(max_depth, warps) > per_cta)
    {
        uint32_t lo = 1, hi = max_depth;          /* largest depth whose records fit with full occupancy (bytes() grows with depth) */
        while(lo < hi) { uint32_t mid = (lo + hi + 1) / 2; if(bytes(mid, warps) <= per_cta) lo = mid; else hi = mid - 1; }
        depth = lo;
    }
    size_t smem = bytes(depth, warps);
    while(smem > ctx->smem_optin && warps > 1) { warps /= 2; smem = bytes(depth, warps); }
    *warps_out = warps; *smem_out = smem;
    if(smem > ctx->smem_optin) return false;
    int ctas_per_sm = (int)((size_t)(227 * 1024) / (smem + 1024));
    int by_threads = (want_ctas * full_warps) / warps;
    if(ctas_per_sm > by_threads) ctas_per_sm = by_threads;
    if(ctas_per_sm < 1) ctas_per_sm = 1;
    *ctas_out = ctas_per_sm;
    return true;
}

extern "C" int drt_cuda_render_kernel_info(drt_cuda_context *ctx, const drt_render_params *params, char *name, size_t name_len, int *warps_per_cta, int *ctas_per_sm)
{
    if(!ctx || !params || params->sample_end <= params->sample_begin) return fail(DRT_CUDA_E_ARG, "bad argument");
    const uint32_t max_depth = params->max_depth;
    if(!ctx->have_scene) return fail(DRT_CUDA_E_STATE, "upload a scene first");
    RenderLaunch L;
    memset(&L, 0, sizeof(L));
    int warps = 0, ctas = 0;
    size_t smem = 0;
    if(!launch_shape(ctx, max_depth, false, L, &warps, &ctas, &smem)) return fail(DRT_CUDA_E_UNSUPPORTED, "one bounce record of this scene does not fit in shared memory");
    if(name && name_len)
        snprintf(name, name_len, "drt::render_kernel<%s,%d,%d,%s,%s>", ctx->f64_geometry ? "double" : "float", ctx->nslots,
                 kernel_mode(ctx), (params->sample_end - params->sample_begin >= 32) ? "true" : "false", L.deep_stride ? "true" : "false");
    if(warps_per_cta) *warps_per_cta = warps;
    if(ctas_per_sm) *ctas_per_sm = ctas;
    return DRT_CUDA_OK;
}

/* starts the work counters of a public call: the next block of the ring, zeroed on `stream` (drt_cuda_get_stats reads the latest) */
static int begin_call(drt_cuda_context *ctx, cudaStream_t stream)
{
    ctx->d_stats = ctx->d_stats_ring + (ctx->stats_calls++ % DRT_RING);
    CU(cudaMemsetAsync(ctx->d_stats, 0, sizeof(DeviceStats), stream));
    return DRT_CUDA_OK;
}

static int launch(drt_cuda_context *ctx, const drt_render_params *p, uint32_t x0, uint32_t y0, uint32_t x1, uint32_t y1,
                  FilmPtrs film, float *dump, int accumulate, cudaStream_t stream, float *record_dump = nullptr,
                  const drt_film *scatter = nullptr, int scatter_count = 0, int scatter_rank = 0, uint64_t scatter_slice = 0, bool keep_stats = false,
                  uint64_t band_begin = 0, uint64_t band_end = 0, const drt_adaptive *adaptive = nullptr, int rows_count = 0, int rows_rank = 0)
{
    if(!ctx->have_scene) return fail(DRT_CUDA_E_STATE, "upload a scene first");
    if(p->width == 0 || p->height == 0 || x1 > p->width || y1 > p->height || x0 >= x1 || y0 >= y1) return fail(DRT_CUDA_E_ARG, "bad image rectangle");
    if(p->sample_end < p->sample_begin) return fail(DRT_CUDA_E_ARG, "bad sample range [%u,%u)", p->sample_begin, p->sample_end);
    CU(cudaSetDevice(ctx->device));
    /* a row shard (adaptive only) of a rank without rows: no launch (a grid of 0 is an error), and the call's counters read zero */
    uint32_t shard_rows = 0;
    if(rows_count && (uint32_t)rows_rank < p->height) shard_rows = (p->height - (uint32_t)rows_rank + (uint32_t)rows_count - 1) / (uint32_t)rows_count;
    if(rows_count && shard_rows == 0)
    {
        int rc = begin_call(ctx, stream);
        if(rc != DRT_CUDA_OK) return rc;
        ctx->last_launches = 0;
        return DRT_CUDA_OK;
    }
    if(p->sample_end == p->sample_begin)
    {
        /* num_pixel_samples 0: render_image's sample loop does not run (daily_ray_trace.c:710) and the films stay as allocated, all zero */
        int rc = keep_stats ? DRT_CUDA_OK : begin_call(ctx, stream);
        if(rc != DRT_CUDA_OK) return rc;
        ctx->last_launches = 0;
        if(film.sum && !accumulate && scatter_count == 0)
        {
            const size_t n = (size_t)ctx->n, w = p->width;
            if(x0 != 0 || x1 != p->width) return fail(DRT_CUDA_E_ARG, "empty sample range on a partial-width rectangle");
            const size_t at = (size_t)y0 * w, cnt = (size_t)(y1 - y0) * w;
            CU(cudaMemsetAsync(film.sum + at * n, 0, cnt * n * 4, stream)); CU(cudaMemsetAsync(film.mean + at * n, 0, cnt * n * 4, stream));
            CU(cudaMemsetAsync(film.m2 + at * n, 0, cnt * n * 4, stream));  CU(cudaMemsetAsync(film.filter + at, 0, cnt * 4, stream));
        }
        return DRT_CUDA_OK;
    }
    RenderLaunch L;
    memset(&L, 0, sizeof(L));
    L.geom = ctx->f64_geometry ? ctx->d_geom64 : ctx->d_geom32;
    L.spd_index = ctx->d_index; L.pool = ctx->d_pool;
    L.film = film; L.path_dump = dump; L.record_dump = record_dump;
    L.width = p->width; L.height = p->height; L.x0 = x0; L.y0 = y0; L.x1 = x1; L.y1 = y1;
    L.sample_begin = p->sample_begin; L.sample_end = p->sample_end; L.max_depth = p->max_depth;
    L.pixel_scheme = p->pixel_scheme; L.seed = p->seed; L.accumulate = accumulate; L.nlights = ctx->nlights;
    uint32_t spp = p->sample_end - p->sample_begin;
    L.pixels_per_task = spp >= 32 ? 1 : 32 / spp;
    for(int i = 0; i < scatter_count; i += 1) L.scatter[i] = film_ptrs(scatter[i]);
    L.scatter_count = (uint32_t)scatter_count; L.scatter_rank = (uint32_t)scatter_rank; L.scatter_slice = (uint32_t)scatter_slice;
    uint32_t rect[4];
    /* max_cast_depth 0 casts no ray at all (cast_ray's loop, daily_ray_trace.c:446): nothing to cull, and the culled pixels' "one closest-hit ray" must not be counted */
    hit_rect(ctx->hit_bound && p->max_depth > 0, ctx->hit_u0, ctx->hit_u1, ctx->hit_v0, ctx->hit_v1, p->width, p->height, rect);
    L.hit_x0 = rect[0]; L.hit_y0 = rect[1]; L.hit_x1 = rect[2]; L.hit_y1 = rect[3];
    if(adaptive)   /* checked by adaptive_args: f32 geometry, >= 32 samples (one pixel per task), no scatter */
    {
        L.adaptive = 1; L.rel_error = adaptive->rel_error; L.min_samples = adaptive->min_samples;
        L.luminance_w = reinterpret_cast<const float *>(static_cast<const unsigned char *>(ctx->d_rgb_tables) + drt_rgb_tables_yw_offset());
    }
    /* record dumps (diagnostics) want the whole record in shared memory; renders keep full occupancy and let deep bounces overflow */
    const bool whole = record_dump != nullptr;
    int warps, ctas_per_sm;
    size_t smem;
    if(!launch_shape(ctx, p->max_depth, whole, L, &warps, &ctas_per_sm, &smem))
        return fail(DRT_CUDA_E_UNSUPPORTED, "%s: max_cast_depth %u with %d lights needs %zu bytes of shared memory per warp (limit %zu)",
                    whole ? "record dump" : "render", p->max_depth, ctx->nlights, smem, ctx->smem_optin);
    uint64_t npix = (uint64_t)(x1 - x0) * (y1 - y0);
    const bool band = band_end > band_begin;
    if(band)
    {
        if(L.pixels_per_task != 1 || scatter_count < 1 || band_end > scatter_slice || x0 != 0 || y0 != 0 || x1 != p->width || y1 != p->height)
            return fail(DRT_CUDA_E_ARG, "a band needs a scattered whole-frame render with at least 32 samples per pixel");
        L.band_chunk = (uint32_t)(band_end - band_begin); L.band_period = (uint32_t)scatter_slice; L.band_base = (uint32_t)band_begin;
    }
    if(rows_count)   /* checked by drt_cuda_render_device_adaptive_rows: an adaptive whole-frame render, no scatter, no band */
    {
        L.band_chunk = p->width; L.band_period = (uint32_t)rows_count * p->width; L.band_base = (uint32_t)rows_rank * p->width;
        L.row_tasks = p->width * shard_rows;
    }
    uint64_t ntasks = band ? (uint64_t)L.band_chunk * scatter_count : rows_count ? (uint64_t)L.row_tasks : (npix + L.pixels_per_task - 1) / L.pixels_per_task;
    if(scatter_count > 1)
        L.task_rotate = band ? (uint32_t)(((uint64_t)scatter_rank * L.band_chunk) % ntasks)
                             : (uint32_t)((((uint64_t)scatter_rank * scatter_slice) / L.pixels_per_task) % ntasks);
    uint64_t grid = (uint64_t)ctx->num_sms * ctas_per_sm;
    uint64_t need = (ntasks + warps - 1) / warps;
    if(grid > need) grid = need;
    if(L.deep_stride)
    {
        /* overflow rows of every resident warp; the buffer only grows.  (Renders of one context that are in flight on different
         * streams would share it: deep renders are one at a time per context.) */
        const size_t need_bytes = (size_t)grid * (size_t)warps * DRT_WARP * L.deep_stride * 4;
        int rc = drt_ensure_buffer(&ctx->d_deep, &ctx->deep_bytes, need_bytes);
        if(rc != DRT_CUDA_OK) return rc;
        L.deep = ctx->d_deep;
    }
    int rc = keep_stats ? DRT_CUDA_OK : begin_call(ctx, stream);
    if(rc != DRT_CUDA_OK) return rc;
    L.stats = ctx->d_stats;
    L.task_counter = ctx->d_counter_ring + (ctx->counter_launches++ % DRT_RING);
    CU(cudaMemsetAsync(L.task_counter, 0, sizeof(unsigned int), stream));
    cudaError_t e = drt_launch_render(L, ctx->f64_geometry, kernel_mode(ctx), ctx->nslots, (int)grid, warps, smem, stream);
    if(e != cudaSuccess) return fail(DRT_CUDA_E_CUDA, "render kernel launch: %s", cudaGetErrorString(e));
    ctx->launches += 1;
    ctx->last_launches = 1;
    return DRT_CUDA_OK;
}

extern "C" int drt_cuda_render_device(drt_cuda_context *ctx, const drt_render_params *params, const drt_film *film, int accumulate, void *stream)
{
    if(!ctx || !params || !film_complete(film)) return fail(DRT_CUDA_E_ARG, "NULL argument");
    return launch(ctx, params, 0, 0, params->width, params->height, film_ptrs(*film), nullptr, accumulate, (cudaStream_t)stream);
}

extern "C" int drt_cuda_render_device_scatter(drt_cuda_context *ctx, const drt_render_params *params, const drt_film *staging, int count, int rank,
                                              uint64_t slice_pixels, void *stream)
{
    if(!ctx || !params || !staging || count < 1 || count > DRT_MAX_PEERS || rank < 0 || rank >= count) return fail(DRT_CUDA_E_ARG, "bad argument (1..%d staging films)", DRT_MAX_PEERS);
    uint64_t npix = (uint64_t)params->width * params->height;
    if(slice_pixels == 0 || slice_pixels * (uint64_t)count < npix || slice_pixels > 0xffffffffull) return fail(DRT_CUDA_E_ARG, "slices of %llu pixels do not cover the image", (unsigned long long)slice_pixels);
    for(int i = 0; i < count; i += 1)
        if(!film_complete(&staging[i])) return fail(DRT_CUDA_E_ARG, "NULL staging film %d", i);
    return launch(ctx, params, 0, 0, params->width, params->height, film_ptrs(staging[0]), nullptr, 0, (cudaStream_t)stream, nullptr, staging, count, rank, slice_pixels);
}

extern "C" int drt_cuda_render_device_scatter_band(drt_cuda_context *ctx, const drt_render_params *params, const drt_film *staging, int count, int rank,
                                                   uint64_t slice_pixels, uint64_t band_begin, uint64_t band_end, int keep_stats, void *stream)
{
    if(!ctx || !params || !staging || count < 1 || count > DRT_MAX_PEERS || rank < 0 || rank >= count) return fail(DRT_CUDA_E_ARG, "bad argument (1..%d staging films)", DRT_MAX_PEERS);
    uint64_t npix = (uint64_t)params->width * params->height;
    if(slice_pixels == 0 || slice_pixels * (uint64_t)count < npix || slice_pixels > 0xffffffffull) return fail(DRT_CUDA_E_ARG, "slices of %llu pixels do not cover the image", (unsigned long long)slice_pixels);
    if(band_begin >= band_end || band_end > slice_pixels) return fail(DRT_CUDA_E_ARG, "bad band [%llu, %llu) of a slice of %llu pixels", (unsigned long long)band_begin, (unsigned long long)band_end, (unsigned long long)slice_pixels);
    for(int i = 0; i < count; i += 1)
        if(!film_complete(&staging[i])) return fail(DRT_CUDA_E_ARG, "NULL staging film %d", i);
    return launch(ctx, params, 0, 0, params->width, params->height, film_ptrs(staging[0]), nullptr, 0, (cudaStream_t)stream, nullptr, staging, count, rank, slice_pixels,
                  keep_stats != 0, band_begin, band_end);
}

int drt_ensure_buffer(float **buf, size_t *have, size_t need)
{
    if(*have >= need) return DRT_CUDA_OK;
    cudaFree(*buf); *buf = nullptr; *have = 0;
    CU(cudaMalloc(buf, need));
    *have = need;
    return DRT_CUDA_OK;
}

int drt_library_film(const drt_cuda_context *ctx, float **buf, size_t *have, size_t npix, drt_film *out)
{
    int rc = drt_ensure_buffer(buf, have, (3 * npix * (size_t)ctx->n + npix) * 4);
    if(rc != DRT_CUDA_OK) return rc;
    *out = film_planes(*buf, npix, ctx->n);
    return DRT_CUDA_OK;
}

/* argument checks of the adaptive entry points (drt_cuda.h) */
static int adaptive_args(const drt_cuda_context *ctx, const drt_render_params *p, const drt_adaptive *a)
{
    if(!ctx->have_scene) return fail(DRT_CUDA_E_STATE, "upload a scene first");
    if(p->sample_end < p->sample_begin) return fail(DRT_CUDA_E_ARG, "bad sample range [%u,%u)", p->sample_begin, p->sample_end);
    const uint32_t range = p->sample_end - p->sample_begin;
    if(!(a->rel_error > 0.f) || !isfinite(a->rel_error))
        return fail(DRT_CUDA_E_ARG, "adaptive sampling: rel_error must be a finite number > 0 (got %g)", (double)a->rel_error);
    if(a->min_samples < 32u || a->min_samples > range)
        return fail(DRT_CUDA_E_ARG, "adaptive sampling: min_samples must lie in [32, %u], the call's sample range [%u,%u) (got %u); "
                    "a pixel is checked after each batch of 32 samples, so the range needs at least 32", range, p->sample_begin, p->sample_end, a->min_samples);
    if(ctx->f64_geometry)
        return fail(DRT_CUDA_E_UNSUPPORTED, "adaptive sampling runs with f32 geometry only: f64 geometry is the branch-flip diagnostic and has no adaptive kernel");
    return DRT_CUDA_OK;
}

extern "C" int drt_cuda_render_device_adaptive(drt_cuda_context *ctx, const drt_render_params *params, const drt_adaptive *adaptive,
                                               const drt_film *film, int accumulate, void *stream)
{
    if(!ctx || !params || !adaptive || !film_complete(film)) return fail(DRT_CUDA_E_ARG, "NULL argument");
    int rc = adaptive_args(ctx, params, adaptive);
    if(rc != DRT_CUDA_OK) return rc;
    return launch(ctx, params, 0, 0, params->width, params->height, film_ptrs(*film), nullptr, accumulate, (cudaStream_t)stream, nullptr, nullptr, 0, 0, 0, false, 0, 0, adaptive);
}

extern "C" int drt_cuda_render_device_adaptive_rows(drt_cuda_context *ctx, const drt_render_params *params, const drt_adaptive *adaptive,
                                                    const drt_film *film, int accumulate, int count, int rank, void *stream)
{
    if(!ctx || !params || !adaptive || !film_complete(film)) return fail(DRT_CUDA_E_ARG, "NULL argument");
    if(count < 1 || count > DRT_MAX_PEERS || rank < 0 || rank >= count) return fail(DRT_CUDA_E_ARG, "bad row shard: rank %d of %d (1..%d ranks)", rank, count, DRT_MAX_PEERS);
    int rc = adaptive_args(ctx, params, adaptive);
    if(rc != DRT_CUDA_OK) return rc;
    return launch(ctx, params, 0, 0, params->width, params->height, film_ptrs(*film), nullptr, accumulate, (cudaStream_t)stream, nullptr, nullptr, 0, 0, 0, false, 0, 0,
                  adaptive, count, rank);
}

/* the non-blocking streams (and events) of render_host's banded read-back, created on first use */
static int band_streams(drt_cuda_context *ctx)
{
    if(ctx->band_render) return DRT_CUDA_OK;
    CU(cudaStreamCreateWithFlags(&ctx->band_render, cudaStreamNonBlocking));
    CU(cudaStreamCreateWithFlags(&ctx->band_copy, cudaStreamNonBlocking));
    for(int i = 0; i < 16; i += 1) CU(cudaEventCreateWithFlags(&ctx->band_done[i], cudaEventDisableTiming));
    return DRT_CUDA_OK;
}

/* render_host and render_host_adaptive (adaptive != NULL) */
static int render_host(drt_cuda_context *ctx, const drt_render_params *params, const drt_adaptive *adaptive, const drt_film *out)
{
    if(!ctx || !params || !film_complete(out)) return fail(DRT_CUDA_E_ARG, "NULL argument");
    if(!ctx->have_scene) return fail(DRT_CUDA_E_STATE, "upload a scene first");
    CU(cudaSetDevice(ctx->device));
    size_t npix = (size_t)params->width * params->height;
    drt_film f;
    int rc = drt_library_film(ctx, &ctx->d_film, &ctx->film_bytes, npix, &f);
    if(rc != DRT_CUDA_OK) return rc;
    /* Large frames are rendered in row bands so that the read-back of a finished band (PCIe) runs under the render of the
     * next one: with pinned host buffers only the last (small) band's copy is exposed.  Rows are contiguous in every plane. */
    const uint64_t paths = (uint64_t)npix * (params->sample_end - params->sample_begin);
    /* band boundaries in 1/16 of the image height: three quarters, then ever smaller bands, so that the copy left exposed
     * after the last render is 1/16 of the film */
    static const int cut[] = { 0, 4, 8, 12, 14, 15, 16 };
    int bands = (paths >= (1ull << 26) && params->height >= 64) ? 6 : 1;
    if(bands > 1)
    {
        rc = band_streams(ctx);
        if(rc != DRT_CUDA_OK) return rc;
    }
    cudaStream_t sr = bands > 1 ? ctx->band_render : 0, sc = bands > 1 ? ctx->band_copy : 0;
    if(bands > 1) CU(cudaDeviceSynchronize());   /* the band streams do not synchronise with the legacy stream */
    const size_t n = (size_t)ctx->n, w = params->width;
    for(int b = 0; b < bands; b += 1)
    {
        const uint32_t y0 = bands > 1 ? (uint32_t)((uint64_t)params->height * cut[b] / 16) : 0u;
        const uint32_t y1 = bands > 1 ? (uint32_t)((uint64_t)params->height * cut[b + 1] / 16) : params->height;
        rc = launch(ctx, params, 0, y0, params->width, y1, film_ptrs(f), nullptr, 0, sr, nullptr, nullptr, 0, 0, 0, b > 0, 0, 0, adaptive);
        if(rc != DRT_CUDA_OK) return rc;
        if(bands > 1) { CU(cudaEventRecord(ctx->band_done[b], sr)); CU(cudaStreamWaitEvent(sc, ctx->band_done[b], 0)); }
        const size_t at = (size_t)y0 * w * n, cnt = (size_t)(y1 - y0) * w * n * 4;
        CU(cudaMemcpyAsync(out->sum + at, f.sum + at, cnt, cudaMemcpyDeviceToHost, sc));
        CU(cudaMemcpyAsync(out->mean + at, f.mean + at, cnt, cudaMemcpyDeviceToHost, sc));
        CU(cudaMemcpyAsync(out->m2 + at, f.m2 + at, cnt, cudaMemcpyDeviceToHost, sc));
        CU(cudaMemcpyAsync(out->filter + (size_t)y0 * w, f.filter + (size_t)y0 * w, (size_t)(y1 - y0) * w * 4, cudaMemcpyDeviceToHost, sc));
    }
    ctx->last_launches = (uint64_t)bands;
    if(bands > 1) { CU(cudaStreamSynchronize(sr)); CU(cudaStreamSynchronize(sc)); }
    CU(cudaStreamSynchronize(0));
    return DRT_CUDA_OK;
}

extern "C" int drt_cuda_render_host(drt_cuda_context *ctx, const drt_render_params *params, const drt_film *out)
{
    return render_host(ctx, params, nullptr, out);
}

extern "C" int drt_cuda_render_host_adaptive(drt_cuda_context *ctx, const drt_render_params *params, const drt_adaptive *adaptive, const drt_film *out)
{
    if(!ctx || !params || !adaptive) return fail(DRT_CUDA_E_ARG, "NULL argument");
    int rc = adaptive_args(ctx, params, adaptive);
    if(rc != DRT_CUDA_OK) return rc;
    return render_host(ctx, params, adaptive, out);
}

/* Every pixel's samples stay on the device that renders its row, so its stopping rule sees its whole film and nothing is merged:
 * device g renders rows y = g (mod count) into its own full-frame film and copies them to out on the same stream.  All renders are
 * queued before any copy. */
extern "C" int drt_cuda_render_host_multi_adaptive(drt_cuda_context **ctxs, int count, const drt_render_params *params, const drt_adaptive *adaptive,
                                                   const drt_film *out)
{
    if(!ctxs || count < 1 || count > DRT_MAX_PEERS || !params || !adaptive || !film_complete(out))
        return fail(DRT_CUDA_E_ARG, "bad argument (1..%d contexts)", DRT_MAX_PEERS);
    for(int g = 0; g < count; g += 1)
    {
        if(!ctxs[g]) return fail(DRT_CUDA_E_ARG, "context %d is NULL", g);
        int rc = adaptive_args(ctxs[g], params, adaptive);
        if(rc != DRT_CUDA_OK) return rc;
        if(ctxs[g]->n != ctxs[0]->n) return fail(DRT_CUDA_E_ARG, "context %d holds another scene", g);
        for(int h = 0; h < g; h += 1) if(ctxs[h]->device == ctxs[g]->device) return fail(DRT_CUDA_E_ARG, "contexts %d and %d share device %d", h, g, ctxs[g]->device);
    }
    const size_t npix = (size_t)params->width * params->height;
    if(npix == 0) return fail(DRT_CUDA_E_ARG, "bad image rectangle");
    int rc = DRT_CUDA_OK;
    drt_film films[DRT_MAX_PEERS];   /* device g's full-frame film */
    for(int g = 0; g < count && rc == DRT_CUDA_OK; g += 1)
    {
        drt_cuda_context *ctx = ctxs[g];
        if((uint32_t)g >= params->height)
        {
            /* a surplus device: no rows, no launch; its counters read zero */
            rc = launch(ctx, params, 0, 0, params->width, params->height, FilmPtrs{}, nullptr, 0, 0, nullptr, nullptr, 0, 0, 0, false, 0, 0, adaptive, count, g);
            continue;
        }
        if(cudaSetDevice(ctx->device) != cudaSuccess) { rc = fail(DRT_CUDA_E_CUDA, "cudaSetDevice(%d)", ctx->device); break; }
        rc = drt_library_film(ctx, &ctx->d_film, &ctx->film_bytes, npix, &films[g]);
        if(rc == DRT_CUDA_OK) rc = band_streams(ctx);
        /* the non-blocking stream does not wait for work of this context on the legacy stream */
        if(rc == DRT_CUDA_OK && cudaDeviceSynchronize() != cudaSuccess) rc = fail(DRT_CUDA_E_CUDA, "device %d: %s", ctx->device, cudaGetErrorString(cudaGetLastError()));
        if(rc != DRT_CUDA_OK) break;
        rc = drt_cuda_render_device_adaptive_rows(ctx, params, adaptive, &films[g], 0, count, g, ctx->band_render);
    }
    /* The read-backs are queued only once every device renders: a copy into pageable host memory returns when it has finished, so
     * queued right after its own render it would hold the host, and the renders of the devices after it, until that render ends. */
    for(int g = 0; g < count && (uint32_t)g < params->height && rc == DRT_CUDA_OK; g += 1)
        rc = drt_cuda_film_read_rows(ctxs[g], &films[g], params->width, params->height, count, g, out, ctxs[g]->band_render);
    for(int g = 0; g < count && (uint32_t)g < params->height; g += 1)
    {
        if(!ctxs[g]->band_render || cudaSetDevice(ctxs[g]->device) != cudaSuccess) continue;
        if(cudaStreamSynchronize(ctxs[g]->band_render) != cudaSuccess && rc == DRT_CUDA_OK)
            rc = fail(DRT_CUDA_E_CUDA, "device %d: %s", ctxs[g]->device, cudaGetErrorString(cudaGetLastError()));
    }
    return rc;
}

extern "C" int drt_cuda_get_stats(drt_cuda_context *ctx, drt_cuda_stats *out)
{
    if(!ctx || !out) return fail(DRT_CUDA_E_ARG, "NULL argument");
    CU(cudaSetDevice(ctx->device));
    CU(cudaDeviceSynchronize());
    DeviceStats s;
    CU(cudaMemcpy(&s, ctx->d_stats, sizeof(s), cudaMemcpyDeviceToHost));
    memset(out, 0, sizeof(*out));
    out->paths = s.paths; out->closest_rays = s.closest_rays; out->shadow_rays = s.shadow_rays;
    out->shaded_bounces = s.shaded_bounces; out->rng_draws = s.rng_draws;
    for(int i = 0; i < 8; i += 1) out->terminated_at_depth[i] = s.terminated_at_depth[i];
    out->reached_depth_cap = s.reached_depth_cap;
    out->kernel_launches = ctx->last_launches;
    return DRT_CUDA_OK;
}

#ifdef DRT_PHASE_CLOCKS
/* Diagnostic builds only (tools/phase_split.py): the warp cycles of the last render call by part of a batch -- trace, batch
 * bookkeeping, replay, other (DRT_PHASE_* in drt_render.cuh).  Not part of include/drt_cuda.h. */
extern "C" int drt_cuda_phase_clocks(drt_cuda_context *ctx, uint64_t out[4])
{
    if(!ctx || !out) return fail(DRT_CUDA_E_ARG, "NULL argument");
    CU(cudaSetDevice(ctx->device));
    CU(cudaDeviceSynchronize());
    DeviceStats s;
    CU(cudaMemcpy(&s, ctx->d_stats, sizeof(s), cudaMemcpyDeviceToHost));
    for(int i = 0; i < 4; i += 1) out[i] = s.phase_clocks[i];
    return DRT_CUDA_OK;
}
#endif

extern "C" int drt_cuda_sample_paths(drt_cuda_context *ctx, const drt_render_params *params,
                                     uint32_t x0, uint32_t y0, uint32_t x1, uint32_t y1, float *out_host)
{
    if(!ctx || !params || !out_host) return fail(DRT_CUDA_E_ARG, "NULL argument");
    if(!ctx->have_scene) return fail(DRT_CUDA_E_STATE, "upload a scene first");
    if(x1 <= x0 || y1 <= y0 || params->sample_end <= params->sample_begin) return fail(DRT_CUDA_E_ARG, "empty rectangle or sample range");
    CU(cudaSetDevice(ctx->device));
    size_t bytes = (size_t)(x1 - x0) * (y1 - y0) * (params->sample_end - params->sample_begin) * (size_t)ctx->n * 4;
    int rc = drt_ensure_buffer(&ctx->d_dump, &ctx->dump_bytes, bytes);
    if(rc != DRT_CUDA_OK) return rc;
    rc = launch(ctx, params, x0, y0, x1, y1, FilmPtrs{}, ctx->d_dump, 0, 0);
    if(rc != DRT_CUDA_OK) return rc;
    CU(cudaMemcpy(out_host, ctx->d_dump, bytes, cudaMemcpyDeviceToHost));
    return DRT_CUDA_OK;
}

extern "C" int drt_cuda_debug_records(drt_cuda_context *ctx, const drt_render_params *params, uint32_t x0, uint32_t y0, uint32_t x1, uint32_t y1,
                                      float *out_host, size_t out_capacity_words, uint32_t *words_per_path)
{
    if(!ctx || !params || !words_per_path) return fail(DRT_CUDA_E_ARG, "NULL argument");
    if(!ctx->have_scene) return fail(DRT_CUDA_E_STATE, "upload a scene first");
    if(x1 <= x0 || y1 <= y0 || params->sample_end <= params->sample_begin) return fail(DRT_CUDA_E_ARG, "empty rectangle or sample range");
    CU(cudaSetDevice(ctx->device));
    if(x1 > params->width || y1 > params->height) return fail(DRT_CUDA_E_ARG, "bad image rectangle");
    RenderLaunch L;
    memset(&L, 0, sizeof(L));
    int warps, ctas;
    size_t smem;
    if(!launch_shape(ctx, params->max_depth, /*whole=*/true, L, &warps, &ctas, &smem))
        return fail(DRT_CUDA_E_UNSUPPORTED, "record dump: max_cast_depth %u with %d lights needs %zu bytes of shared memory per warp (limit %zu)",
                    params->max_depth, ctx->nlights, smem, ctx->smem_optin);
    *words_per_path = L.path_words;
    if(!out_host) return DRT_CUDA_OK;
    size_t words = (size_t)(x1 - x0) * (y1 - y0) * (params->sample_end - params->sample_begin) * (size_t)*words_per_path;
    if(words > out_capacity_words) return fail(DRT_CUDA_E_ARG, "record buffer too small: need %zu words", words);
    int rc = drt_ensure_buffer(&ctx->d_dump, &ctx->dump_bytes, words * 4);
    if(rc != DRT_CUDA_OK) return rc;
    rc = launch(ctx, params, x0, y0, x1, y1, FilmPtrs{}, nullptr, 0, 0, ctx->d_dump);
    if(rc != DRT_CUDA_OK) return rc;
    CU(cudaMemcpy(out_host, ctx->d_dump, words * 4, cudaMemcpyDeviceToHost));
    return DRT_CUDA_OK;
}

extern "C" int drt_cuda_film_to_rgb(drt_cuda_context *ctx, const drt_film *film, uint32_t width, uint32_t height, int which,
                                    float *rgb_device, uint32_t *bgra_device, void *stream)
{
    if(!ctx || !film || which < 0 || which > 2) return fail(DRT_CUDA_E_ARG, "bad argument");
    if(!ctx->have_scene) return fail(DRT_CUDA_E_STATE, "upload a scene first");
    CU(cudaSetDevice(ctx->device));
    const float *plane = which == 0 ? film->sum : which == 1 ? film->mean : film->m2;
    const float *filter = which == 0 ? film->filter : nullptr;
    if(!plane || (which == 0 && !filter)) return fail(DRT_CUDA_E_ARG, "film plane is NULL");
    const uint64_t npix64 = (uint64_t)width * height;
    if(npix64 == 0 || npix64 > 0xffffffffull) return fail(DRT_CUDA_E_ARG, "%u x %u pixels out of range", width, height);
    uint32_t npix = (uint32_t)npix64;
    int grid = ctx->num_sms * 8;
    drt_launch_film_to_rgb(ctx->d_rgb_tables, plane, filter, which == 2, npix, rgb_device, bgra_device, grid, (cudaStream_t)stream);
    CU(cudaGetLastError());
    ctx->launches += 1;
    return DRT_CUDA_OK;
}

extern "C" int drt_cuda_film_merge(drt_cuda_context *ctx, const drt_film *dst, const drt_film *src, uint32_t width, uint32_t height, void *stream)
{
    if(!ctx || !dst || !src) return fail(DRT_CUDA_E_ARG, "NULL argument");
    if(!ctx->have_scene) return fail(DRT_CUDA_E_STATE, "upload a scene first");
    CU(cudaSetDevice(ctx->device));
    drt_launch_film_merge(film_ptrs(*dst), film_ptrs(*src), (uint32_t)ctx->n, (size_t)width * height, ctx->num_sms * 8, (cudaStream_t)stream);
    CU(cudaGetLastError());
    ctx->launches += 2;
    return DRT_CUDA_OK;
}

static bool overlaps(const float *a, size_t na, const float *b, size_t nb) { return a < b + nb && b < a + na; }

/* argument checks of the denoise entry points (drt_cuda.h), before anything is copied or launched */
static int denoise_args(const drt_cuda_context *ctx, const drt_film *film, uint32_t width, uint32_t height, const drt_denoise *opt, const float *out)
{
    if(!ctx || !film || !opt || !out) return fail(DRT_CUDA_E_ARG, "NULL argument");
    if(!ctx->have_scene) return fail(DRT_CUDA_E_STATE, "upload a scene first");
    if(!film->mean || !film->m2 || !film->filter) return fail(DRT_CUDA_E_ARG, "denoise: the film needs its mean, m2 and filter planes");
    if(width == 0 || height == 0 || (uint64_t)width * height > 0xffffffffull)
        return fail(DRT_CUDA_E_ARG, "denoise: width and height must be > 0, and width x height < 2^32 (got %u x %u)", width, height);
    if(opt->search_radius < 1 || opt->search_radius > 15) return fail(DRT_CUDA_E_ARG, "denoise: search_radius must lie in 1..15 (got %u)", opt->search_radius);
    if(opt->patch_radius > 4) return fail(DRT_CUDA_E_ARG, "denoise: patch_radius must lie in 0..4 (got %u)", opt->patch_radius);
    /* the filter takes k^2 as an f32: it must be a normal number, so that neither 1e-10 + k^2 (v_a + v_b) nor its product overflows
     * to inf or vanishes for every finite pair of variances */
    const float kk = opt->strength * opt->strength;
    if(!(opt->strength > 0.f) || !isnormal(kk))
        return fail(DRT_CUDA_E_ARG, "denoise: strength must lie in [2^-63, 2^64), so that strength^2 is a normal f32 (got %g)",
                    (double)opt->strength);
    const size_t npix = (size_t)width * height, plane = npix * (size_t)ctx->n;
    if(overlaps(out, plane, film->mean, plane) || overlaps(out, plane, film->m2, plane) || overlaps(out, plane, film->filter, npix))
        return fail(DRT_CUDA_E_ARG, "denoise: mean_out overlaps the film's mean, m2 or filter plane");
    return DRT_CUDA_OK;
}

/* guide, then filter, on `stream` (arguments checked) */
static int denoise(drt_cuda_context *ctx, const drt_film *film, uint32_t width, uint32_t height, const drt_denoise *opt, float *out, cudaStream_t stream)
{
    const size_t npix = (size_t)width * height;
    int rc = drt_ensure_buffer(&ctx->d_denoise, &ctx->denoise_bytes, 3 * npix * sizeof(float));
    if(rc != DRT_CUDA_OK) return rc;
    const float *yw = reinterpret_cast<const float *>(static_cast<const unsigned char *>(ctx->d_rgb_tables) + drt_rgb_tables_yw_offset());
    if(!ctx->denoise_done) CU(cudaEventCreateWithFlags(&ctx->denoise_done, cudaEventDisableTiming));
    CU(cudaStreamWaitEvent(stream, ctx->denoise_done, 0));   /* the previous call's filter has read the guide planes */
    drt_launch_denoise_guide(yw, film->mean, film->m2, film->filter, (uint32_t)npix, ctx->n, ctx->d_denoise, ctx->num_sms * 8, stream);
    CU(cudaGetLastError());
    CU(drt_launch_denoise_filter(film->mean, ctx->d_denoise, width, height, ctx->n, (int)opt->search_radius, (int)opt->patch_radius,
                                 opt->strength, out, stream));
    CU(cudaEventRecord(ctx->denoise_done, stream));
    ctx->launches += 2;
    return DRT_CUDA_OK;
}

extern "C" int drt_cuda_film_denoise(drt_cuda_context *ctx, const drt_film *film, uint32_t width, uint32_t height, const drt_denoise *opt,
                                     float *mean_out, void *stream)
{
    int rc = denoise_args(ctx, film, width, height, opt, mean_out);
    if(rc != DRT_CUDA_OK) return rc;
    CU(cudaSetDevice(ctx->device));
    return denoise(ctx, film, width, height, opt, mean_out, (cudaStream_t)stream);
}

/* The film goes up into the library-owned film (d_film): its mean, m2 and filter planes hold the input, its sum plane the output. */
extern "C" int drt_cuda_film_denoise_host(drt_cuda_context *ctx, const drt_film *film, uint32_t width, uint32_t height, const drt_denoise *opt,
                                          float *mean_out)
{
    int rc = denoise_args(ctx, film, width, height, opt, mean_out);
    if(rc != DRT_CUDA_OK) return rc;
    CU(cudaSetDevice(ctx->device));
    const size_t npix = (size_t)width * height, bytes = npix * (size_t)ctx->n * sizeof(float);
    drt_film f;
    rc = drt_library_film(ctx, &ctx->d_film, &ctx->film_bytes, npix, &f);
    if(rc != DRT_CUDA_OK) return rc;
    CU(cudaMemcpyAsync(f.mean, film->mean, bytes, cudaMemcpyHostToDevice, 0));
    CU(cudaMemcpyAsync(f.m2, film->m2, bytes, cudaMemcpyHostToDevice, 0));
    CU(cudaMemcpyAsync(f.filter, film->filter, npix * sizeof(float), cudaMemcpyHostToDevice, 0));
    rc = denoise(ctx, &f, width, height, opt, f.sum, 0);
    if(rc != DRT_CUDA_OK) return rc;
    CU(cudaMemcpyAsync(mean_out, f.sum, bytes, cudaMemcpyDeviceToHost, 0));
    CU(cudaStreamSynchronize(0));
    return DRT_CUDA_OK;
}

extern "C" int drt_cuda_film_alloc(drt_cuda_context *ctx, uint32_t width, uint32_t height, drt_film *out)
{
    if(!ctx || !out) return fail(DRT_CUDA_E_ARG, "NULL argument");
    if(!ctx->have_scene) return fail(DRT_CUDA_E_STATE, "upload a scene first");
    CU(cudaSetDevice(ctx->device));
    size_t npix = (size_t)width * height, plane = npix * (size_t)ctx->n * 4;
    memset(out, 0, sizeof(*out));
    cudaError_t e = cudaMalloc(&out->sum, plane);
    if(e == cudaSuccess) e = cudaMalloc(&out->mean, plane);
    if(e == cudaSuccess) e = cudaMalloc(&out->m2, plane);
    if(e == cudaSuccess) e = cudaMalloc(&out->filter, npix * 4);
    if(e == cudaSuccess) e = cudaMemset(out->sum, 0, plane);
    if(e == cudaSuccess) e = cudaMemset(out->mean, 0, plane);
    if(e == cudaSuccess) e = cudaMemset(out->m2, 0, plane);
    if(e == cudaSuccess) e = cudaMemset(out->filter, 0, npix * 4);
    if(e != cudaSuccess)
    {
        cudaFree(out->sum); cudaFree(out->mean); cudaFree(out->m2); cudaFree(out->filter);
        memset(out, 0, sizeof(*out));
        return fail(DRT_CUDA_E_CUDA, "film_alloc %ux%u: %s", width, height, cudaGetErrorString(e));
    }
    return DRT_CUDA_OK;
}

extern "C" int drt_cuda_film_free(drt_cuda_context *ctx, drt_film *film)
{
    if(!ctx || !film) return fail(DRT_CUDA_E_ARG, "NULL argument");
    CU(cudaSetDevice(ctx->device));
    cudaFree(film->sum); cudaFree(film->mean); cudaFree(film->m2); cudaFree(film->filter);
    memset(film, 0, sizeof(*film));
    return DRT_CUDA_OK;
}

extern "C" int drt_cuda_film_ipc_export(drt_cuda_context *ctx, const drt_film *film, unsigned char handles[4][64])
{
    if(!ctx || !film || !handles) return fail(DRT_CUDA_E_ARG, "NULL argument");
    CU(cudaSetDevice(ctx->device));
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "CUDA IPC handle size");
    float *ptrs[4] = { film->sum, film->filter, film->mean, film->m2 };
    for(int i = 0; i < 4; i += 1)
    {
        cudaIpcMemHandle_t h;
        CU(cudaIpcGetMemHandle(&h, ptrs[i]));
        memcpy(handles[i], &h, 64);
    }
    return DRT_CUDA_OK;
}

extern "C" int drt_cuda_film_ipc_open(drt_cuda_context *ctx, const unsigned char handles[4][64], drt_film *out)
{
    if(!ctx || !handles || !out) return fail(DRT_CUDA_E_ARG, "NULL argument");
    CU(cudaSetDevice(ctx->device));
    void *ptrs[4] = { nullptr, nullptr, nullptr, nullptr };
    for(int i = 0; i < 4; i += 1)
    {
        cudaIpcMemHandle_t h;
        memcpy(&h, handles[i], 64);
        CU(cudaIpcOpenMemHandle(&ptrs[i], h, cudaIpcMemLazyEnablePeerAccess));
    }
    out->sum = (float *)ptrs[0]; out->filter = (float *)ptrs[1]; out->mean = (float *)ptrs[2]; out->m2 = (float *)ptrs[3];
    return DRT_CUDA_OK;
}

extern "C" int drt_cuda_film_ipc_close(drt_cuda_context *ctx, drt_film *mapped)
{
    if(!ctx || !mapped) return fail(DRT_CUDA_E_ARG, "NULL argument");
    CU(cudaSetDevice(ctx->device));
    cudaIpcCloseMemHandle(mapped->sum); cudaIpcCloseMemHandle(mapped->filter); cudaIpcCloseMemHandle(mapped->mean); cudaIpcCloseMemHandle(mapped->m2);
    memset(mapped, 0, sizeof(*mapped));
    return DRT_CUDA_OK;
}

extern "C" int drt_cuda_buffer_alloc(drt_cuda_context *ctx, size_t bytes, void **out)
{
    if(!ctx || !out || bytes == 0) return fail(DRT_CUDA_E_ARG, "bad argument");
    CU(cudaSetDevice(ctx->device));
    CU(cudaMalloc(out, bytes));
    CU(cudaMemset(*out, 0, bytes));
    return DRT_CUDA_OK;
}

extern "C" int drt_cuda_buffer_free(drt_cuda_context *ctx, void *ptr)
{
    if(!ctx) return fail(DRT_CUDA_E_ARG, "NULL argument");
    CU(cudaSetDevice(ctx->device));
    CU(cudaFree(ptr));
    return DRT_CUDA_OK;
}

extern "C" int drt_cuda_buffer_ipc_export(drt_cuda_context *ctx, const void *ptr, unsigned char handle[64])
{
    if(!ctx || !ptr || !handle) return fail(DRT_CUDA_E_ARG, "NULL argument");
    CU(cudaSetDevice(ctx->device));
    cudaIpcMemHandle_t h;
    CU(cudaIpcGetMemHandle(&h, const_cast<void *>(ptr)));
    memcpy(handle, &h, 64);
    return DRT_CUDA_OK;
}

extern "C" int drt_cuda_buffer_ipc_open(drt_cuda_context *ctx, const unsigned char handle[64], void **out)
{
    if(!ctx || !handle || !out) return fail(DRT_CUDA_E_ARG, "NULL argument");
    CU(cudaSetDevice(ctx->device));
    cudaIpcMemHandle_t h;
    memcpy(&h, handle, 64);
    CU(cudaIpcOpenMemHandle(out, h, cudaIpcMemLazyEnablePeerAccess));
    return DRT_CUDA_OK;
}

extern "C" int drt_cuda_buffer_ipc_close(drt_cuda_context *ctx, void *mapped)
{
    if(!ctx || !mapped) return fail(DRT_CUDA_E_ARG, "NULL argument");
    CU(cudaSetDevice(ctx->device));
    CU(cudaIpcCloseMemHandle(mapped));
    return DRT_CUDA_OK;
}

extern "C" int drt_cuda_film_merge_many(drt_cuda_context *ctx, const drt_film *dst, const drt_film *srcs, int count, uint32_t width, uint32_t height,
                                        uint64_t pixel_begin, uint64_t pixel_end, uint32_t *bgra_sum, uint32_t *bgra_mean, uint32_t *bgra_var, void *stream)
{
    if(!ctx || !dst || !srcs || count < 1 || count > 16) return fail(DRT_CUDA_E_ARG, "bad argument (1..16 films)");
    if(!ctx->have_scene) return fail(DRT_CUDA_E_STATE, "upload a scene first");
    uint64_t npix = (uint64_t)width * height;
    if(pixel_begin > pixel_end || pixel_end > npix) return fail(DRT_CUDA_E_ARG, "bad pixel range");
    if((bgra_sum || bgra_mean || bgra_var) && !(bgra_sum && bgra_mean && bgra_var)) return fail(DRT_CUDA_E_ARG, "give all three image buffers or none");
    CU(cudaSetDevice(ctx->device));
    FilmPtrs films[16];
    for(int i = 0; i < count; i += 1) films[i] = film_ptrs(srcs[i]);
    if(pixel_end > pixel_begin)
    {
        drt_launch_film_gather_merge(ctx->d_rgb_tables, count, films, film_ptrs(*dst), (uint32_t)pixel_begin, (uint32_t)pixel_end, 0u, 0u, bgra_sum, bgra_mean, bgra_var,
                                     ctx->num_sms * 8, (cudaStream_t)stream);
        CU(cudaGetLastError());
        ctx->launches += 1;
    }
    return DRT_CUDA_OK;
}

extern "C" int drt_cuda_film_merge_slices(drt_cuda_context *ctx, const drt_film *dst, const drt_film *staging, int count, uint64_t slice_pixels,
                                          uint32_t width, uint32_t height, uint64_t pixel_begin, uint64_t pixel_end,
                                          uint32_t *bgra_sum, uint32_t *bgra_mean, uint32_t *bgra_var, void *stream)
{
    if(!ctx || !dst || !staging || count < 1 || count > DRT_MAX_PEERS) return fail(DRT_CUDA_E_ARG, "bad argument (1..%d ranks)", DRT_MAX_PEERS);
    if(!ctx->have_scene) return fail(DRT_CUDA_E_STATE, "upload a scene first");
    uint64_t npix = (uint64_t)width * height;
    if(pixel_begin > pixel_end || pixel_end > npix || pixel_end - pixel_begin > slice_pixels) return fail(DRT_CUDA_E_ARG, "bad pixel range");
    if((bgra_sum || bgra_mean || bgra_var) && !(bgra_sum && bgra_mean && bgra_var)) return fail(DRT_CUDA_E_ARG, "give all three image buffers or none");
    CU(cudaSetDevice(ctx->device));
    const size_t n = (size_t)ctx->n;
    FilmPtrs films[DRT_MAX_PEERS];
    for(int g = 0; g < count; g += 1)   /* rank g's partial film of this slice: staging pixels [g * slice, (g + 1) * slice) */
        films[g] = FilmPtrs{ staging->sum + (size_t)g * slice_pixels * n, staging->filter + (size_t)g * slice_pixels,
                             staging->mean + (size_t)g * slice_pixels * n, staging->m2 + (size_t)g * slice_pixels * n };
    /* staging is indexed from the first pixel of the owner's slice; [pixel_begin, pixel_end) may be a part (a band) of it */
    const uint64_t slice_begin = slice_pixels ? (pixel_begin / slice_pixels) * slice_pixels : 0;
    if(pixel_end > pixel_begin && pixel_end - slice_begin > slice_pixels) return fail(DRT_CUDA_E_ARG, "pixel range crosses a slice boundary");
    if(pixel_end > pixel_begin)
    {
        /* merged planes of the slice go to a local scratch film first and travel to dst_device (the root's film: usually peer
         * memory) as four contiguous copies: the copy engines move large blocks over NVLink about twice as fast as the
         * kernel's 4-byte-per-lane peer stores did (measured: 763 MB into the root in 2.2 ms from kernel stores) */
        const size_t spx = (size_t)(pixel_end - pixel_begin), plane = spx * n * 4;
        drt_film d;
        int rc = drt_library_film(ctx, &ctx->d_slice, &ctx->slice_bytes, spx, &d);
        if(rc != DRT_CUDA_OK) return rc;
        drt_launch_film_gather_merge(ctx->d_rgb_tables, count, films, film_ptrs(d), (uint32_t)pixel_begin, (uint32_t)pixel_end, (uint32_t)slice_begin,
                                     (uint32_t)pixel_begin, bgra_sum, bgra_mean, bgra_var, ctx->num_sms * 8, (cudaStream_t)stream);
        CU(cudaGetLastError());
        const size_t at = (size_t)pixel_begin * n;
        CU(cudaMemcpyAsync(dst->sum + at, d.sum, plane, cudaMemcpyDefault, (cudaStream_t)stream));
        CU(cudaMemcpyAsync(dst->mean + at, d.mean, plane, cudaMemcpyDefault, (cudaStream_t)stream));
        CU(cudaMemcpyAsync(dst->m2 + at, d.m2, plane, cudaMemcpyDefault, (cudaStream_t)stream));
        CU(cudaMemcpyAsync(dst->filter + pixel_begin, d.filter, spx * 4, cudaMemcpyDefault, (cudaStream_t)stream));
        ctx->launches += 1;
    }
    return DRT_CUDA_OK;
}

extern "C" int drt_cuda_measure_fp32_peak(drt_cuda_context *ctx, int packed, double *tflops)
{
    if(!ctx || !tflops) return fail(DRT_CUDA_E_ARG, "NULL argument");
    CU(cudaSetDevice(ctx->device));
    float *d_out = nullptr;
    cudaEvent_t a = nullptr, b = nullptr;
    cudaError_t e = cudaMalloc(&d_out, 4);
    if(e == cudaSuccess) e = cudaEventCreate(&a);
    if(e == cudaSuccess) e = cudaEventCreate(&b);
    const int iters = 4096, grid = ctx->num_sms * 8;
    double best = 0.0;
    for(int rep = 0; rep < 5 && e == cudaSuccess; rep += 1)
    {
        e = cudaEventRecord(a, 0);
        drt_launch_fma_peak(packed, d_out, iters, grid, 0);
        if(e == cudaSuccess) e = cudaEventRecord(b, 0);
        if(e == cudaSuccess) e = cudaEventSynchronize(b);
        float ms = 0.f;
        if(e == cudaSuccess) e = cudaEventElapsedTime(&ms, a, b);
        if(e != cudaSuccess) break;
        double flops = (double)grid * 256.0 * (double)iters * 16.0 * 2.0;
        double t = flops / (ms * 1e-3) / 1e12;
        if(rep > 0 && t > best) best = t;
    }
    if(a) cudaEventDestroy(a);
    if(b) cudaEventDestroy(b);
    cudaFree(d_out);
    if(e != cudaSuccess) return fail(DRT_CUDA_E_CUDA, "fp32 peak probe: %s", cudaGetErrorString(e));
    *tflops = best;
    return DRT_CUDA_OK;
}
