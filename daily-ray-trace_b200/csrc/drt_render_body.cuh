/*
 * csrc/drt_render_body.cuh -- the body of the render kernel, included (no include guard) inside render_kernel and
 * render_kernel_adaptive of drt_render.cuh.  Those two are the only places that include it; they declare
 *   R, NS, MODE, PAIRED, DEEP   as template parameters or constants, and
 *   ADAPTIVE                    constexpr bool: a paired (one pixel per task) launch whose pixels stop early (pixel_converged).
 * The body sits textually inside each __global__ function rather than in an inlined __device__ function: the compiler then makes the
 * same inlining and range decisions as for a kernel of its own, so render_kernel compiles to the same code with adaptive sampling in
 * the tree as without it.  All adaptive code is behind `if constexpr(ADAPTIVE)`.
 */
    constexpr bool ALLFAST = MODE != 0;   /* compact records, film parked in shared memory while tracing */
    /* LOCKSTEP (a kernel whose hot code does not fit the 32 KB instruction cache; DRT_LOCKSTEP says which modes): the warps of a CTA
     * run their phases together -- a gate (an mbarrier that every warp arrives at once per phase and leaves for good when it runs
     * out of pixels) in front of phase 1 and of phase 2 -- so that at any time the SM fetches the code of ONE phase. */
    constexpr bool LOCKSTEP = MODE == 2 ? ((DRT_LOCKSTEP & 2) != 0) : MODE == 0 ? ((DRT_LOCKSTEP & 1) != 0) : ((DRT_LOCKSTEP & 4) != 0);
    __shared__ unsigned long long phase_bar;
    __shared__ uint32_t gates_off;
#ifdef DRT_PHASE_CLOCKS
    __shared__ unsigned long long s_phase[4];
    uint32_t phase_t = 0;
    if(threadIdx.x < 4) s_phase[threadIdx.x] = 0ull;
#endif
    const uint32_t bar_addr = (uint32_t)__cvta_generic_to_shared(&phase_bar);
    if(LOCKSTEP && threadIdx.x == 0)
    {
        asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" :: "r"(bar_addr), "r"(blockDim.x >> 5) : "memory");
        gates_off = L.scatter_count > 1 ? 1u : 0u;   /* see DRT_GATE_PATIENCE_CYCLES in drt_device.cuh */
    }
    extern __shared__ __align__(16) unsigned char smem_raw[];
    GeomT<R> *sg = reinterpret_cast<GeomT<R> *>(smem_raw);
    size_t off = (sizeof(GeomT<R>) + 15) & ~size_t(15);
    SpdIndex *six = reinterpret_cast<SpdIndex *>(smem_raw + off);
    off += (sizeof(SpdIndex) + 15) & ~size_t(15);
    float *spool = reinterpret_cast<float *>(smem_raw + off);
    off += (size_t)L.pool_words * 4;
    unsigned long long *s_stats = reinterpret_cast<unsigned long long *>(smem_raw + off);
    off += 16 * 8;
    off = (off + 15) & ~size_t(15);
    float *srec = reinterpret_cast<float *>(smem_raw + off);
    float *spark = srec + (size_t)(blockDim.x >> 5) * L.path_stride * DRT_WARP;   /* film parking, (3 NS + 2) * 32 words per warp */

    /* stage the scene once per (persistent) CTA */
    {
        const uint32_t *src = reinterpret_cast<const uint32_t *>(L.geom);
        uint32_t *dst = reinterpret_cast<uint32_t *>(sg);
#pragma unroll 1
        for(uint32_t i = threadIdx.x; i < sizeof(GeomT<R>) / 4; i += blockDim.x) dst[i] = src[i];
        src = reinterpret_cast<const uint32_t *>(L.spd_index);
        dst = reinterpret_cast<uint32_t *>(six);
#pragma unroll 1
        for(uint32_t i = threadIdx.x; i < sizeof(SpdIndex) / 4; i += blockDim.x) dst[i] = src[i];
#pragma unroll 1
        for(uint32_t i = threadIdx.x; i < L.pool_words; i += blockDim.x) spool[i] = L.pool[i];
        if(threadIdx.x < 16) s_stats[threadIdx.x] = 0ull;
    }
    __syncthreads();
    const GeomT<R> &g = *sg;
    const SpdIndex &ix = *six;

    const uint32_t lane = threadIdx.x & 31u, warp = threadIdx.x >> 5;
    const uint32_t lane16 = lane & (DRT_HALF - 1), half = lane >> 4;
#ifdef DRT_PHASE_CLOCKS
    asm volatile("mov.u32 %0, %%clock;" : "=r"(phase_t) :: "memory");
#endif
    float *rec = srec + (size_t)warp * L.path_stride * DRT_WARP;   /* word w of slot s at rec[s * path_stride + w] */
    const uint32_t stride = L.path_stride;
    float *park = spark + (size_t)warp * (3 * NS + 2) * DRT_WARP + lane;
    /* this warp's 32 overflow rows in global memory (deep renders: bounces past L.smem_depth; RenderLaunch::deep) */
    float *deep_w = DEEP ? L.deep + (size_t)(blockIdx.x * (blockDim.x >> 5) + warp) * DRT_WARP * L.deep_stride : nullptr;
    const float *pool_lane = spool + lane16;
    const uint32_t rw = L.x1 - L.x0, npix = rw * (L.y1 - L.y0);
    const uint32_t spp = L.sample_end - L.sample_begin;
    const uint32_t n = (uint32_t)ix.n;
    const uint32_t ntasks = (PAIRED && L.band_chunk) ? L.band_chunk * L.scatter_count : (npix + L.pixels_per_task - 1) / L.pixels_per_task;
    const bool have_film = L.film.sum != nullptr;
    /* A task is one pixel with all its samples (spp >= 32: `paired`, the film stays in registers across the pixel's batches of
     * 32 paths) or 32/spp whole pixels traced as ONE batch.  Either way phase 2 walks the batch pixel by pixel, both half
     * warps shading samples of the same pixel, two paths at a time. */
    constexpr bool paired = PAIRED;
    /* the pixel's finished film goes to `film`, or (multi-GPU scatter) to the staging film of the rank that owns the pixel */
    auto store_pixel = [&](uint32_t gpix, const PixelFilm<NS> &f)
    {
        FilmPtrs out = L.film;
        uint32_t at = gpix;
        if(L.scatter_count)
        {
            const uint32_t owner = gpix / L.scatter_slice;
            out = L.scatter[owner];
            at = L.scatter_rank * L.scatter_slice + (gpix - owner * L.scatter_slice);
        }
        film_store<NS>(out, at, n, lane, f);
    };
    const bool dumping = L.path_dump || L.record_dump;

    uint32_t tally[4] = { 0u, 0u, 0u, 0u };   /* closest rays, shadow rays, shaded bounces, rng draws of this lane */
    uint32_t traced = 0;
    uint32_t gate_parity = 0;
    auto gate = [&]()
    {
        if constexpr(LOCKSTEP)
        {
            /* The gates only steer WHEN the warps of a CTA run their phases (one phase's code in the instruction cache at a time); no
             * data passes through them.  So they are allowed to fail safe: a warp that has waited DRT_GATE_PATIENCE_CYCLES (about 10 ms,
             * two orders above a phase) switches the CTA's gates off for the rest of the launch instead of waiting on. */
            if(*reinterpret_cast<volatile uint32_t *>(&gates_off)) return;
            if(lane == 0) asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" :: "r"(bar_addr) : "memory");
            __syncwarp();
            /* try_wait with a suspend-time hint: the warp sleeps in hardware until the phase completes (or the hint expires) instead of
             * spinning -- a spinning gate took 27 % of the kernel's issued instructions (profiles/r2_ncu_classed_kernel.md) */
            uint32_t ok = 0;
            const long long t0 = clock64();
            while(!ok)
            {
                asm volatile("{ .reg .pred p; mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3; selp.u32 %0, 1, 0, p; }"
                             : "=r"(ok) : "r"(bar_addr), "r"(gate_parity), "r"(DRT_GATE_SUSPEND_NS) : "memory");
                if(!ok && (clock64() - t0 > DRT_GATE_PATIENCE_CYCLES || *reinterpret_cast<volatile uint32_t *>(&gates_off)))
                {
                    gates_off = 1u;
                    break;
                }
            }
            gate_parity ^= 1u;
        }
    };
    for(;;)
    {
        uint32_t task = 0;
        if(lane == 0) task = atomicAdd(L.task_counter, 1u);
        task = __shfl_sync(0xffffffffu, task, 0);
        if(task >= ntasks)
        {
            /* out of pixels: this warp leaves the gates for good (it is in front of a phase-1 gate, like every warp that still works) */
            if(LOCKSTEP && lane == 0) asm volatile("mbarrier.arrive_drop.shared::cta.b64 _, [%0];" :: "r"(bar_addr) : "memory");
            break;
        }
        task += L.task_rotate;
        if(task >= ntasks) task -= ntasks;
        uint32_t p_begin = task * L.pixels_per_task;
        if(paired && L.band_chunk)   /* a band of a scattered render: the same part of every owner's slice */
        {
            p_begin = (p_begin / L.band_chunk) * L.band_period + L.band_base + p_begin % L.band_chunk;
            if(p_begin >= L.width * L.height) continue;
        }
        const uint32_t p_end = paired ? p_begin + 1u : min(p_begin + L.pixels_per_task, npix);
        const uint32_t total = (p_end - p_begin) * spp;
        traced += total;

        PixelFilm<NS> film;
        film.clear();
        const uint32_t task_x = L.x0 + p_begin % rw, task_y = L.y0 + p_begin / rw;   /* first pixel of the task */
        if(paired && L.accumulate && have_film) film = film_load<NS>(L.film, task_y * L.width + task_x, n, lane);

        if(paired && !dumping && (task_x < L.hit_x0 || task_x >= L.hit_x1 || task_y < L.hit_y0 || task_y >= L.hit_y1))
        {
            /* a pixel that cannot see a surface: all its samples at once */
            uint32_t taken = total;
            if constexpr(ADAPTIVE)
            {
                /* batch by batch, as far as the stopping rule takes the pixel */
                for(uint32_t q0 = 0; q0 < total; q0 += DRT_WARP)
                {
                    const uint32_t count = min((uint32_t)DRT_WARP, total - q0);
                    if(half == 0) film.add_zeros(count);
                    if(pixel_converged<NS>(film, L, n, lane16)) { taken = q0 + count; break; }
                }
                traced -= total - taken;
            }
            else if(half == 0) film.add_zeros(total);
            if(lane == 0)
            {
                atomicAdd(&s_stats[1], (unsigned long long)taken);
                atomicAdd(&s_stats[4], (unsigned long long)((L.pixel_scheme == DRT_PIXEL_RANDOM) ? 2u * taken : 0u));
                atomicAdd(&s_stats[5], (unsigned long long)taken);
            }
            film.merge_halves();
            if(have_film) store_pixel(task_y * L.width + task_x, film);
            continue;
        }
        for(uint32_t q0 = 0; q0 < total; q0 += DRT_WARP)
        {
            /* ---- phase 1: lane = path ---- */
            DRT_PHASE_CUT(DRT_PHASE_OTHER);
            gate();
            if((ALLFAST || DRT_PARK_GENERAL) && paired) film.park(park);
            const uint32_t q = q0 + lane;
            uint32_t bin = 9, general = 0;
            uint32_t my_px = 0, my_s = q;      /* pixel of the batch and sample index inside the pixel */
            if(!paired) { my_px = q / spp; my_s = q - my_px * spp; }
            if(q < total)
            {
                uint32_t x = task_x, y = task_y;
                if(!paired) { const uint32_t lp = p_begin + my_px; x = L.x0 + lp % rw; y = L.y0 + lp / rw; }
                if(x < L.hit_x0 || x >= L.hit_x1 || y < L.hit_y0 || y >= L.hit_y1)
                {
                    /* the pixel cannot see a surface (RenderLaunch::hit_*): its path is the camera ray's two draws and one closest-hit
                     * ray that ends on the escape material */
                    rec[lane * stride + REC_NB] = 0.f;
                    tally[0] += 1; tally[3] += (L.pixel_scheme == DRT_PIXEL_RANDOM) ? 2u : 0u;
                    bin = 0;
                }
                else
                {
                    uint32_t r = trace_path<R, MODE, DEEP>(g, ix, L, rec + lane * stride, deep_w + (size_t)lane * L.deep_stride, x, y, L.sample_begin + my_s, tally);
                    bin = r & 255u; general = r >> 8;
                }
            }
            __syncwarp();
            DRT_PHASE_CUT(DRT_PHASE_TRACE);
            gate();
            /* compact records: the film stays parked through the replay, which accumulates BatchStats instead */
            if(!ALLFAST && DRT_PARK_GENERAL && paired) film.unpark(park);
            {
                /* termination histogram: one shared-memory atomic per distinct bin of the batch (bin 9 = idle lane) */
                const uint32_t peers = __match_any_sync(0xffffffffu, bin);
                if(bin < 9u && lane == (uint32_t)__ffs(peers) - 1u) atomicAdd(&s_stats[5 + bin], (unsigned long long)__popc(peers));
            }
            /* ---- phase 2: half warp = path, lane16 = wavelength ---- */
            const uint32_t count = min((uint32_t)DRT_WARP, total - q0);
            const uint32_t my_nb = __float_as_uint(rec[lane * stride + REC_NB]);
            if(paired && !dumping && !__any_sync(0xffffffffu, lane < count && my_nb != 0u))
            {
                /* no path of the batch has a bounce record (every sample left the scene): nothing to replay */
                if(ALLFAST) film.unpark(park);
                if(half == 0) film.add_zeros(count);
                __syncwarp();
                DRT_PHASE_CUT(DRT_PHASE_BOOK);
                if constexpr(ADAPTIVE)
                    if(pixel_converged<NS>(film, L, n, lane16)) { traced -= total - (q0 + count); break; }
                continue;
            }
            /* K5, warp scope: order the batch by pixel, and inside a pixel so that the two halves of the warp get paths of like
             * cost: paths without any bounce record first, then plastic-only paths by bounce count, then paths that need the
             * general shader by bounce count; idle lanes last.  A 32-wide bitonic sort over (key, lane).  The film is a
             * sum / Welford accumulation, so the order only changes rounding. */
            const uint32_t cls = (my_nb == 0u) ? 0u : min((my_nb & 0xffffu) + (my_nb >> 16 ? 1u : 0u), 15u) + (general ? 16u : 0u);
            uint32_t v = (lane >= count) ? 0xffffffffu : (((my_px << 5) | cls) << 5) | lane;
#pragma unroll
            for(uint32_t k = 2; k <= 32; k <<= 1)
#pragma unroll
                for(uint32_t j = k >> 1; j > 0; j >>= 1)
                {
                    uint32_t other = __shfl_xor_sync(0xffffffffu, v, j);
                    bool keep_min = ((lane & k) == 0) == ((lane & j) == 0);
                    v = keep_min ? min(v, other) : max(v, other);
                }
            const uint32_t per_px = paired ? count : spp;            /* slots of one pixel in this batch */
            const uint32_t npx = paired ? 1u : count / spp;
#pragma unroll 1
            for(uint32_t px = 0; px < npx; px += 1)
            {
                const uint32_t lp = p_begin + px;
                uint32_t gpix = 0;
                /* compact records: the film of a pixel is loaded (or cleared) after the replay, so it takes no registers during it */
                auto start_film = [&]()
                {
                    if(!paired)
                    {
                        gpix = (L.y0 + lp / rw) * L.width + L.x0 + lp % rw;
                        film.clear();
                        if(L.accumulate && have_film) film = film_load<NS>(L.film, gpix, n, lane);
                    }
                };
                if(!ALLFAST) start_film();
                const uint32_t lo = px * per_px;
                const uint32_t nzero = __popc(__ballot_sync(0xffffffffu, lane < count && my_px == px && my_nb == 0u));
                if(!ALLFAST && half == 0) film.add_zeros(nzero);   /* paths that contributed nothing */
                if(dumping)
                    for(uint32_t i = lo; i < lo + nzero; i += 1)
                    {
                        const uint32_t slot = __shfl_sync(0xffffffffu, v, i) & 31u;
                        const uint32_t s_in = paired ? q0 + slot : slot - px * spp;
                        if(half == 0) dump_path<NS>(L.record_dump, L.path_dump, L.path_words, rec + slot * stride, nullptr, nullptr, (size_t)lp * spp + s_in, n, lane16);
                    }
                BatchStats<NS> bs;
                if(ALLFAST) bs.clear();
                DRT_PHASE_CUT(DRT_PHASE_BOOK);
                for(uint32_t i = lo + nzero; i < lo + per_px; i += 2)
                {
                    const uint32_t pos = i + half;
                    const uint32_t slot = __shfl_sync(0xffffffffu, v, pos & 31u) & 31u;
                    const uint32_t nb = __shfl_sync(0xffffffffu, my_nb, slot);
                    if(pos < lo + per_px)
                    {
                        float c[NS];
                        if constexpr(ALLFAST)
                        {
                            unsigned long long r2[BatchStats<NS>::NP1];
                            float r1;
                            replay_compact<NS, MODE, DEEP>(rec + slot * stride, deep_w + (size_t)slot * L.deep_stride, nb, ix, spool, pool_lane, lane16, L, r2, r1);
                            bs.add(r2, r1, i == lo + nzero);
                            if(dumping)
                            {
#pragma unroll
                                for(int k = 0; k < NS / 2; k += 1) upk2(r2[k], c[2 * k], c[2 * k + 1]);
                                if(NS & 1) c[NS - 1] = r1;
                            }
                        }
                        else
                        {
                            replay_path<NS, DEEP>(rec + slot * stride, deep_w + (size_t)slot * L.deep_stride, nb, g, ix, spool, pool_lane, lane16, L, c);
                            film.add(c);
                        }
                        if(dumping)
                        {
                            float cc[NS];   /* a copy whose address is taken only here: c itself stays in registers */
#pragma unroll
                            for(int k = 0; k < NS; k += 1) cc[k] = c[k];
                            dump_path<NS>(L.record_dump, L.path_dump, L.path_words, rec + slot * stride, cc, ALLFAST ? spool + ix.light_pairs : nullptr,
                                          (size_t)lp * spp + (paired ? q0 + slot : slot - px * spp), n, lane16);
                        }
                    }
                }
                DRT_PHASE_CUT(DRT_PHASE_REPLAY);
                if constexpr(ALLFAST)
                {
                    if(paired) film.unpark(park);
                    else start_film();
                    film.add_batch(half == 0 ? nzero : 0u, bs, spool + ix.light_pairs, lane16);
                }
                if(!paired)
                {
                    film.merge_halves();
                    if(have_film) store_pixel(gpix, film);
                }
            }
            __syncwarp();
            DRT_PHASE_CUT(DRT_PHASE_BOOK);
            /* A warp that ends its pixel here has passed both gates of this batch, like one that ends it with its last batch: the
             * phase gates of the classed kernel see no difference. */
            if constexpr(ADAPTIVE)
                if(pixel_converged<NS>(film, L, n, lane16)) { traced -= total - (q0 + count); break; }
        }
        if(paired)
        {
            film.merge_halves();
            if(have_film) store_pixel(task_y * L.width + task_x, film);
        }
    }

    DRT_PHASE_CUT(DRT_PHASE_OTHER);
    /* work counters: one shared-memory atomic per warp per counter, then one global atomic per CTA per counter */
#pragma unroll
    for(int k = 0; k < 4; k += 1)
    {
        unsigned long long v = tally[k];
#pragma unroll
        for(int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
        if(lane == 0) atomicAdd(&s_stats[1 + k], v);
    }
    if(lane == 0) atomicAdd(&s_stats[0], (unsigned long long)traced);
    __syncthreads();
    if(threadIdx.x < 14 && s_stats[threadIdx.x])
        atomicAdd(reinterpret_cast<unsigned long long *>(L.stats) + threadIdx.x, s_stats[threadIdx.x]);
#ifdef DRT_PHASE_CLOCKS
    if(threadIdx.x < 4) atomicAdd(&L.stats->phase_clocks[threadIdx.x], s_phase[threadIdx.x]);
#endif
