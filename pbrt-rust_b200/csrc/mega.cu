// The one-kernel forms of the path tracer: k_zt_mega ((0,2)-sequence sampler under the path integrator), k_vol_mega (volpath) and
// k_vol_mega_grid (volpath with grid media), with their launchers.  They are compiled with the exact-arithmetic flags of render.cu, but
// in a translation unit of their own (csrc/Makefile): their out-of-line per-material shade bodies are the slowest thing ptxas sees in
// this library (with the textured bin they took the build from 3 to 7.5 minutes inside render.o), and as a separate unit they compile
// next to render.cu instead of after it.
#include "path.cuh"

namespace pb {

// The (0,2)-sequence sampler under the PathIntegrator, one kernel: a tile's paths are inherently serial (every draw of
// every path advances the tile's PCG32), so the wavefront form spends its time launching 13 kernels per path segment for a
// few hundred threads.  Here ONE thread per tile (one warp per CTA, lane 0 working) walks its tile's pixels, samples and
// bounces start to finish -- camera sample, closest hit, shade, shadow ray, MIS ray, film -- with the same device
// functions, in the same order per tile, hence the same random stream and the same image as the wavefront form.
template <int BIN, bool INST>
static __device__ __noinline__ ShadeOut zt_shade(const RenderDev* Rp, uint32_t id) { return shade_path<BIN, INST, true>(*Rp, id); }
template <bool INST>
__global__ void __launch_bounds__(32 * PB_ZT_WARPS) k_zt_mega(RenderDev R, const RenderDev* Rdev, uint32_t lanes) {
    // `lanes` tiles per warp: 1 when there are few tiles (pure latency), more when one-lane warps would fill the issue slots.  The warps of a CTA pass
    // the phases of a trip together (barriers between them), as k_vol_mega's do and for the same reason: the instruction cache.
    const uint32_t warp = threadIdx.x >> 5, ln = threadIdx.x & 31u;
    const uint32_t j = (blockIdx.x * (blockDim.x >> 5) + warp) * lanes + ln;
    unsigned long long n_camera = 0, n_closest = 0, n_shadow = 0, n_zero = 0, n_iter = 0;
    bool ok = false;
    if (ln < lanes && j < R.n_tiles_sel) {
        uint32_t t = R.tile_begin + ((j / R.tile_group) * R.tile_mod + R.tile_rem) * R.tile_group + (j % R.tile_group);
        ZtTile* tp = R.zt.tiles + j;
        R.pixel[j] = PB_NO_SAMPLE;
        int tx, ty;
        if (tile_xy(R, t, &tx, &ty) && t < R.tile_end) {
            int x0 = R.sampler.sb[0] + tx * 16, y0 = R.sampler.sb[1] + ty * 16;
            int x1 = min(x0 + 16, R.sampler.sb[2]), y1 = min(y0 + 16, R.sampler.sb[3]);
            tp->x0 = x0; tp->y0 = y0; tp->w = (uint32_t)max(x1 - x0, 0); tp->npix = tp->w * (uint32_t)max(y1 - y0, 0);
            tp->pixel_idx = 0; tp->sample_idx = 0; tp->cur1d = 0; tp->cur2d = 0;
            zt_set_sequence(*tp, (unsigned long long)((long long)ty * R.ntx + tx));
            ok = zt_next_path(R, j, true);
        }
    }
    uint2 stack_mem[PB_STACK_SIZE(INST)];
    LocalStack stack{stack_mem};
    // ONE flat loop, a path vertex per trip: a lane whose path has ended goes on to its tile's next sample in the same trip count as its
    // neighbours' next vertex, instead of waiting at the end of a nested path loop for the warp's longest path.
    if (ok) n_camera += 1;
    for (;;) {
        if (!__syncthreads_or(ok)) break;
        int bin = Q_MISS;
        TravRay r;
        if (ok) {
            n_iter += 1;
            float4 a = R.ray[2 * j], b = R.ray[2 * j + 1];
            trav_init(R.scene, r, f3(a.x, a.y, a.z), f3(b.x, b.y, b.z), a.w);
            trav_run<false, INST>(R.scene, r, stack, 0);
            n_closest += 1;
            bin = store_closest_hit(R, j, r);
        }
        __syncthreads();
        ShadeOut o = {false, false, false, false, false};
        if (ok) {
            switch (bin) {
                case Q_MATTE: o = zt_shade<Q_MATTE, INST>(Rdev, j); break;
                case Q_PLASTIC: o = zt_shade<Q_PLASTIC, INST>(Rdev, j); break;
                case Q_MIRROR: o = zt_shade<Q_MIRROR, INST>(Rdev, j); break;
                case Q_GLASS: o = zt_shade<Q_GLASS, INST>(Rdev, j); break;
                case Q_METAL: o = zt_shade<Q_METAL, INST>(Rdev, j); break;
                case Q_NOMAT: o = zt_shade<Q_NOMAT, INST>(Rdev, j); break;
                case Q_TEX: o = zt_shade<Q_TEX, INST>(Rdev, j); break;
                default: o = zt_shade<Q_MISS, INST>(Rdev, j); break;
            }
            if (o.zero_rad) n_zero += 1;
        }
        __syncthreads();
        if (ok && o.push_shadow) {
            float4 a = R.sh_ray[2 * j], b = R.sh_ray[2 * j + 1];
            trav_init(R.scene, r, f3(a.x, a.y, a.z), f3(b.x, b.y, b.z), a.w);
            trav_run<true, INST>(R.scene, r, stack, 0);
            n_shadow += 1;
            if (!r.found) shadow_unoccluded(R, j);
        }
        __syncthreads();
        if (ok && o.push_mis) {
            float4 a = R.mis_ray[2 * j], b = R.mis_ray[2 * j + 1];
            trav_init(R.scene, r, f3(a.x, a.y, a.z), f3(b.x, b.y, b.z), a.w);
            trav_run<false, INST>(R.scene, r, stack, 0);
            n_closest += 1;
            mis_resolve<INST>(R, j, r);
        }
        if (ok && !o.push_next) {
            // finished path -> film (integrator.rs:350-368 sanity rule), then the tile's next sample
            float4 Le = R.L_eta[j];
            rgb L(Le.x, Le.y, Le.z);
            float y = lum(L);
            if (L.r != L.r || L.g != L.g || L.b != L.b) L = rgb(0.0f);
            else if (y < -1.0e-5f) L = rgb(0.0f);
            else if (isinf(y)) L = rgb(0.0f);
            film_add_sample_lane(R, R.pfilm[j], L);
            ok = zt_next_path(R, j, false);
            if (ok) n_camera += 1;
        }
    }
    atomicAdd(&R.cnt->camera_rays, n_camera); atomicAdd(&R.cnt->closest_rays, n_closest); atomicAdd(&R.cnt->shadow_rays, n_shadow);
    atomicAdd(&R.cnt->zero_radiance, n_zero); atomicMax(&R.cnt->iterations, n_iter);
}


// ---------------------------------------------------------------------------
// VolPathIntegrator (src/integrators/volpath.rs:82-221) with homogeneous media: one kernel, a thread per path
// ---------------------------------------------------------------------------
// A volumetric path is a chain of data-dependent loops -- medium sampling in front of every vertex, the two transmittance loops of
// estimate_direct (VisibilityTester::tr, Scene::intersect_tr) that walk through any number of material-less boundaries, a sample
// stream whose length depends on which of them ran -- so it is written as the reference writes it: one thread owns a path from its
// camera sample to the film, claims the next camera sample when it is done (warp-aggregated fetch-add on the call's item cursor),
// and calls the same traversal (exact TU) and shading functions as the surface path integrator.  Path state lives in the slot
// arrays of RenderDev (slot = global thread index), the volume-only state in the thread (VolState).

// HomogeneousMedium::sample (homogeneous.rs:35-72) in front of the vertex the path ray of slot `id` has just found, then volpath.rs:114.
// Returns 0: no medium interaction (go on with the surface / the miss), 1: interaction sampled at vs->mi_p, 2: beta is black.
PB_D int vol_sample_medium(const RenderDev& R, uint32_t id, VolState* vs, bool found, float t_hit) {
    float4 bs = R.beta_st[id];
    rgb beta(bs.x, bs.y, bs.z);
    bool sampled = false;
    if (vs->medium >= 0) {
        const float4 ra = R.ray[2 * id], rb = R.ray[2 * id + 1];
        const f3 o(ra.x, ra.y, ra.z), d(rb.x, rb.y, rb.z);
        const float t_max = found ? t_hit : ra.w;  // Scene::intersect leaves the hit distance in ray.t_max
        DirectSampler smp;
        smp.prefetch(R, id);
        const pbrt_b200_medium m = R.scene.media[vs->medium];
        const rgb st = medium_sigma_t(m), ss = rgb3(m.sigma_s);
        const int channel = min((int)(smp.get_1d() * 3.0f), 2);
        const float stc = channel == 0 ? st.r : (channel == 1 ? st.g : st.b);
        const float dist = -logf(1.0f - smp.get_1d()) / stc;
        const float dl = len(d);
        const float t = fminf(dist / dl, t_max);
        sampled = t < t_max;
        if (sampled) vs->mi_p = o + d * t;
        const float tt = fminf(t, PB_FLT_MAX);
        const rgb Tr(expf((-st.r * tt) * dl), expf((-st.g * tt) * dl), expf((-st.b * tt) * dl));
        const rgb density = sampled ? st * Tr : Tr;
        float pdf = 0.0f;
        pdf += density.r; pdf += density.g; pdf += density.b;
        pdf *= 1.0f / 3.0f;
        if (pdf == 0.0f) pdf = 1.0f;
        beta = beta * (sampled ? Tr * ss / pdf : Tr / pdf);
        R.beta_st[id] = make_float4(beta.r, beta.g, beta.b, bs.w);
        smp.end(R, id);
    }
    if (is_black(beta)) return 2;
    return sampled ? 1 : 0;
}

// The medium branch of VolPathIntegrator::li (volpath.rs:117-133): uniform_sample_onelight / estimate_direct with the phase function
// in the BSDF's place (integrator.rs:140-146,183-188), then HenyeyGreenstein::sample_p for the next direction.
// PART as in shade_path: 0 = the whole vertex; 1 = up to the light sample (a vertex that goes on returns neither push_next nor
// push_dead); 2 = the new direction and roulette (k_vol_mega_grid).
template <bool INST, int PART = 0>
static __device__ __noinline__ ShadeOut vol_shade_medium(const RenderDev* Rp, uint32_t id, VolState* vs) {
    const RenderDev& R = *Rp;
    ShadeOut out{false, false, false, false, false};
    const float4 rb = R.ray[2 * id + 1];
    const f3 rd(rb.x, rb.y, rb.z);
    const float time = rb.w;
    float4 Le = R.L_eta[id], bs = R.beta_st[id];
    rgb beta(bs.x, bs.y, bs.z);
    uint32_t st = __float_as_uint(bs.w);
    uint32_t bounces = st & 0xffffu;
    if (bounces >= (uint32_t)R.max_depth) { out.push_dead = true; return out; }
    DirectSampler smp;
    smp.prefetch(R, id);
    const f3 p = vs->mi_p, wo = -rd, zero(0.f, 0.f, 0.f);
    const float g = R.scene.media[vs->medium].g;
    if constexpr (PART != 2) if (R.n_lights > 0) {
        float u1 = smp.get_1d();
        const float* ld_cdf = R.ld_cdf; const float* ld_func = R.ld_func; float ld_func_int = R.ld_func_int;
        if (R.sp.enabled) {
            int sl = R.sp.slot[spatial_voxel(R, p)];
            if (sl >= 0) { ld_cdf = R.sp.cdf + (size_t)sl * (R.n_lights + 1); ld_func = R.sp.func + (size_t)sl * R.n_lights; ld_func_int = R.sp.func_int[sl]; }
            else atomicExch(R.sp.counters + 2, 1u);
        }
        uint32_t ln = find_interval_cdf(ld_cdf, (int)R.n_lights + 1, u1);
        float selpdf = ld_func_int > 0.0f ? ld_func[ln] / (ld_func_int * (float)R.n_lights) : 0.0f;
        bool zero_rad = true;
        if (selpdf != 0.0f) {
            float2 ulight = smp.get_2d();
            float2 uscatt = smp.get_2d();
            const pbrt_b200_light& light = R.scene.lights[ln];
            bool delta = is_delta_light(light);
            LightSample ls;
            light_sample_li<INST>(R, ln, p, ulight, ls, zero, zero);
            if (ls.pdf > 0.0f && !is_black(ls.Li)) {
                float ph = phase_hg(dot(wo, ls.wi), g);
                if (ph != 0.0f) {
                    f3 o = offset_ray_origin(p, zero, zero, ls.p1 - p);
                    f3 tg = offset_ray_origin(ls.p1, ls.p1_err, ls.p1_n, o - ls.p1);
                    f3 d = tg - o;
                    rgb f(ph);
                    rgb Ld = delta ? f * ls.Li / ls.pdf : f * ls.Li * power_heuristic(ls.pdf, ph) / ls.pdf;
                    rgb add = beta * (Ld / selpdf);
                    store_ray(R.sh_ray, id, o, d, 1.0f - PB_SHADOW_EPSILON, time);
                    R.sh_contrib[id] = make_float4(add.r, add.g, add.b, 0.f);
                    vs->sh_medium = vs->medium; vs->p1 = ls.p1; vs->p1_err = ls.p1_err; vs->p1_n = ls.p1_n;
                    out.push_shadow = true;
                    zero_rad = false;
                }
            }
            if (!delta) {
                f3 wi(0.f, 0.f, 0.f);
                float ph = hg_sample_p(g, wo, &wi, uscatt);
                if (ph != 0.0f && ph > 0.0f) {
                    Surf ref;
                    ref.p = p; ref.p_error = zero; ref.n = zero; ref.wo = wo; ref.sh_n = zero; ref.sh_dpdu = zero;
                    float lpdf = light_pdf_li<INST>(R, ln, ref, wi);
                    if (lpdf != 0.0f) {
                        float weight = power_heuristic(ph, lpdf);
                        rgb fac = beta * (rgb(ph) * weight / ph / selpdf);
                        store_ray(R.mis_ray, id, offset_ray_origin(p, zero, zero, wi), wi, PB_INF, time);
                        R.mis_contrib[id] = make_float4(fac.r, fac.g, fac.b, __uint_as_float(ln));
                        vs->mis_medium = vs->medium;
                        out.push_mis = true;
                        zero_rad = false;
                    }
                }
            }
        }
        out.zero_rad = zero_rad;
    }
    if constexpr (PART == 1) { smp.end(R, id); return out; }
    // volpath.rs:127-132: new direction from the phase function; the ray stays in the medium
    f3 wi(0.f, 0.f, 0.f);
    hg_sample_p(g, wo, &wi, smp.get_2d());
    store_ray(R.ray, id, offset_ray_origin(p, zero, zero, wi), wi, PB_INF, time);
    bool alive = true;
    {   // Russian roulette, volpath.rs:206-214 (specular_bounce = false)
        rgb rrbeta = beta * Le.w;
        float mc = max_comp(rrbeta);
        if (mc < R.rr_threshold && bounces > 3) {
            float qv = fmaxf(1.0f - mc, 0.05f);
            if (smp.get_1d() < qv) alive = false;
            else beta = beta / (1.0f - qv);
        }
    }
    smp.end(R, id);
    if (alive) {
        bounces += 1;
        R.beta_st[id] = make_float4(beta.r, beta.g, beta.b, __uint_as_float(bounces));
        out.push_next = true;
    } else out.push_dead = true;
    return out;
}

template <int BIN, bool INST, int PART = 0>
static __device__ __noinline__ ShadeOut vol_shade(const RenderDev* Rp, uint32_t id, VolState* vs) { return shade_path<BIN, INST, false, true, PART>(*Rp, id, vs); }

#define PB_VOL_SEGMENT_CAP 4096u   /* transmittance loops: boundaries crossed by one shadow / MIS ray before it is given up (hang guard) */
#define PB_VOL_VERTEX_CAP 65536u   /* path loop: boundary crossings lower the bounce count, so max_depth alone does not bound it */
#define PB_VOL_TRACK_CAP 65536u    /* grid media: steps of one delta / ratio tracking loop before the path is ended (hang guard; oracle: ORC_VOL_TRACK_CAP) */
template <bool INST>
__global__ void __launch_bounds__(PB_VOL_BLOCK) k_vol_mega(RenderDev R, const RenderDev* Rdev, unsigned long long total_items, int camera_medium) {
    const uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;  // slot
    const unsigned lane = threadIdx.x & 31u;
    unsigned long long n_camera = 0, n_closest = 0, n_zero = 0, n_iter = 0;
    uint2 stack_mem[PB_STACK_SIZE(INST)];
    LocalStack stack{stack_mem};
    VolState vs;
    // ONE flat loop, a path vertex per trip: a lane whose path has ended claims its next camera sample at the top of the following trip, so the
    // warp stays full and every lane is in the same phase of a vertex (trace, medium / surface shade, shadow walk, MIS walk).  The nested form
    // (a path loop inside a sample loop) reconverged only when the warp's LONGEST path had ended: lanes idled for the rest of it.
    bool have = false, exhausted = false, alive = false;
    uint32_t vertices = 0;
    for (;;) {
        {   // lanes without a path share one fetch-add
            const bool need = !have && !exhausted;
            const unsigned m = __ballot_sync(0xffffffffu, need);
            if (need) {
                const int leader = __ffs(m) - 1;
                unsigned long long base = 0;
                if ((int)lane == leader) base = atomicAdd(&R.cnt->item_cursor, (unsigned long long)__popc(m));
                base = __shfl_sync(m, base, leader);
                const unsigned long long item = base + (unsigned long long)__popc(m & ((1u << lane) - 1u));
                if (item >= total_items) exhausted = true;
                else if (gen_camera_path(R, item, j)) {
                    n_camera += 1;
                    vs.medium = camera_medium;
                    have = true; alive = true; vertices = 0;
                }
            }
        }
        // ncu on the 64-thread form: issue slots 7 % busy, 52 of 57 stall cycles per instruction are `no_instruction` -- sixteen warps per SM each
        // somewhere else in 100s of KB of code miss the instruction cache all the time.  One 512-thread CTA per SM whose warps pass the phases of a
        // trip TOGETHER (barriers between trace / shade / shadow walk / MIS walk) keeps the SM inside one region of the code at a time.
        if (!__syncthreads_or(have || !exhausted)) break;
        if (have) {
            if (vertices++ >= PB_VOL_VERTEX_CAP) alive = false;
        }
        int bin = Q_MISS, ms = 2;
        TravRay r;
        if (have && alive) {
            n_iter += 1;
            {
                float4 a = R.ray[2 * j], b = R.ray[2 * j + 1];
                trav_init(R.scene, r, f3(a.x, a.y, a.z), f3(b.x, b.y, b.z), a.w);
                trav_run<false, INST>(R.scene, r, stack, 0);
                n_closest += 1;
            }
            bin = store_closest_hit(R, j, r);
            ms = vol_sample_medium(R, j, &vs, r.found, r.hit.t);
        }
        __syncthreads();
        ShadeOut o = {false, false, false, false, false};  // ms == 2: the path ends here (volpath.rs:114)
        if (have && alive) {
            if (ms == 2) {}
            else if (ms == 1) o = vol_shade_medium<INST>(Rdev, j, &vs);
            else switch (bin) {
                case Q_MATTE: o = vol_shade<Q_MATTE, INST>(Rdev, j, &vs); break;
                case Q_PLASTIC: o = vol_shade<Q_PLASTIC, INST>(Rdev, j, &vs); break;
                case Q_MIRROR: o = vol_shade<Q_MIRROR, INST>(Rdev, j, &vs); break;
                case Q_GLASS: o = vol_shade<Q_GLASS, INST>(Rdev, j, &vs); break;
                case Q_METAL: o = vol_shade<Q_METAL, INST>(Rdev, j, &vs); break;
                case Q_NOMAT: o = vol_shade<Q_NOMAT, INST>(Rdev, j, &vs); break;
                case Q_TEX: if (INST) { o = vol_shade<Q_TEX, true>(Rdev, j, &vs); break; }  // textured scenes run the full-featured family (launch_vol_mega)
                default: o = vol_shade<Q_MISS, INST>(Rdev, j, &vs); break;
            }
            if (o.zero_rad) n_zero += 1;
        }
        __syncthreads();
        if (have && alive) {
            if (o.push_shadow) {  // VisibilityTester::tr, light.rs:125-150
                float4 a = R.sh_ray[2 * j], b = R.sh_ray[2 * j + 1];
                f3 ro(a.x, a.y, a.z), rdir(b.x, b.y, b.z);
                float t_max = a.w;
                int med = vs.sh_medium;
                rgb Tr(1.0f);
                bool blocked = false;
                for (uint32_t seg = 0;; ++seg) {
                    if (seg >= PB_VOL_SEGMENT_CAP) { blocked = true; break; }
                    trav_init(R.scene, r, ro, rdir, t_max);
                    trav_run<false, INST>(R.scene, r, stack, 0);
                    n_closest += 1;
                    if (r.found && R.scene.prims[r.hit.slot].material >= 0) { blocked = true; break; }
                    if (med >= 0) Tr = Tr * medium_tr(R.scene.media[med], rdir, r.found ? r.hit.t : t_max);
                    if (!r.found) break;
                    uint32_t fl;
                    Surf si = surface_at_hit<INST>(R.scene, r.hit.inst, r.hit.slot, ro, rdir, r.hit.t, r.hit.b0, r.hit.b1, r.hit.b2, &fl);
                    const VolInterface mi = vol_hit_interface(R.scene, r.hit.slot, med);
                    const f3 o2 = offset_ray_origin(si.p, si.p_error, si.n, vs.p1 - si.p);  // spawn_rayto_interaction, interaction.rs:46-52
                    const f3 tg = offset_ray_origin(vs.p1, vs.p1_err, vs.p1_n, o2 - vs.p1);
                    rdir = tg - o2; ro = o2; t_max = 1.0f - PB_SHADOW_EPSILON;
                    med = vol_medium_for(mi, si.n, rdir);
                }
                if (!blocked) {
                    float4 c = R.sh_contrib[j], L = R.L_eta[j];
                    L.x += c.x * Tr.r; L.y += c.y * Tr.g; L.z += c.z * Tr.b;
                    R.L_eta[j] = L;
                }
            }
        }
        __syncthreads();
        if (have && alive) {
            if (o.push_mis) {  // Scene::intersect_tr, scene.rs:68-87, then integrator.rs:218-232
                float4 a = R.mis_ray[2 * j], b = R.mis_ray[2 * j + 1];
                f3 ro(a.x, a.y, a.z);
                const f3 rdir(b.x, b.y, b.z);
                int med = vs.mis_medium;
                const float4 c = R.mis_contrib[j];
                const uint32_t ln = __float_as_uint(c.w);
                rgb Tr(1.0f), li(0.0f);
                for (uint32_t seg = 0; seg < PB_VOL_SEGMENT_CAP; ++seg) {
                    trav_init(R.scene, r, ro, rdir, PB_INF);
                    trav_run<false, INST>(R.scene, r, stack, 0);
                    n_closest += 1;
                    if (med >= 0) Tr = Tr * medium_tr(R.scene.media[med], rdir, r.found ? r.hit.t : PB_INF);
                    if (!r.found) {
                        const pbrt_b200_light& l = R.scene.lights[ln];
                        if (l.type == PBRT_B200_LIGHT_INFINITE) li = rgb3(l.L);
                        break;
                    }
                    const pbrt_b200_prim pr = R.scene.prims[r.hit.slot];
                    uint32_t fl;
                    Surf si = surface_at_hit<INST>(R.scene, r.hit.inst, r.hit.slot, ro, rdir, r.hit.t, r.hit.b0, r.hit.b1, r.hit.b2, &fl);
                    if (pr.material >= 0) {
                        if (pr.area_light == (int)ln) {
                            const pbrt_b200_light& al = R.scene.lights[ln];
                            if (al.two_sided || dot(si.n, -rdir) > 0.0f) li = rgb3(al.L);
                        }
                        break;
                    }
                    const VolInterface mi = vol_hit_interface(R.scene, r.hit.slot, med);
                    ro = offset_ray_origin(si.p, si.p_error, si.n, rdir);
                    med = vol_medium_for(mi, si.n, rdir);
                }
                if (!is_black(li)) {
                    float4 L = R.L_eta[j];
                    L.x += c.x * li.r * Tr.r; L.y += c.y * li.g * Tr.g; L.z += c.z * li.b * Tr.b;
                    R.L_eta[j] = L;
                }
            }
            alive = o.push_next;
        }
        if (have && !alive) {
            float4 Le = R.L_eta[j];
            rgb L(Le.x, Le.y, Le.z);
            float y = lum(L);  // integrator.rs:350-368
            if (L.r != L.r || L.g != L.g || L.b != L.b) L = rgb(0.0f);
            else if (y < -1.0e-5f) L = rgb(0.0f);
            else if (isinf(y)) L = rgb(0.0f);
            film_add_sample_lane(R, R.pfilm[j], L);
            have = false;
        }
    }
    atomicAdd(&R.cnt->camera_rays, n_camera); atomicAdd(&R.cnt->closest_rays, n_closest);
    atomicAdd(&R.cnt->zero_radiance, n_zero); atomicMax(&R.cnt->iterations, n_iter);
}

// ---------------------------------------------------------------------------
// GridDensityMedium (src/media/grid.rs, a port of pbrt-v3 media/grid.{h,cpp}), exact fp32 with the reference's operation order
// ---------------------------------------------------------------------------
// GridDensityMedium::d: 0 outside [0,nx) x [0,ny) x [0,nz)
PB_D float grid_d(const DevGrid& g, int x, int y, int z) {
    if (x < 0 || y < 0 || z < 0 || x >= (int)g.nx || y >= (int)g.ny || z >= (int)g.nz) return 0.0f;
    return __ldg(g.density + ((size_t)z * g.ny + (size_t)y) * g.nx + (size_t)x);
}
PB_D float grid_lerp(float t, float a, float b) { return (1.0f - t) * a + t * b; }  // pbrt.rs lerp
// GridDensityMedium::density: trilinear over the voxel centres (no hardware filtering: its 8-bit weights are not this arithmetic)
PB_D float grid_density(const DevGrid& g, f3 p) {
    const float sx = p.x * (float)g.nx - 0.5f, sy = p.y * (float)g.ny - 0.5f, sz = p.z * (float)g.nz - 0.5f;
    const float fx = floorf(sx), fy = floorf(sy), fz = floorf(sz);
    const int x = (int)fx, y = (int)fy, z = (int)fz;
    const float dx = sx - fx, dy = sy - fy, dz = sz - fz;
    const float d00 = grid_lerp(dx, grid_d(g, x, y, z), grid_d(g, x + 1, y, z));
    const float d10 = grid_lerp(dx, grid_d(g, x, y + 1, z), grid_d(g, x + 1, y + 1, z));
    const float d01 = grid_lerp(dx, grid_d(g, x, y, z + 1), grid_d(g, x + 1, y, z + 1));
    const float d11 = grid_lerp(dx, grid_d(g, x, y + 1, z + 1), grid_d(g, x + 1, y + 1, z + 1));
    const float d0 = grid_lerp(dy, d00, d10), d1 = grid_lerp(dy, d01, d11);
    return grid_lerp(dz, d0, d1);
}
// The common head of sample / tr: world_to_medium(Ray(o, normalize(d), t_max * |d|)) (Transform::transform_ray with its
// origin nudge), clipped to Bounds3(0,0,0)-(1,1,1) by the t0/t1 form of Bounds3::intersect_p.  false: the ray misses the box.
PB_D bool grid_clip(const DevGrid& g, f3 o, f3 d, float t_max, f3* mo, f3* md, float* t0_out, float* t1_out) {
    float mt;
    xf_ray(g.world_to_medium, o, normalize(d), t_max * len(d), mo, md, &mt);
    float t0 = 0.0f, t1 = mt;
    const float ro[3] = {mo->x, mo->y, mo->z}, rd[3] = {md->x, md->y, md->z};
    for (int i = 0; i < 3; ++i) {
        const float inv = 1.0f / rd[i];
        float tn = (0.0f - ro[i]) * inv, tf = (1.0f - ro[i]) * inv;
        if (tn > tf) { const float tmp = tn; tn = tf; tf = tmp; }
        tf *= 1.0f + 2.0f * gamma_n(3);
        t0 = tn > t0 ? tn : t0;
        t1 = tf < t1 ? tf : t1;
        if (t0 > t1) return false;
    }
    *t0_out = t0; *t1_out = t1;
    return true;
}
// One tracking step, t -= ln(1 - u) * inv_max_density / sigma_t.  A grid whose sigma_t * max_density is 0 (an all-zero grid) is
// vacuum: sample and tr return weight 1 before they draw anything (instead of stepping by 0 * inf), so such a scene uses the sample
// stream -- and renders the image -- of the same scene without the medium.
PB_D bool grid_is_vacuum(const DevGrid& g, float sigma_t) { return !(g.max_density > 0.0f && sigma_t > 0.0f); }
PB_D float grid_step(const DevGrid& g, float sigma_t, float t, float u) { return t - logf(1.0f - u) * g.inv_max_density / sigma_t; }
// GridDensityMedium::sample (delta tracking).  Returns true with *p = ray_world(t) and *w = sigma_s / sigma_t when it samples an
// interaction; otherwise *w = 1.  *gave_up: the loop ran PB_VOL_TRACK_CAP steps.
PB_D bool grid_sample(const DevGrid& g, const pbrt_b200_medium& m, f3 o, f3 d, float t_max, DirectSampler& smp, f3* p, rgb* w, bool* gave_up) {
    *w = rgb(1.0f);
    f3 mo, md;
    float t0, t1;
    const float st = m.sigma_a[0] + m.sigma_s[0];
    if (grid_is_vacuum(g, st) || !grid_clip(g, o, d, t_max, &mo, &md, &t0, &t1)) return false;
    float t = t0;
    for (uint32_t k = 0;; ++k) {
        if (k >= PB_VOL_TRACK_CAP) { *gave_up = true; return false; }
        t = grid_step(g, st, t, smp.get_1d());
        if (t >= t1) break;
        if (grid_density(g, mo + md * t) * g.inv_max_density > smp.get_1d()) {
            *p = o + d * t;
            *w = rgb(m.sigma_s[0] / st, m.sigma_s[1] / st, m.sigma_s[2] / st);
            return true;
        }
    }
    return false;
}
// GridDensityMedium::tr (ratio tracking with Russian roulette); unlike HomogeneousMedium::tr it draws from the sampler.
PB_D float grid_tr(const DevGrid& g, const pbrt_b200_medium& m, f3 o, f3 d, float t_max, DirectSampler& smp, bool* gave_up) {
    f3 mo, md;
    float t0, t1;
    const float st = m.sigma_a[0] + m.sigma_s[0];
    if (grid_is_vacuum(g, st) || !grid_clip(g, o, d, t_max, &mo, &md, &t0, &t1)) return 1.0f;
    float tr = 1.0f, t = t0;
    for (uint32_t k = 0;; ++k) {
        if (k >= PB_VOL_TRACK_CAP) { *gave_up = true; return 0.0f; }
        t = grid_step(g, st, t, smp.get_1d());
        if (t >= t1) break;
        tr *= 1.0f - fmaxf(0.0f, grid_density(g, mo + md * t) * g.inv_max_density);
        if (tr < 0.1f) {
            const float q = fmaxf(0.05f, 1.0f - tr);
            if (smp.get_1d() < q) return 0.0f;
            tr /= 1.0f - q;
        }
    }
    return tr;
}
// Medium::tr of either kind
PB_D rgb vol_medium_tr(const pbrt_b200_medium& m, const DevGrid* grids, f3 o, f3 d, float t_max, DirectSampler& smp, bool* gave_up) {
    if (m.grid == 0) return medium_tr(m, d, t_max);
    return rgb(grid_tr(grids[m.grid - 1], m, o, d, t_max, smp, gave_up));
}
// vol_sample_medium for scenes with grid media: Medium::sample of either kind in front of the vertex, then volpath.rs:114.
// Returns 0 / 1 / 2 as vol_sample_medium, and 2 when the tracking loop gave up.
PB_D int vol_sample_medium_grid(const RenderDev& R, const DevGrid* grids, uint32_t id, VolState* vs, bool found, float t_hit) {
    if (vs->medium < 0 || R.scene.media[vs->medium].grid == 0) return vol_sample_medium(R, id, vs, found, t_hit);
    const pbrt_b200_medium m = R.scene.media[vs->medium];
    float4 bs = R.beta_st[id];
    const float4 ra = R.ray[2 * id], rb = R.ray[2 * id + 1];
    DirectSampler smp;
    smp.prefetch(R, id);
    rgb w;
    bool gave_up = false;
    const bool sampled = grid_sample(grids[m.grid - 1], m, f3(ra.x, ra.y, ra.z), f3(rb.x, rb.y, rb.z), found ? t_hit : ra.w, smp, &vs->mi_p, &w, &gave_up);
    smp.end(R, id);
    if (gave_up) return 2;
    const rgb beta = rgb(bs.x, bs.y, bs.z) * w;
    R.beta_st[id] = make_float4(beta.r, beta.g, beta.b, bs.w);
    if (is_black(beta)) return 2;
    return sampled ? 1 : 0;
}

// Volpath for scenes with grid media.  Their transmittance loops draw from the sampler, and the reference draws those samples between the
// light sample and the next direction (estimate_direct, then BSDF::sample_f / phase sampling and roulette), so a vertex runs in two
// halves around the walks and a trip has five phases: trace + medium sampling, direct lighting (PART 1), shadow walk, MIS walk,
// continuation (PART 2).  Barriers between the phases as in k_vol_mega.  Full-featured: instances, sphere lights and every bin.
__global__ void __launch_bounds__(PB_VOL_BLOCK) k_vol_mega_grid(RenderDev R, const RenderDev* Rdev, unsigned long long total_items, int camera_medium, const DevGrid* grids) {
    constexpr bool INST = true;
    const uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;  // slot
    const unsigned lane = threadIdx.x & 31u;
    unsigned long long n_camera = 0, n_closest = 0, n_zero = 0, n_iter = 0;
    uint2 stack_mem[PB_STACK_SIZE(INST)];
    LocalStack stack{stack_mem};
    VolState vs;
    // ONE flat loop, a path vertex per trip: a lane whose path has ended claims its next camera sample at the top of the following trip, so the
    // warp stays full and every lane is in the same phase of a vertex (trace, medium / surface shade, shadow walk, MIS walk).  The nested form
    // (a path loop inside a sample loop) reconverged only when the warp's LONGEST path had ended: lanes idled for the rest of it.
    bool have = false, exhausted = false, alive = false;
    uint32_t vertices = 0;
    for (;;) {
        {   // lanes without a path share one fetch-add
            const bool need = !have && !exhausted;
            const unsigned m = __ballot_sync(0xffffffffu, need);
            if (need) {
                const int leader = __ffs(m) - 1;
                unsigned long long base = 0;
                if ((int)lane == leader) base = atomicAdd(&R.cnt->item_cursor, (unsigned long long)__popc(m));
                base = __shfl_sync(m, base, leader);
                const unsigned long long item = base + (unsigned long long)__popc(m & ((1u << lane) - 1u));
                if (item >= total_items) exhausted = true;
                else if (gen_camera_path(R, item, j)) {
                    n_camera += 1;
                    vs.medium = camera_medium;
                    have = true; alive = true; vertices = 0;
                }
            }
        }
        // ncu on the 64-thread form: issue slots 7 % busy, 52 of 57 stall cycles per instruction are `no_instruction` -- sixteen warps per SM each
        // somewhere else in 100s of KB of code miss the instruction cache all the time.  One 512-thread CTA per SM whose warps pass the phases of a
        // trip TOGETHER (barriers between trace / shade / shadow walk / MIS walk) keeps the SM inside one region of the code at a time.
        if (!__syncthreads_or(have || !exhausted)) break;
        if (have) {
            if (vertices++ >= PB_VOL_VERTEX_CAP) alive = false;
        }
        int bin = Q_MISS, ms = 2;
        TravRay r;
        if (have && alive) {
            n_iter += 1;
            {
                float4 a = R.ray[2 * j], b = R.ray[2 * j + 1];
                trav_init(R.scene, r, f3(a.x, a.y, a.z), f3(b.x, b.y, b.z), a.w);
                trav_run<false, INST>(R.scene, r, stack, 0);
                n_closest += 1;
            }
            bin = store_closest_hit(R, j, r);
            ms = vol_sample_medium_grid(R, grids, j, &vs, r.found, r.hit.t);
        }
        __syncthreads();
        ShadeOut o = {false, false, false, false, false};  // ms == 2: the path ends here (volpath.rs:114)
        if (have && alive) {
            if (ms == 2) {}
            else if (ms == 1) o = vol_shade_medium<INST, 1>(Rdev, j, &vs);
            else switch (bin) {
                case Q_MATTE: o = vol_shade<Q_MATTE, INST, 1>(Rdev, j, &vs); break;
                case Q_PLASTIC: o = vol_shade<Q_PLASTIC, INST, 1>(Rdev, j, &vs); break;
                case Q_MIRROR: o = vol_shade<Q_MIRROR, INST, 1>(Rdev, j, &vs); break;
                case Q_GLASS: o = vol_shade<Q_GLASS, INST, 1>(Rdev, j, &vs); break;
                case Q_METAL: o = vol_shade<Q_METAL, INST, 1>(Rdev, j, &vs); break;
                case Q_NOMAT: o = vol_shade<Q_NOMAT, INST, 1>(Rdev, j, &vs); break;
                case Q_TEX: if (INST) { o = vol_shade<Q_TEX, true, 1>(Rdev, j, &vs); break; }
                default: o = vol_shade<Q_MISS, INST, 1>(Rdev, j, &vs); break;
            }
            if (o.zero_rad) n_zero += 1;
        }
        // the vertex's continuation is pending (PART 1 returned neither push_next nor push_dead); a tracking loop that gave up ends the path
        const bool cont = have && alive && ms != 2 && !o.push_next && !o.push_dead;
        bool gave_up = false;
        __syncthreads();
        if (have && alive) {
            if (o.push_shadow) {  // VisibilityTester::tr, light.rs:125-150
                float4 a = R.sh_ray[2 * j], b = R.sh_ray[2 * j + 1];
                f3 ro(a.x, a.y, a.z), rdir(b.x, b.y, b.z);
                float t_max = a.w;
                int med = vs.sh_medium;
                rgb Tr(1.0f);
                bool blocked = false;
                DirectSampler smp;
                smp.prefetch(R, j);
                for (uint32_t seg = 0;; ++seg) {
                    if (seg >= PB_VOL_SEGMENT_CAP) { blocked = true; break; }
                    trav_init(R.scene, r, ro, rdir, t_max);
                    trav_run<false, INST>(R.scene, r, stack, 0);
                    n_closest += 1;
                    if (r.found && R.scene.prims[r.hit.slot].material >= 0) { blocked = true; break; }
                    if (med >= 0) Tr = Tr * vol_medium_tr(R.scene.media[med], grids, ro, rdir, r.found ? r.hit.t : t_max, smp, &gave_up);
                    if (gave_up) { blocked = true; break; }
                    if (!r.found) break;
                    uint32_t fl;
                    Surf si = surface_at_hit<INST>(R.scene, r.hit.inst, r.hit.slot, ro, rdir, r.hit.t, r.hit.b0, r.hit.b1, r.hit.b2, &fl);
                    const VolInterface mi = vol_hit_interface(R.scene, r.hit.slot, med);
                    const f3 o2 = offset_ray_origin(si.p, si.p_error, si.n, vs.p1 - si.p);  // spawn_rayto_interaction, interaction.rs:46-52
                    const f3 tg = offset_ray_origin(vs.p1, vs.p1_err, vs.p1_n, o2 - vs.p1);
                    rdir = tg - o2; ro = o2; t_max = 1.0f - PB_SHADOW_EPSILON;
                    med = vol_medium_for(mi, si.n, rdir);
                }
                smp.end(R, j);
                if (!blocked) {
                    float4 c = R.sh_contrib[j], L = R.L_eta[j];
                    L.x += c.x * Tr.r; L.y += c.y * Tr.g; L.z += c.z * Tr.b;
                    R.L_eta[j] = L;
                }
            }
        }
        __syncthreads();
        if (have && alive) {
            if (o.push_mis) {  // Scene::intersect_tr, scene.rs:68-87, then integrator.rs:218-232
                float4 a = R.mis_ray[2 * j], b = R.mis_ray[2 * j + 1];
                f3 ro(a.x, a.y, a.z);
                const f3 rdir(b.x, b.y, b.z);
                int med = vs.mis_medium;
                const float4 c = R.mis_contrib[j];
                const uint32_t ln = __float_as_uint(c.w);
                rgb Tr(1.0f), li(0.0f);
                DirectSampler smp;
                smp.prefetch(R, j);
                for (uint32_t seg = 0; seg < PB_VOL_SEGMENT_CAP && !gave_up; ++seg) {
                    trav_init(R.scene, r, ro, rdir, PB_INF);
                    trav_run<false, INST>(R.scene, r, stack, 0);
                    n_closest += 1;
                    if (med >= 0) Tr = Tr * vol_medium_tr(R.scene.media[med], grids, ro, rdir, r.found ? r.hit.t : PB_INF, smp, &gave_up);
                    if (gave_up) break;
                    if (!r.found) {
                        const pbrt_b200_light& l = R.scene.lights[ln];
                        if (l.type == PBRT_B200_LIGHT_INFINITE) li = rgb3(l.L);
                        break;
                    }
                    const pbrt_b200_prim pr = R.scene.prims[r.hit.slot];
                    uint32_t fl;
                    Surf si = surface_at_hit<INST>(R.scene, r.hit.inst, r.hit.slot, ro, rdir, r.hit.t, r.hit.b0, r.hit.b1, r.hit.b2, &fl);
                    if (pr.material >= 0) {
                        if (pr.area_light == (int)ln) {
                            const pbrt_b200_light& al = R.scene.lights[ln];
                            if (al.two_sided || dot(si.n, -rdir) > 0.0f) li = rgb3(al.L);
                        }
                        break;
                    }
                    const VolInterface mi = vol_hit_interface(R.scene, r.hit.slot, med);
                    ro = offset_ray_origin(si.p, si.p_error, si.n, rdir);
                    med = vol_medium_for(mi, si.n, rdir);
                }
                smp.end(R, j);
                if (!gave_up && !is_black(li)) {
                    float4 L = R.L_eta[j];
                    L.x += c.x * li.r * Tr.r; L.y += c.y * li.g * Tr.g; L.z += c.z * li.b * Tr.b;
                    R.L_eta[j] = L;
                }
            }
            alive = (o.push_next || cont) && !gave_up;
        }
        __syncthreads();
        if (have && alive && cont) {  // phase 5: the continuation, after the walks have drawn their samples
            ShadeOut o2 = {false, false, false, false, false};
            if (ms == 1) o2 = vol_shade_medium<INST, 2>(Rdev, j, &vs);
            else switch (bin) {
                case Q_MATTE: o2 = vol_shade<Q_MATTE, INST, 2>(Rdev, j, &vs); break;
                case Q_PLASTIC: o2 = vol_shade<Q_PLASTIC, INST, 2>(Rdev, j, &vs); break;
                case Q_MIRROR: o2 = vol_shade<Q_MIRROR, INST, 2>(Rdev, j, &vs); break;
                case Q_GLASS: o2 = vol_shade<Q_GLASS, INST, 2>(Rdev, j, &vs); break;
                case Q_METAL: o2 = vol_shade<Q_METAL, INST, 2>(Rdev, j, &vs); break;
                case Q_NOMAT: o2 = vol_shade<Q_NOMAT, INST, 2>(Rdev, j, &vs); break;
                case Q_TEX: o2 = vol_shade<Q_TEX, INST, 2>(Rdev, j, &vs); break;
                default: break;  // a miss has no continuation
            }
            alive = o2.push_next;
        }
        if (have && !alive) {
            float4 Le = R.L_eta[j];
            rgb L(Le.x, Le.y, Le.z);
            float y = lum(L);  // integrator.rs:350-368
            if (L.r != L.r || L.g != L.g || L.b != L.b) L = rgb(0.0f);
            else if (y < -1.0e-5f) L = rgb(0.0f);
            else if (isinf(y)) L = rgb(0.0f);
            film_add_sample_lane(R, R.pfilm[j], L);
            have = false;
        }
    }
    atomicAdd(&R.cnt->camera_rays, n_camera); atomicAdd(&R.cnt->closest_rays, n_closest);
    atomicAdd(&R.cnt->zero_radiance, n_zero); atomicMax(&R.cnt->iterations, n_iter);
}

void launch_zt_mega(const RenderDev& R, const RenderDev* rdev, uint32_t lanes, uint32_t nblk, cudaStream_t stream) {
    k_zt_mega<true><<<nblk, 32 * PB_ZT_WARPS, 0, stream>>>(R, rdev, lanes);
}
// grids != nullptr: the scene has grid media, and k_vol_mega_grid runs whatever else the scene has
void launch_vol_mega(const RenderDev& R, const RenderDev* rdev, unsigned long long total_items, int camera_medium, bool full, const DevGrid* grids, int grid,
                     cudaStream_t stream) {
    if (grids) k_vol_mega_grid<<<grid, PB_VOL_BLOCK, 0, stream>>>(R, rdev, total_items, camera_medium, grids);
    else if (full) k_vol_mega<true><<<grid, PB_VOL_BLOCK, 0, stream>>>(R, rdev, total_items, camera_medium);
    else k_vol_mega<false><<<grid, PB_VOL_BLOCK, 0, stream>>>(R, rdev, total_items, camera_medium);
}
int vol_mega_blocks_per_sm(bool full, bool grids) {
    int per_sm = 1;
    if (grids) cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_vol_mega_grid, PB_VOL_BLOCK, 0);
    else if (full) cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_vol_mega<true>, PB_VOL_BLOCK, 0);
    else cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_vol_mega<false>, PB_VOL_BLOCK, 0);
    return per_sm;
}
}  // namespace pb
