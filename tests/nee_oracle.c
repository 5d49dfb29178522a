/*
 * tests/nee_oracle.c — TEST INFRASTRUCTURE: the next-event estimation of RTNW_F_NEXT_EVENT (include/rtnw.h) restated on the CPU
 * on top of tests/light_oracle.c (its light densities and light samples, pdf_of / sample_of) and oracle/rtnw_oracle.c (camera ray,
 * world->hit, scatter, textures, sample stream).  It follows k_render<.., RENDER_NEE> (csrc/rtnw_cuda.cu) operation for
 * operation, in the recursive form of the oracle's color().  The light table is the library's own (rtnw_scene_inspect table 4,
 * 8 floats per light), and light_leaf[k] is the leaf id of light k's record (table 1), which is what the oracle's hit records
 * carry.  tests/test_next_event.py compiles it with the oracle's flags plus -fwrapv (the shadow query's depth word passes
 * INT_MAX in the stream's int depth) into a temporary directory.
 */
#include "light_oracle.c"

typedef struct { light_table t; const int32_t* leaf; } nee_lights;

/* p_ref(e) of a lambertian (normal n) or isotropic vertex */
static float ref_density(int lambertian, vec3 n, vec3 e) {
    if (!lambertian) return 0.0795774715f;
    const float c = dot(e, n);
    return c > 0.f ? c * c * c * 0.636619772f : 0.f;
}
/* p_L(e) */
static float lights_density(nee_lights N, vec3 p, vec3 e) {
    float sum = 0.f;
    for (int k = 0; k < N.t.n; ++k) sum += pdf_of(N.t.t + 8 * k, p, e);
    return sum / (float)N.t.n;
}
static int is_light_leaf(nee_lights N, int leaf) {
    for (int k = 0; k < N.t.n; ++k)
        if (N.leaf[k] == leaf) return 1;
    return 0;
}

/* color() with next-event estimation: r is the path's ray of depth `depth` and throughput T; w_b weighs an emission of the light
 * table that r finds.  The path's terms are added to *acc in the order of its rays; *shadows counts the shadow queries. */
static void nee_color(const ctx* c, nee_lights N, const ray* r, int depth, vec3 T, float w_b, const rtnw_render_params* P,
                      vec3* acc, uint64_t* shadows) {
    hit_record rec;
    if (world_hit(c, r, P->t_min, P->t_max, &rec)) {
        const rtnw_material* m = &c->d->materials[rec.mat];
        if (m->kind == RTNW_MAT_DIFFUSE_LIGHT) {
            const float w = is_light_leaf(N, rec.leaf) ? w_b : 1.f;
            *acc = vadd(*acc, smul(w, vmul(T, material_emitted(c->d, rec.mat, rec.u, rec.v, rec.p))));
            return;
        }
        ray scattered;
        vec3 attenuation;
        if (depth < P->max_depth && material_scatter(c, rec.mat, r, &rec, &attenuation, &scattered)) {
            const vec3 T1 = vmul(T, attenuation);
            float w1 = 1.f;
            if (m->kind == RTNW_MAT_LAMBERTIAN || m->kind == RTNW_MAT_ISOTROPIC) {
                const int lam = m->kind == RTNW_MAT_LAMBERTIAN;
                const vec3 e1 = unit_vector(scattered.B);
                const float pr1 = ref_density(lam, rec.normal, e1), pl1 = lights_density(N, rec.p, e1);
                if (pl1 > 0.f) w1 = pr1 / (pr1 + pl1);
                const uint32_t ctr[4] = {0xffffffffu, 1u + (uint32_t)depth, c->g->sample, c->g->pixel};
                uint32_t u[4];
                philox4x32_10(ctr, c->g->key, u);
                int k = (int)((float)u01(u[0]) * (float)N.t.n);
                if (k > N.t.n - 1) k = N.t.n - 1;
                vec3 e;
                if (sample_of(N.t.t + 8 * k, rec.p, (float)u01(u[1]), (float)u01(u[2]), &e)) {
                    const float pr = ref_density(lam, rec.normal, e);
                    if (pr > 0.f) {
                        const float W = pr / (pr + lights_density(N, rec.p, e));
                        ray sr;
                        sr.A = rec.p; sr.B = e; sr.time = scattered.time;
                        const int saved = c->g->depth;
                        c->g->depth = (int)(0x80000000u + (uint32_t)depth - 2u);  /* world_hit's ++: medium key word 1 + depth = 0x80000000 | d */
                        hit_record sh;
                        if (world_hit(c, &sr, P->t_min, P->t_max, &sh) && is_light_leaf(N, sh.leaf))
                            *acc = vadd(*acc, smul(W, vmul(T1, material_emitted(c->d, sh.mat, sh.u, sh.v, sh.p))));
                        c->g->depth = saved;
                        ++*shadows;
                    }
                }
            }
            nee_color(c, N, &scattered, depth + 1, T1, w1, P, acc, shadows);
        }
        return;
    }
    if (P->background == RTNW_BG_SKY) {
        vec3 unit_direction = unit_vector(r->B);
        float t = 0.5 * (unit_direction.e[1] + 1.0);
        *acc = vadd(*acc, vmul(T, vadd(smul(1.0 - t, V(1.0, 1.0, 1.0)), smul(t, V(0.5, 0.7, 1.0)))));
    }
}

/* rtnw_oracle_render with RTNW_F_NEXT_EVENT honoured as rtnw_render honours it: next-event estimation when the flag and RTNW_F_EMIT
 * are set and the table (n_lights lights of 8 floats, light_leaf[k] = leaf id of light k) is not empty, else the oracle's own
 * color().  Whole images; sample_begin / sample_stride / ROTATE as there.  *shadow_queries = the shadow rays traced. */
int nee_oracle_render(const rtnw_scene_desc* d, const float* lights, const int32_t* light_leaf, int n_lights, const rtnw_camera* cam,
                      const rtnw_render_params* P, float* accum, uint64_t* shadow_queries) {
    stream g;
    stream_init(&g, P->seed);
    ctx c = {d, &g};
    nee_lights N = {{lights, n_lights}, light_leaf};
    const int nee = (P->flags & RTNW_F_NEXT_EVENT) && (P->flags & RTNW_F_EMIT) && n_lights > 0;
    *shadow_queries = 0;
    for (int j = P->ny - 1; j >= 0; j--) {
        for (int i = 0; i < P->nx; i++) {
            vec3 col = V(0, 0, 0);
            int s_begin = P->sample_begin, s_count = P->sample_count;
            if (P->flags & RTNW_F_ROTATE_SAMPLES) {
                const int g_ = P->sample_stride, pix = j * P->nx + i;
                s_begin = ((P->sample_begin - pix) % g_ + g_) % g_;
                s_count = s_begin < P->sample_count ? (P->sample_count - s_begin + g_ - 1) / g_ : 0;
            }
            for (int k = 0; k < s_count; k++) {
                const int s = s_begin + k * P->sample_stride;
                begin_path(&g, (uint32_t)(j * P->nx + i), (uint32_t)s);
                ray r = camera_ray(cam, P->nx, P->ny, i, j, &g);
                vec3 temp = V(0, 0, 0);
                if (nee) nee_color(&c, N, &r, 0, V(1, 1, 1), 1.f, P, &temp, shadow_queries);
                else temp = color(&c, &r, 0, P);
                if (P->flags & RTNW_F_DE_NAN)
                    for (int q = 0; q < 3; ++q)
                        if (!(temp.e[q] == temp.e[q])) temp.e[q] = 0;
                col = vadd(col, temp);
            }
            for (int q = 0; q < 3; ++q) accum[3 * ((size_t)j * P->nx + i) + q] = col.e[q];
        }
    }
    return RTNW_OK;
}
