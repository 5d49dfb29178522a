/*
 * tests/aov_oracle.c — TEST INFRASTRUCTURE: the first-hit feature buffers of rtnw_render_aov (include/rtnw.h), restated on the
 * CPU on top of the C restatement of the reference (oracle/rtnw_oracle.c, included whole so that its camera ray, world->hit,
 * textures and sample stream are the very functions the other parity tests pin).  tests/test_aov.py compiles it with the
 * oracle's flags (gcc -std=gnu11 -O2 -ffp-contract=off, glibc libm) into a temporary directory.
 */
#include "rtnw_oracle.c"

/* First-hit feature buffers (include/rtnw.h: rtnw_render_aov): per pixel and sample, the first ray of the render path
 * (begin_path, camera_ray), one world->hit at depth 0, and per-pixel sums in sample order.  Buffers as rtnw_render_aov's. */
int rtnw_oracle_aov(const rtnw_scene_desc* d, const rtnw_camera* cam, const rtnw_render_params* P, float* albedo, float* normal,
                    float* depth, int32_t* hits, int32_t* prim_id) {
    stream g;
    stream_init(&g, P->seed);
    ctx c = {d, &g};
    for (int j = P->ny - 1; j >= 0; j--) {
        for (int i = 0; i < P->nx; i++) {
            const size_t q = (size_t)j * P->nx + i;
            vec3 alb = V(0, 0, 0), nrm = V(0, 0, 0);
            float dep = 0;
            int n = 0, id = -1;
            for (int k = 0; k < P->sample_count; k++) {
                const int s = P->sample_begin + k * P->sample_stride;
                begin_path(&g, (uint32_t)q, (uint32_t)s);
                const ray r = camera_ray(cam, P->nx, P->ny, i, j, &g);
                hit_record rec;
                if (world_hit(&c, &r, P->t_min, P->t_max, &rec)) {
                    const rtnw_material* m = &d->materials[rec.mat];
                    vec3 a;
                    switch (m->kind) {
                        case RTNW_MAT_METAL: a = V(m->albedo[0], m->albedo[1], m->albedo[2]); break;
                        case RTNW_MAT_DIELECTRIC: a = V(1, 1, 1); break;
                        case RTNW_MAT_DIFFUSE_LIGHT:
                            a = texture_value(d, m->tex, rec.u, rec.v, rec.p);
                            a = V(fminf(a.e[0], 1.f), fminf(a.e[1], 1.f), fminf(a.e[2], 1.f));
                            break;
                        default: a = texture_value(d, m->tex, rec.u, rec.v, rec.p); break; /* lambertian, isotropic */
                    }
                    alb = vadd(alb, a);
                    nrm = vadd(nrm, rec.normal);
                    dep += rec.t * length(r.B);
                    n++;
                    if (k == 0) id = d->prim_ids ? d->prim_ids[rec.leaf] : rec.leaf;
                } else if (P->background == RTNW_BG_SKY) { /* color()'s miss, TNW/Chapter01_Motion Blur.cpp:29-31 */
                    vec3 unit_direction = unit_vector(r.B);
                    float t = 0.5 * (unit_direction.e[1] + 1.0);
                    alb = vadd(alb, vadd(smul(1.0 - t, V(1.0, 1.0, 1.0)), smul(t, V(0.5, 0.7, 1.0))));
                }
            }
            for (int e = 0; e < 3; ++e) { albedo[3 * q + e] = alb.e[e]; normal[3 * q + e] = nrm.e[e]; }
            depth[q] = dep;
            hits[q] = n;
            prim_id[q] = id;
        }
    }
    return RTNW_OK;
}
