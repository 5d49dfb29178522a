/*
 * tests/light_oracle.c — TEST INFRASTRUCTURE: the light sampling of RTNW_F_LIGHT_SAMPLING (include/rtnw.h) restated on the CPU on
 * top of the C restatement of the reference (oracle/rtnw_oracle.c, included whole so that its camera ray, world->hit, scatter,
 * textures and sample stream are the very functions the other parity tests pin).  It follows csrc/rtnw_device.cuh
 * (light_pdf, sample_light, mixture_scatter) draw for draw and operation for operation.  The light table is the library's own
 * (rtnw_scene_inspect table 4, 8 floats per light), passed in by the caller.  tests/test_light_sampling.py compiles it with the
 * oracle's flags (gcc -std=gnu11 -O2 -ffp-contract=off, glibc libm) into a temporary directory.
 */
#include "rtnw_oracle.c"

static int light_kind(const float* l) { int k; memcpy(&k, &l[6], 4); return k; }
static vec3 cross(vec3 a, vec3 b) {
    return V(a.e[1] * b.e[2] - a.e[2] * b.e[1], a.e[2] * b.e[0] - a.e[0] * b.e[2], a.e[0] * b.e[1] - a.e[1] * b.e[0]);
}

/* p_k(e): solid-angle density with which light k samples the unit direction e from p; 0 where the ray (p, e) misses it */
static float rect_pdf(int n, int a, int b, const float* l, vec3 p, vec3 e) {
    const float t = (l[4] - p.e[n]) / e.e[n];
    if (!(t > 0.f)) return 0.f;
    const float x = p.e[a] + t * e.e[a], y = p.e[b] + t * e.e[b];
    if (x < l[0] || x > l[1] || y < l[2] || y > l[3]) return 0.f;
    return t * t / (fabsf(e.e[n]) * l[5]);
}
static float pdf_of(const float* l, vec3 p, vec3 e) {
    switch (light_kind(l)) {
        case RTNW_PRIM_RECT_XY: return rect_pdf(2, 0, 1, l, p, e);
        case RTNW_PRIM_RECT_XZ: return rect_pdf(1, 0, 2, l, p, e);
        case RTNW_PRIM_RECT_YZ: return rect_pdf(0, 1, 2, l, p, e);
        default: {
            const vec3 oc = vsub(V(l[0], l[1], l[2]), p);
            const float d2 = dot(oc, oc), r2 = l[3] * l[3];
            if (!(d2 > r2)) return 0.f;
            const float cmax = sqrtf(1.f - r2 / d2);
            if (!(dot(e, unit_vector(oc)) >= cmax)) return 0.f;
            return 1.f / (6.28318531f * (1.f - cmax));
        }
    }
}
/* a unit direction towards light l from p for the draws (u1, u2); 0 when p is inside or on a sphere light */
static int sample_of(const float* l, vec3 p, float u1, float u2, vec3* d) {
    const int kind = light_kind(l);
    if (kind != RTNW_PRIM_SPHERE) {
        const float a = l[0] + u1 * (l[1] - l[0]), b = l[2] + u2 * (l[3] - l[2]);
        const vec3 q = kind == RTNW_PRIM_RECT_XY ? V(a, b, l[4]) : (kind == RTNW_PRIM_RECT_XZ ? V(a, l[4], b) : V(l[4], a, b));
        *d = unit_vector(vsub(q, p));
        return 1;
    }
    const vec3 oc = vsub(V(l[0], l[1], l[2]), p);
    const float d2 = dot(oc, oc), r2 = l[3] * l[3];
    if (!(d2 > r2)) return 0;
    const float cmax = sqrtf(1.f - r2 / d2);
    const float z = 1.f + u2 * (cmax - 1.f), phi = 6.28318531f * u1, s = sqrtf(1.f - z * z);
    const vec3 w = unit_vector(oc);
    const vec3 v = unit_vector(cross(w, fabsf(w.e[0]) > 0.9f ? V(0.f, 1.f, 0.f) : V(1.f, 0.f, 0.f)));
    const vec3 u = cross(w, v);
    *d = vadd(vadd(smul(cosf(phi) * s, u), smul(sinf(phi) * s, v)), smul(z, w));
    return 1;
}

typedef struct { const float* t; int n; } light_table;

/* material::scatter with the one-sample mixture of the light table and the reference's density (include/rtnw.h) */
static int mixture_scatter(const ctx* c, light_table L, int mat, const ray* r_in, const hit_record* rec, vec3* attenuation, ray* scattered) {
    const rtnw_material* m = &c->d->materials[mat];
    const int mix = m->kind == RTNW_MAT_LAMBERTIAN || m->kind == RTNW_MAT_ISOTROPIC;
    const float u = mix ? (float)draw(c->g) : 1.f;
    if (u < 0.5f) { /* light branch */
        int k = (int)(2.f * u * (float)L.n);
        if (k > L.n - 1) k = L.n - 1;
        const float u1 = (float)draw(c->g), u2 = (float)draw(c->g);
        vec3 d;
        if (!sample_of(L.t + 8 * k, rec->p, u1, u2, &d)) return 0;
        scattered->A = rec->p; scattered->B = d; scattered->time = m->kind == RTNW_MAT_LAMBERTIAN ? r_in->time : 0.f;
        *attenuation = texture_value(c->d, m->tex, rec->u, rec->v, rec->p);
    } else if (!material_scatter(c, mat, r_in, rec, attenuation, scattered)) {
        return 0;
    }
    if (!mix) return 1;
    const vec3 e = unit_vector(scattered->B);
    float p_ref = 0.0795774715f;
    if (m->kind == RTNW_MAT_LAMBERTIAN) {
        const float cs = dot(e, rec->normal);
        if (!(cs > 0.f)) return 0;
        p_ref = cs * cs * cs * 0.636619772f;
    }
    float sum = 0.f;
    for (int k = 0; k < L.n; ++k) sum += pdf_of(L.t + 8 * k, rec->p, e);
    const float w = p_ref / (0.5f * p_ref + 0.5f * (sum / (float)L.n));
    *attenuation = smul(w, *attenuation);
    return 1;
}

/* color(), PSC/main.cpp:25-46, as in oracle/rtnw_oracle.c with the mixture scatter when L.n > 0 */
static vec3 light_color(const ctx* c, light_table L, const ray* r, int depth, const rtnw_render_params* P) {
    hit_record rec;
    if (world_hit(c, r, P->t_min, P->t_max, &rec)) {
        ray scattered;
        vec3 attenuation;
        const int emit = (P->flags & RTNW_F_EMIT) != 0;
        vec3 emitted = emit ? material_emitted(c->d, rec.mat, rec.u, rec.v, rec.p) : V(0, 0, 0);
        if (depth < P->max_depth && (L.n > 0 ? mixture_scatter(c, L, rec.mat, r, &rec, &attenuation, &scattered)
                                             : material_scatter(c, rec.mat, r, &rec, &attenuation, &scattered))) {
            vec3 rest = light_color(c, L, &scattered, depth + 1, P);
            if (emit) return vadd(emitted, vmul(attenuation, rest));
            return vmul(attenuation, rest);
        }
        return emitted;
    }
    if (P->background == RTNW_BG_SKY) {
        vec3 unit_direction = unit_vector(r->B);
        float t = 0.5 * (unit_direction.e[1] + 1.0);
        return vadd(smul(1.0 - t, V(1.0, 1.0, 1.0)), smul(t, V(0.5, 0.7, 1.0)));
    }
    return V(0, 0, 0);
}

/* rtnw_oracle_render with RTNW_F_LIGHT_SAMPLING honoured as rtnw_render honours it: the mixture when the flag and RTNW_F_EMIT are
 * set and the table (n_lights lights of 8 floats) is not empty.  Whole images; sample_begin / sample_stride / ROTATE as there. */
int light_oracle_render(const rtnw_scene_desc* d, const float* lights, int n_lights, const rtnw_camera* cam,
                        const rtnw_render_params* P, float* accum) {
    stream g;
    stream_init(&g, P->seed);
    ctx c = {d, &g};
    light_table L = {lights, ((P->flags & RTNW_F_LIGHT_SAMPLING) && (P->flags & RTNW_F_EMIT)) ? n_lights : 0};
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
                vec3 temp = light_color(&c, L, &r, 0, P);
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

/* light k's p_k for n unit directions dirs (n x 3) from the point p */
void light_pdf(const float* lights, int k, const float* p, const float* dirs, size_t n, float* out) {
    for (size_t i = 0; i < n; ++i) out[i] = pdf_of(lights + 8 * k, V(p[0], p[1], p[2]), V(dirs[3 * i], dirs[3 * i + 1], dirs[3 * i + 2]));
}

/* light k's sampled directions from p for n draw pairs u (n x 2, first draw first); ok[i] = 0 where it cannot be sampled */
void sample_light(const float* lights, int k, const float* p, const float* u, size_t n, float* dirs, int32_t* ok) {
    for (size_t i = 0; i < n; ++i) {
        vec3 d = V(0, 0, 0);
        ok[i] = sample_of(lights + 8 * k, V(p[0], p[1], p[2]), u[2 * i], u[2 * i + 1], &d);
        for (int q = 0; q < 3; ++q) dirs[3 * i + q] = d.e[q];
    }
}
