/*
 * tests/denoise_oracle.c — TEST INFRASTRUCTURE: the feature-guided denoiser of rtnw_denoise (include/rtnw.h) restated in plain C
 * from its definition: spatial-only SVGF, i.e. the edge-avoiding a-trous filter of Dammertz et al. 2010 with the
 * variance-guided luminance weight of Schied et al. 2017 and a spatial variance estimate in place of the temporal one.
 * Every step is float32 with + - * /, sqrtf, fabsf and floorf in one fixed order, so the kernels must match it bit for bit.
 * tests/test_denoise.py and tests/test_denoise_cpu.py compile it with the oracle's flags (gcc -std=gnu11 -O2
 * -ffp-contract=off) into a temporary directory.
 */
#include <math.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

#include "rtnw.h"

/* the filter's constants (include/rtnw.h documents them) */
#define DN_EPS_ALBEDO 1e-3f  /* albedo floor of the demodulation */
#define DN_EPS_DEPTH 1e-3f   /* depth tolerance, relative to the centre pixel's depth */
#define DN_EPS_LUM 1e-4f     /* luminance tolerance where the variance is 0 */
#define DN_LUM_R 0.2126f     /* Rec. 709 luminance of the irradiance */
#define DN_LUM_G 0.7152f
#define DN_LUM_B 0.0722f

/* exp(-x) for x >= 0: 2^-y with y = x*log2(e) = n + f, n integer, f in [0, 1); 2^-f by a Horner polynomial whose constant
 * term is exactly 1, 2^-n from the exponent bits.  0 for x >= 88 (below the smallest float), +inf and NaN. */
float rtnw_dn_exp_neg(float x) {
    if (!(x < 88.f)) return 0.f;
    const float y = x * 1.44269502f;
    const float n = floorf(y);
    const float f = y - n;
    const float p = 1.f + f * (-6.93147063e-01f + f * (2.40224302e-01f + f * (-5.54905124e-02f + f * (9.57873557e-03f +
                    f * (-1.27437152e-03f + f * 1.08902554e-04f)))));
    const uint32_t bits = (uint32_t)(127 - (int)n) << 23;
    float two_n;
    memcpy(&two_n, &bits, 4);
    return p * two_n;
}

void rtnw_oracle_exp_neg(const float* x, size_t n, float* out) {
    for (size_t i = 0; i < n; i++) out[i] = rtnw_dn_exp_neg(x[i]);
}

typedef struct {
    int nx, ny, k;  /* image size, normal_power_log2 */
    float sigma_z;
    const int* hit;
    const float* n;     /* normalised normal, 3 per pixel */
    const float* z;     /* depth */
    const float* gx;    /* |dz/dx|, |dz/dy| */
    const float* gy;
} feats;

static float lum(const float* e) { return DN_LUM_R * e[0] + DN_LUM_G * e[1] + DN_LUM_B * e[2]; }

/* max(0, n_p . n_q)^(2^k) */
static float normal_weight(const feats* F, int p, int q) {
    const float* a = F->n + 3 * p;
    const float* b = F->n + 3 * q;
    const float d = a[0] * b[0] + a[1] * b[1] + a[2] * b[2];
    float w = d > 0.f ? d : 0.f;
    for (int s = 0; s < F->k; s++) w = w * w;
    return w;
}

/* |z_p - z_q| / (sigma_z * |grad z_p . (dx, dy)| + eps * z_p), the gradient's components taken as absolute values */
static float depth_distance(const feats* F, int p, int q, int dx, int dy) {
    const float ox = (float)abs(dx), oy = (float)abs(dy);
    return fabsf(F->z[p] - F->z[q]) / (F->sigma_z * (F->gx[p] * ox + F->gy[p] * oy) + DN_EPS_DEPTH * F->z[p]);
}

int rtnw_oracle_denoise(const float* color_sums, const rtnw_aov* aov, int32_t nx, int32_t ny, int32_t ns,
                        const rtnw_denoise_params* dp, float* rgb_out) {
    const int np = nx * ny;
    const float fns = (float)ns;
    int* hit = malloc(sizeof(int) * np);
    float* nrm = malloc(sizeof(float) * 3 * np);
    float* z = malloc(sizeof(float) * np);
    float* gx = malloc(sizeof(float) * np);
    float* gy = malloc(sizeof(float) * np);
    float* alb = malloc(sizeof(float) * 3 * np);  /* a' = max(albedo mean, eps) */
    float* e = malloc(sizeof(float) * 3 * np);    /* irradiance, current pass */
    float* var = malloc(sizeof(float) * np);
    float* e2 = malloc(sizeof(float) * 3 * np);
    float* var2 = malloc(sizeof(float) * np);
    if (!hit || !nrm || !z || !gx || !gy || !alb || !e || !var || !e2 || !var2) return -1;

    /* per-pixel inputs and demodulation */
    for (int p = 0; p < np; p++) {
        hit[p] = aov->hits[p] > 0;
        for (int c = 0; c < 3; c++) {
            const float a = aov->albedo[3 * p + c] / fns;
            alb[3 * p + c] = a > DN_EPS_ALBEDO ? a : DN_EPS_ALBEDO;
            e[3 * p + c] = (color_sums[3 * p + c] / fns) / alb[3 * p + c];
        }
        nrm[3 * p] = nrm[3 * p + 1] = nrm[3 * p + 2] = 0.f;
        z[p] = 0.f;
        if (hit[p]) {
            const float h = (float)aov->hits[p];
            const float x = aov->normal[3 * p] / h, y = aov->normal[3 * p + 1] / h, w = aov->normal[3 * p + 2] / h;
            const float len = sqrtf(x * x + y * y + w * w);
            if (len > 0.f) {
                nrm[3 * p] = x / len; nrm[3 * p + 1] = y / len; nrm[3 * p + 2] = w / len;
            }
            z[p] = aov->depth[p] / h;
        }
    }
    /* depth gradient: central differences over hit neighbours, one-sided next to a miss or the border, else 0 */
    for (int j = 0; j < ny; j++) {
        for (int i = 0; i < nx; i++) {
            const int p = j * nx + i;
            gx[p] = gy[p] = 0.f;
            if (!hit[p]) continue;
            for (int axis = 0; axis < 2; axis++) {
                const int lo_ok = axis == 0 ? i > 0 : j > 0, hi_ok = axis == 0 ? i < nx - 1 : j < ny - 1;
                const int lo = axis == 0 ? p - 1 : p - nx, hi = axis == 0 ? p + 1 : p + nx;
                const int l = lo_ok && hit[lo], h = hi_ok && hit[hi];
                float g = 0.f;
                if (l && h) g = fabsf(z[hi] - z[lo]) * 0.5f;
                else if (h) g = fabsf(z[hi] - z[p]);
                else if (l) g = fabsf(z[p] - z[lo]);
                if (axis == 0) gx[p] = g; else gy[p] = g;
            }
        }
    }
    const feats F = {nx, ny, dp->normal_power_log2, dp->sigma_depth, hit, nrm, z, gx, gy};

    /* variance of the luminance over 7x7, weights w_n * exp(-d_z), the centre exactly 1 */
    for (int j = 0; j < ny; j++) {
        for (int i = 0; i < nx; i++) {
            const int p = j * nx + i;
            float sw = 0.f, s1 = 0.f, s2 = 0.f;
            for (int dy = -3; dy <= 3; dy++) {
                for (int dx = -3; dx <= 3; dx++) {
                    const int qi = i + dx, qj = j + dy;
                    if (qi < 0 || qi >= nx || qj < 0 || qj >= ny) continue;
                    const int q = qj * nx + qi;
                    if (hit[q] != hit[p]) continue;
                    float w = 1.f;
                    if (q != p && hit[p]) w = normal_weight(&F, p, q) * rtnw_dn_exp_neg(depth_distance(&F, p, q, dx, dy));
                    const float l = lum(e + 3 * q);
                    sw = sw + w;
                    s1 = s1 + w * l;
                    s2 = s2 + w * l * l;
                }
            }
            const float m1 = s1 / sw, m2 = s2 / sw;
            const float v = m2 - m1 * m1;
            var[p] = v > 0.f ? v : 0.f;
        }
    }

    static const float H[5] = {1.f / 16.f, 1.f / 4.f, 3.f / 8.f, 1.f / 4.f, 1.f / 16.f};
    for (int it = 0; it < dp->iterations; it++) {
        const int step = 1 << it;
        for (int j = 0; j < ny; j++) {
            for (int i = 0; i < nx; i++) {
                const int p = j * nx + i;
                /* 3x3 binomial blur of the variance over the neighbours p may mix with: same hit class, weights w_n for hits */
                float gs = 0.f, gw = 0.f;
                for (int dy = -1; dy <= 1; dy++) {
                    for (int dx = -1; dx <= 1; dx++) {
                        const int qi = i + dx, qj = j + dy;
                        if (qi < 0 || qi >= nx || qj < 0 || qj >= ny) continue;
                        const int q = qj * nx + qi;
                        if (hit[q] != hit[p]) continue;
                        float w = (float)((2 - abs(dx)) * (2 - abs(dy)));
                        if (q != p && hit[p]) w = w * normal_weight(&F, p, q);
                        gs = gs + w * var[q];
                        gw = gw + w;
                    }
                }
                const float lp = lum(e + 3 * p);
                const float dl_den = dp->sigma_luminance * sqrtf(gs / gw) + DN_EPS_LUM;
                float sw = 0.f, sv = 0.f, s[3] = {0.f, 0.f, 0.f};
                for (int b = -2; b <= 2; b++) {
                    for (int a = -2; a <= 2; a++) {
                        const int dx = a * step, dy = b * step;
                        const int qi = i + dx, qj = j + dy;
                        if (qi < 0 || qi >= nx || qj < 0 || qj >= ny) continue;
                        const int q = qj * nx + qi;
                        if (hit[q] != hit[p]) continue;
                        float w;
                        if (q == p) {
                            w = H[2] * H[2];
                        } else {
                            const float dl = fabsf(lp - lum(e + 3 * q)) / dl_den;
                            if (hit[p]) {
                                const float dz = depth_distance(&F, p, q, dx, dy);
                                w = H[a + 2] * H[b + 2] * normal_weight(&F, p, q) * rtnw_dn_exp_neg(dz + dl);
                            } else {
                                w = H[a + 2] * H[b + 2] * rtnw_dn_exp_neg(dl);
                            }
                        }
                        sw = sw + w;
                        for (int c = 0; c < 3; c++) s[c] = s[c] + w * e[3 * q + c];
                        sv = sv + w * w * var[q];
                    }
                }
                for (int c = 0; c < 3; c++) e2[3 * p + c] = s[c] / sw;
                var2[p] = sv / (sw * sw);
            }
        }
        float* t = e; e = e2; e2 = t;
        t = var; var = var2; var2 = t;
    }
    for (int p = 0; p < 3 * np; p++) rgb_out[p] = e[p] * alb[p];  /* remodulation */
    free(hit); free(nrm); free(z); free(gx); free(gy); free(alb); free(e); free(var); free(e2); free(var2);
    return 0;
}
