// rtnw_cuda.cu — librtnw.so: sm_100a kernels + the C-ABI of include/rtnw.h.
//
// Replaces the sample loop of the reference (PSC/main.cpp:299-313) and everything it calls.  There is no CPU
// implementation in this library: every compute entry point needs a CUDA device.
#include <cuda_runtime.h>

#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <type_traits>
#include <vector>

#include "rtnw.h"
#include "rtnw_device.cuh"

using namespace rtnw_dev;

#ifndef RTNW_MIN_BLOCKS
#define RTNW_MIN_BLOCKS 2   // resident blocks per SM the register allocation is sized for (block size: RTNW_BLOCK, rtnw_device.cuh)
#endif

#define RTNW_MAX_CHUNKS 64
#define RTNW_MAX_DEVICES 16

// ================================================================================================ kernels
struct render_args {
    scene_view S;
    rtnw_camera cam;
    rtnw_render_params p;
    float* accum;                 // nx*ny*3 sums, index (j*nx+i)*3+c
    unsigned long long* fixed;    // chunks > 1: nx*ny*3 fixed-point sums (add_fixed / k_finish_fixed), all zero between renders
    int chunks;                   // each pixel's samples are cut into this many contiguous ranges, one work item each
    int chunk_total;              // range c of a pixel with n samples: k in [cum[c]*n/total, cum[c+1]*n/total)
    int chunk_cum[RTNW_MAX_CHUNKS + 1];
    unsigned long long* ctr;      // [0] next pixel, [1] rays, [2] box tests, [3] primitive tests, [4] task stack overflows
};

// Partial sums of the sample ranges of a pixel are added in 64-bit fixed point with integer atomics: integer addition
// commutes, so the pixel's sum is the same bits whatever order the ranges finish in, with ONE plane of scratch instead of
// one float plane per range.  Value = round(v * 2^41), always even; bit 0 is a sticky "not a number" flag (a NaN or infinite
// partial sum — only possible without RTNW_F_DE_NAN — makes the pixel NaN, as `col += temp` does in the reference).
// Resolution 4.5e-13, range +-2^22 (larger partial sums saturate; radiance sums are < 1e5).
__device__ __forceinline__ void add_fixed(unsigned long long* dst, float v) {
    if (v - v == 0.f) {  // finite
        const float c = fminf(fmaxf(v, -4194303.f), 4194303.f);
        const long long q = __double2ll_rn((double)c * 1099511627776.0) << 1;  // 2^40, then << 1
        if (q != 0) atomicAdd(dst, (unsigned long long)q);
    } else {
        atomicOr(dst, 1ull);
    }
}
__device__ __forceinline__ float from_fixed(unsigned long long u) {
    if (u & 1ull) return __int_as_float(0x7fc00000);
    return (float)((double)(long long)u * (1.0 / 2199023255552.0));  // 2^-41, one rounding
}

// the reference-exact kernels traverse one BVH item at a time; the RTNW_F_FAST_BVH kernels two together (two ray frames)
template <bool FAST> using block_smem = coop_smem<FAST ? 2 : 1>;

// The sample loop of PSC/main.cpp:299-313 as ONE persistent megakernel.
//
// One thread owns one work item at a time — a pixel and a contiguous range of its samples (pick_chunks): the samples
// are traced back to back and summed in sample order like `col += temp` in the reference; the partial sums of a pixel's
// ranges are added in 64-bit fixed point (add_fixed: integer atomics commute, so a pixel's sum never depends on scheduling).  A
// thread that finishes its item pulls the next one from a global counter (warp-aggregated atomic); a thread whose path
// ends starts the next sample of its item in the same round (path regeneration, which absorbs the 51-bounce tail).
//
// The block advances in rounds, one ray per thread per round: regenerate -> closest hit -> shade.  The closest hit is
// block-cooperative (coop_closest_hit): list items in lockstep, BVH items as uniform tasks from shared-memory queues.
// A per-lane traversal state machine was measured at 2-13 active lanes of 32 per instruction (profiles/r1-r3*.txt);
// this form keeps every phase uniform across the warp.
template <bool COUNT, bool FAST>
__global__ void __launch_bounds__(RTNW_BLOCK, RTNW_MIN_BLOCKS) k_render(const render_args P) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    typedef block_smem<FAST> SM;
    SM& sm = *reinterpret_cast<SM*>(smem_raw);
    constexpr unsigned FULL = 0xffffffffu;
    const unsigned lane = threadIdx.x & 31u;
    const int nx = P.p.nx, ny = P.p.ny;
    const unsigned long long npix = (unsigned long long)P.p.pixel_count;  // render_core fills in the default subset
    const bool accumulate = (P.p.flags & RTNW_F_ACCUMULATE) != 0;
    const bool rotate = (P.p.flags & RTNW_F_ROTATE_SAMPLES) != 0;
    const uint32_t k0 = (uint32_t)P.p.seed, k1 = (uint32_t)(P.p.seed >> 32);
    const bool emit = (P.p.flags & RTNW_F_EMIT) != 0;
    const bool denan = (P.p.flags & RTNW_F_DE_NAN) != 0;
    const bool sky = P.p.background == RTNW_BG_SKY;

    coop_init<SM>(sm);
    __syncthreads();
    int r3 = 0;  // index of the cooperative traversal's next round, mod 3 (coop_bvh_item)
#ifdef RTNW_ROUND_STATS
    const long long t_start = clock64();
#endif
    // The work item of a thread (pixel, sample range, running sum) lives in shared memory: it is touched when a path
    // ends, i.e. once every few rounds, and would otherwise occupy eight registers across every round.
    int me = threadIdx.x % RTNW_BLOCK;  // index of this thread's work item in sm.acc / sm.span
    bool alive = true, need = true, has_item = false;
    int depth = 0;
    f3 T = mk3(0.f, 0.f, 0.f);
    ray_t wr;
    wr.o = T; wr.d = mk3(1.f, 1.f, 1.f); wr.time = 0.f;
    rng_t g;
    g.begin(k0, k1, 0, 0);
    unsigned n_rays = 0;  // per thread; summed in 64 bits below
    unsigned long long box_total = 0, prim_total = 0;
    trav_counters cnt;
    cnt.box_tests = 0; cnt.prim_tests = 0;

    for (;;) {
        // ---- next sample of the pixel, or next pixel, PSC/main.cpp:299-308
        if (alive && need && has_item) {
            const float4 acc = sm.acc[me];
            if (__float_as_int(acc.w) == sm.span[me].y) {  // k == end of the range: the item is finished
                const int4 it = sm.span[me];  // z = pixel, w = sample range
                if (P.chunks > 1) {  // partial sum of one sample range
                    unsigned long long* dst = P.fixed + 3ull * (unsigned long long)it.z;
                    add_fixed(dst, acc.x); add_fixed(dst + 1, acc.y); add_fixed(dst + 2, acc.z);
                } else {
                    float* dst = P.accum + 3ull * (unsigned long long)it.z;
                    if (accumulate) { dst[0] += acc.x; dst[1] += acc.y; dst[2] += acc.z; }
                    else { dst[0] = acc.x; dst[1] = acc.y; dst[2] = acc.z; }
                }
                has_item = false;
            }
        }
        const bool want = alive && need && !has_item;
        const unsigned m = __ballot_sync(FULL, want);
        if (m) {
            const int leader = __ffs(m) - 1;
            unsigned long long base = 0;
            if ((int)lane == leader) base = atomicAdd(&P.ctr[0], (unsigned long long)__popc(m));
            base = __shfl_sync(FULL, base, leader);
            if (want) {
                const unsigned long long mine = base + (unsigned long long)__popc(m & ((1u << lane) - 1u));
                if (mine >= npix * (unsigned long long)P.chunks) alive = false;
                else {
                    const int chunk = (int)(mine / npix);  // work item = (sample range, pixel), range-major
                    const int pix = P.p.pixel_begin + (int)(mine % npix) * P.p.pixel_stride;
                    int k = 0, s_begin = P.p.sample_begin, s_count = P.p.sample_count;
                    if (rotate) {  // RTNW_F_ROTATE_SAMPLES: ownership of the samples rotates with the pixel index
                        const int g = P.p.sample_stride;
                        s_begin = ((P.p.sample_begin - pix) % g + g) % g;
                        s_count = s_begin < P.p.sample_count ? (P.p.sample_count - s_begin + g - 1) / g : 0;
                    }
                    if (P.chunks > 1) {  // this item's range of the pixel's samples
                        k = (int)((long long)P.chunk_cum[chunk] * s_count / P.chunk_total);
                        s_count = (int)((long long)P.chunk_cum[chunk + 1] * s_count / P.chunk_total);
                    }
                    sm.acc[me] = make_float4(0.f, 0.f, 0.f, __int_as_float(k));
                    sm.span[me] = make_int4(s_begin, s_count, pix, chunk);
                    has_item = true;
                }
            }
        }
        if (__syncthreads_count(alive) == 0) break;  // the block is done
        if (alive && need && has_item) {
            const int k = __float_as_int(sm.acc[me].w);
            const int4 sp = sm.span[me];
            if (k < sp.y) {
                const int pix = sp.z;
                const int s = sp.x + k * P.p.sample_stride;
                sm.acc[me].w = __int_as_float(k + 1);
                g.begin(k0, k1, (uint32_t)pix, (uint32_t)s);
                camera_ray(P.cam, nx, ny, pix % nx, pix / nx, g, wr);
                depth = 0;
                T = mk3(1.f, 1.f, 1.f);
                need = false;
            }
        }
        // ---- world->hit(r, t_min, t_max, rec), PSC/main.cpp:27
        medium_key mk;
        mk.k0 = k0; mk.k1 = k1; mk.pixel = (uint32_t)sm.span[me].z; mk.sample = g.sample; mk.depth = (uint32_t)depth;
        const bool tracing = alive && !need;  // a pixel that owns no sample of this call has no ray (RTNW_F_ROTATE_SAMPLES, ns < G)
#ifdef RTNW_ROUND_STATS
        const long long c0 = clock64();
#endif
        const hkey_t key = coop_closest_hit<COUNT, FAST, SM>(P.S, sm, wr, tracing, P.p.t_min, P.p.t_max, mk, cnt, r3);
#ifdef RTNW_ROUND_STATS
        if (threadIdx.x == 0) { RTNW_STAT(10, 1); RTNW_STAT(11, clock64() - c0); }
        const long long c1 = clock64();
#endif
        // ---- one level of color(), PSC/main.cpp:25-46, in iterative form (DESIGN.md §5)
        if (tracing) {
            ++n_rays;
            f3 L = mk3(0.f, 0.f, 0.f);  // radiance of this path: only its last ray (a light, or the sky) adds any, so it need not live across rounds
            hit_t h;
            key_to_hit(P.S, key, P.p.t_max, h);
            need = true;
            if (h.rec >= 0) {
                surf_t s;
                // does value(u,v,p) of this hit's texture read u,v?  (only image_texture does, PSC/surface_texture.h:19-30;
                // a checker forwards u,v to its children, so it is treated as if it did)
                const int mat_id = __float_as_int(__ldg(&P.S.recs[h.rec].b).w);
                const float4 m0 = __ldg(reinterpret_cast<const float4*>(P.S.materials + mat_id));
                bool want_uv = false;
                if (__float_as_int(m0.y) >= 0 && __float_as_uint(m0.x) != RTNW_MAT_METAL && __float_as_uint(m0.x) != RTNW_MAT_DIELECTRIC) {
                    const uint32_t tk = __float_as_uint(__ldg(reinterpret_cast<const float4*>(P.S.textures + __float_as_int(m0.y))).x);
                    want_uv = tk == RTNW_TEX_IMAGE || tk == RTNW_TEX_CHECKER;
                }
                finish_hit(P.S, wr, h, s, want_uv);
                if (__float_as_uint(m0.x) == RTNW_MAT_DIFFUSE_LIGHT) {  // the only material that emits; it never scatters
                    if (emit) L = L + T * texture_value(P.S, __float_as_int(m0.y), s.u, s.v, s.p);
                } else if (depth < P.p.max_depth) {
                    ray_t sc;
                    f3 att;
                    if (material_scatter(P.S, s.mat, wr, s, g, att, sc)) {
                        T = T * att;
                        wr = sc;
                        ++depth;
                        need = false;
                    }
                }
            } else if (sky) {
                L = L + T * sky_color(wr.d);
            }
            if (need) {  // the path ended: PSC/main.cpp:311-312
                if (denan) {
                    if (!(L.x == L.x)) L.x = 0.f;
                    if (!(L.y == L.y)) L.y = 0.f;
                    if (!(L.z == L.z)) L.z = 0.f;
                }
                float4 acc = sm.acc[me];  // col += de_nan(color(...)), PSC/main.cpp:311-312
                acc.x += L.x; acc.y += L.y; acc.z += L.z;
                sm.acc[me] = acc;
            }
        }
#ifdef RTNW_ROUND_STATS
        if (threadIdx.x == 0) RTNW_STAT(13, clock64() - c1);
#endif
    }
#ifdef RTNW_ROUND_STATS
    if (threadIdx.x == 0) RTNW_STAT(12, clock64() - t_start);
#endif
    __syncthreads();
    if (threadIdx.x % RTNW_BLOCK == 0 && sm.overflow) atomicAdd(&P.ctr[4], 1ull);
    // work counters: one atomic per warp
    if (COUNT) { box_total = cnt.box_tests; prim_total = cnt.prim_tests; }
    unsigned long long rays_total = n_rays;
    for (int o = 16; o > 0; o >>= 1) rays_total += __shfl_xor_sync(FULL, rays_total, o);
    if (lane == 0) atomicAdd(&P.ctr[1], rays_total);
    if (COUNT) {
        for (int o = 16; o > 0; o >>= 1) {
            box_total += __shfl_xor_sync(FULL, box_total, o);
            prim_total += __shfl_xor_sync(FULL, prim_total, o);
        }
        if (lane == 0) { atomicAdd(&P.ctr[2], box_total); atomicAdd(&P.ctr[3], prim_total); }
    }
}

// one world->hit() per ray, PSC/main.cpp:27 — the same block-cooperative closest hit the renderer uses
template <bool FAST>
__global__ void __launch_bounds__(RTNW_BLOCK) k_trace(const scene_view S, const rtnw_ray* __restrict__ rays, size_t n, float t_min,
                                                      float t_max, uint64_t seed, rtnw_hit* __restrict__ out) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    typedef block_smem<FAST> SM;
    SM& sm = *reinterpret_cast<SM*>(smem_raw);
    const size_t q = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    const bool active = q < n;  // idle threads of the last block still work on the block's BVH tasks
    rtnw_ray in;
    memset(&in, 0, sizeof in);
    in.direction[0] = 1.f;
    if (active) in = rays[q];
    ray_t r;
    r.o = mk3(in.origin[0], in.origin[1], in.origin[2]);
    r.d = mk3(in.direction[0], in.direction[1], in.direction[2]);
    r.time = in.time;
    medium_key mk;
    mk.k0 = (uint32_t)seed; mk.k1 = (uint32_t)(seed >> 32); mk.pixel = in.key; mk.sample = 0; mk.depth = 0;
    trav_counters cnt;
    cnt.box_tests = 0; cnt.prim_tests = 0;
    coop_init<SM>(sm);
    __syncthreads();
    int r3 = 0;
    const hkey_t key = coop_closest_hit<false, FAST, SM>(S, sm, r, active, t_min, t_max, mk, cnt, r3);
    if (!active) return;
    hit_t h;
    key_to_hit(S, key, t_max, h);
    rtnw_hit o;
    memset(&o, 0, sizeof o);
    o.prim_id = -1;
    o.mat_id = -1;
    if (h.rec >= 0) {
        surf_t s;
        finish_hit(S, r, h, s);
        o.prim_id = S.rec_leaf[h.rec];
        o.sub_id = h.face;
        o.t = h.t;
        o.p[0] = s.p.x; o.p[1] = s.p.y; o.p[2] = s.p.z;
        o.normal[0] = s.n.x; o.normal[1] = s.n.y; o.normal[2] = s.n.z;
        o.u = s.u; o.v = s.v;
        o.mat_id = s.mat;
    }
    out[q] = o;
}

struct aov_args {
    scene_view S;
    rtnw_camera cam;
    rtnw_render_params p;
    float* albedo;                // nx*ny*3 sums
    float* normal;                // nx*ny*3 sums
    float* depth;                 // nx*ny sums
    int32_t* hits;                // nx*ny counts
    int32_t* prim_id;             // nx*ny leaf ids of sample k = 0
    unsigned long long* ctr;      // [4] task stack overflows
};

// First-hit feature buffers (rtnw_render_aov): one thread per pixel traces, for each of its samples, exactly the first ray
// k_render traces for that (pixel, sample) — same stream, same camera_ray, same medium key at depth 0 — and sums what the
// hit shows.  Every pixel has sample_count samples, so every thread of the block runs the same number of cooperative rounds.
// The running sums of a pixel live in shared memory, as k_render's work items do: in registers they would be live across
// the media's Philox call inside the traversal, and spill.
template <bool FAST> struct aov_smem {
    block_smem<FAST> coop;
    float4 acc[RTNW_BLOCK];    // albedo xyz, depth
    float4 nrm[RTNW_BLOCK];    // normal xyz, w = hits (int bits)
};

// the first ray of the path (pix, s), as k_render starts it.  Not inlined: inside the sample loop the compiler would hoist the
// pixel's coordinates and the shutter interval out of it, and those values, live across the traversal, would spill.
__device__ __noinline__ ray_t aov_camera_ray(const rtnw_camera& cam, int nx, int ny, int pix, int s, uint64_t seed) {
    rng_t g;
    g.begin((uint32_t)seed, (uint32_t)(seed >> 32), (uint32_t)pix, (uint32_t)s);
    ray_t r;
    camera_ray(cam, nx, ny, pix % nx, pix / nx, g, r);
    return r;
}

template <bool FAST>
__global__ void __launch_bounds__(RTNW_BLOCK) k_aov(const __grid_constant__ aov_args P) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    typedef block_smem<FAST> SM;
    aov_smem<FAST>& A = *reinterpret_cast<aov_smem<FAST>*>(smem_raw);
    SM& sm = A.coop;
    const int me = threadIdx.x;
    const int nx = P.p.nx, ny = P.p.ny;
    const int pix = blockIdx.x * blockDim.x + threadIdx.x;
    const bool active = pix < nx * ny;  // idle threads of the last block still work on the block's BVH tasks (with a ray below the image)
    const uint32_t k0 = (uint32_t)P.p.seed, k1 = (uint32_t)(P.p.seed >> 32);
    trav_counters cnt;
    cnt.box_tests = 0; cnt.prim_tests = 0;
    coop_init<SM>(sm);
    A.acc[me] = make_float4(0.f, 0.f, 0.f, 0.f);
    A.nrm[me] = make_float4(0.f, 0.f, 0.f, __int_as_float(0));
    __syncthreads();
    int r3 = 0;
    for (int k = 0; k < P.p.sample_count; ++k) {
        const int s = P.p.sample_begin + k * P.p.sample_stride;
        const ray_t r = aov_camera_ray(P.cam, nx, ny, pix, s, P.p.seed);
        medium_key mk;
        mk.k0 = k0; mk.k1 = k1; mk.pixel = (uint32_t)pix; mk.sample = (uint32_t)s; mk.depth = 0;
        const hkey_t key = coop_closest_hit<false, FAST, SM>(P.S, sm, r, active, P.p.t_min, P.p.t_max, mk, cnt, r3);
        if (!active) continue;
        hit_t h;
        key_to_hit(P.S, key, P.p.t_max, h);
        if (h.rec < 0) {
            if (k == 0) P.prim_id[pix] = -1;
            if (P.p.background == RTNW_BG_SKY) {
                const f3 c = sky_color(r.d);
                float4 acc = A.acc[me];
                acc.x += c.x; acc.y += c.y; acc.z += c.z;
                A.acc[me] = acc;
            }
            continue;
        }
        if (k == 0) P.prim_id[pix] = __ldg(&P.S.rec_leaf[h.rec]);
        // u,v only when the hit material's texture reads them: the rule of k_render
        const int mat_id = __float_as_int(__ldg(&P.S.recs[h.rec].b).w);
        const float4 m0 = __ldg(reinterpret_cast<const float4*>(P.S.materials + mat_id));
        const uint32_t mkind = __float_as_uint(m0.x);
        bool want_uv = false;
        if (__float_as_int(m0.y) >= 0 && mkind != RTNW_MAT_METAL && mkind != RTNW_MAT_DIELECTRIC) {
            const uint32_t tk = __float_as_uint(__ldg(reinterpret_cast<const float4*>(P.S.textures + __float_as_int(m0.y))).x);
            want_uv = tk == RTNW_TEX_IMAGE || tk == RTNW_TEX_CHECKER;
        }
        surf_t sf;
        finish_hit(P.S, r, h, sf, want_uv);
        f3 a;  // the attenuation scatter() returns; a light's emission clamped to 1
        if (mkind == RTNW_MAT_METAL) {
            const float4 m1 = __ldg(reinterpret_cast<const float4*>(P.S.materials + mat_id) + 1);
            a = mk3(m1.x, m1.y, m1.z);
        } else if (mkind == RTNW_MAT_DIELECTRIC) {
            a = mk3(1.f, 1.f, 1.f);
        } else {
            a = texture_value(P.S, __float_as_int(m0.y), sf.u, sf.v, sf.p);
            if (mkind == RTNW_MAT_DIFFUSE_LIGHT) a = mk3(fminf(a.x, 1.f), fminf(a.y, 1.f), fminf(a.z, 1.f));
        }
        float4 acc = A.acc[me];
        acc.x += a.x; acc.y += a.y; acc.z += a.z;
        acc.w += h.t * length(r.d);
        A.acc[me] = acc;
        float4 nrm = A.nrm[me];
        nrm.x += sf.n.x; nrm.y += sf.n.y; nrm.z += sf.n.z;
        nrm.w = __int_as_float(__float_as_int(nrm.w) + 1);
        A.nrm[me] = nrm;
    }
    __syncthreads();
    if (threadIdx.x % RTNW_BLOCK == 0 && sm.overflow) atomicAdd(&P.ctr[4], 1ull);
    if (!active) return;
    const size_t q = (size_t)pix;
    const float4 acc = A.acc[me], nrm = A.nrm[me];
    P.albedo[3 * q] = acc.x; P.albedo[3 * q + 1] = acc.y; P.albedo[3 * q + 2] = acc.z;
    P.normal[3 * q] = nrm.x; P.normal[3 * q + 1] = nrm.y; P.normal[3 * q + 2] = nrm.z;
    P.depth[q] = acc.w;
    P.hits[q] = __float_as_int(nrm.w);
}

// ---- rtnw_denoise: spatial-only SVGF (include/rtnw.h).  One thread per pixel, 2D blocks.  Every operation is float32 in the
// order of the C restatement tests/denoise_oracle.c (--fmad=false: no contraction), so the two agree bit for bit.
#define DN_EPS_ALBEDO 1e-3f  // albedo floor of the demodulation
#define DN_EPS_DEPTH 1e-3f   // depth tolerance, relative to the centre pixel's depth
#define DN_EPS_LUM 1e-4f     // luminance tolerance where the variance is 0
#define DN_LUM_R 0.2126f     // Rec. 709 luminance of the irradiance
#define DN_LUM_G 0.7152f
#define DN_LUM_B 0.0722f
#define DN_BX 32
#define DN_BY 8

struct dn_args {
    int nx, ny, k;           // image size, normal_power_log2
    float fns, sigma_l, sigma_z;
    const float* color;      // nx*ny*3 sums
    const float* albedo;     // nx*ny*3 sums
    const float* normal;     // nx*ny*3 sums
    const float* depth;      // nx*ny sums
    const int32_t* hits;     // nx*ny
    float4* ev[2];           // irradiance xyz, variance (ping-pong)
    float4* feat;            // normalised normal xyz, depth (0 for misses)
    float2* grad;            // |dz/dx|, |dz/dy|
    unsigned char* hit;      // hits > 0
    float* out;              // nx*ny*3 denoised means (may alias color: only k_dn_prepare reads it)
};

// exp(-x) for x >= 0: 2^-y, y = x*log2(e) = n + f, f in [0, 1): a Horner polynomial for 2^-f (constant term exactly 1) times
// 2^-n from the exponent bits; 0 for x >= 88, +inf and NaN.  Within 1e-5 relative of exp (tests/test_denoise_cpu.py).
__device__ __forceinline__ float dn_exp_neg(float x) {
    if (!(x < 88.f)) return 0.f;
    const float y = x * 1.44269502f;
    const float n = floorf(y);
    const float f = y - n;
    const float p = 1.f + f * (-6.93147063e-01f + f * (2.40224302e-01f + f * (-5.54905124e-02f + f * (9.57873557e-03f +
                    f * (-1.27437152e-03f + f * 1.08902554e-04f)))));
    return p * __uint_as_float((uint32_t)(127 - (int)n) << 23);
}

__device__ __forceinline__ float dn_lum(float4 e) { return DN_LUM_R * e.x + DN_LUM_G * e.y + DN_LUM_B * e.z; }

// max(0, n_p . n_q)^(2^k)
__device__ __forceinline__ float dn_normal_weight(float4 a, float4 b, int k) {
    const float d = a.x * b.x + a.y * b.y + a.z * b.z;
    float w = d > 0.f ? d : 0.f;
    for (int s = 0; s < k; ++s) w = w * w;
    return w;
}

// |z_p - z_q| / (sigma_z * |grad z_p . (dx, dy)| + eps * z_p), the gradient's components taken as absolute values
__device__ __forceinline__ float dn_depth_distance(float zp, float zq, float2 g, float sigma_z, int dx, int dy) {
    const float ox = (float)abs(dx), oy = (float)abs(dy);
    return fabsf(zp - zq) / (sigma_z * (g.x * ox + g.y * oy) + DN_EPS_DEPTH * zp);
}

__device__ __forceinline__ float dn_albedo(const dn_args& P, int p, int c) {
    const float a = __ldg(&P.albedo[3 * p + c]) / P.fns;
    return a > DN_EPS_ALBEDO ? a : DN_EPS_ALBEDO;
}

__device__ __forceinline__ float dn_depth(const dn_args& P, int q) { return __ldg(&P.depth[q]) / (float)__ldg(&P.hits[q]); }

// means, demodulation, normalised normal, hit flag, depth gradient
__global__ void __launch_bounds__(DN_BX * DN_BY) k_dn_prepare(const __grid_constant__ dn_args P) {
    const int i = blockIdx.x * DN_BX + threadIdx.x, j = blockIdx.y * DN_BY + threadIdx.y;
    if (i >= P.nx || j >= P.ny) return;
    const int p = j * P.nx + i;
    const int h = __ldg(&P.hits[p]);
    float4 e;
    e.x = (__ldg(&P.color[3 * p]) / P.fns) / dn_albedo(P, p, 0);
    e.y = (__ldg(&P.color[3 * p + 1]) / P.fns) / dn_albedo(P, p, 1);
    e.z = (__ldg(&P.color[3 * p + 2]) / P.fns) / dn_albedo(P, p, 2);
    e.w = 0.f;
    float4 f = make_float4(0.f, 0.f, 0.f, 0.f);
    float2 g = make_float2(0.f, 0.f);
    if (h > 0) {
        const float fh = (float)h;
        const float x = __ldg(&P.normal[3 * p]) / fh, y = __ldg(&P.normal[3 * p + 1]) / fh, w = __ldg(&P.normal[3 * p + 2]) / fh;
        const float len = sqrtf(x * x + y * y + w * w);
        if (len > 0.f) { f.x = x / len; f.y = y / len; f.z = w / len; }
        f.w = __ldg(&P.depth[p]) / fh;
        for (int axis = 0; axis < 2; ++axis) {
            const bool lo_ok = axis == 0 ? i > 0 : j > 0, hi_ok = axis == 0 ? i < P.nx - 1 : j < P.ny - 1;
            const int lo = axis == 0 ? p - 1 : p - P.nx, hi = axis == 0 ? p + 1 : p + P.nx;
            const bool l = lo_ok && __ldg(&P.hits[lo]) > 0, u = hi_ok && __ldg(&P.hits[hi]) > 0;
            float d = 0.f;
            if (l && u) d = fabsf(dn_depth(P, hi) - dn_depth(P, lo)) * 0.5f;
            else if (u) d = fabsf(dn_depth(P, hi) - f.w);
            else if (l) d = fabsf(f.w - dn_depth(P, lo));
            if (axis == 0) g.x = d; else g.y = d;
        }
    }
    P.ev[0][p] = e;
    P.feat[p] = f;
    P.grad[p] = g;
    P.hit[p] = h > 0;
}

// variance of the luminance over 7x7, weights w_n * exp(-d_z) (1 at the centre); reads ev[0], writes ev[1] = (e, var)
__global__ void __launch_bounds__(DN_BX * DN_BY) k_dn_variance(const __grid_constant__ dn_args P) {
    const int i = blockIdx.x * DN_BX + threadIdx.x, j = blockIdx.y * DN_BY + threadIdx.y;
    if (i >= P.nx || j >= P.ny) return;
    const int p = j * P.nx + i;
    const bool hp = P.hit[p];
    const float4 fp = P.feat[p];
    const float2 gp = P.grad[p];
    float sw = 0.f, s1 = 0.f, s2 = 0.f;
    for (int dy = -3; dy <= 3; ++dy) {
        const int qj = j + dy;
        if (qj < 0 || qj >= P.ny) continue;
        for (int dx = -3; dx <= 3; ++dx) {
            const int qi = i + dx;
            if (qi < 0 || qi >= P.nx) continue;
            const int q = qj * P.nx + qi;
            if ((bool)__ldg(&P.hit[q]) != hp) continue;
            float w = 1.f;
            if (q != p && hp) {
                const float4 fq = __ldg(&P.feat[q]);
                w = dn_normal_weight(fp, fq, P.k) * dn_exp_neg(dn_depth_distance(fp.w, fq.w, gp, P.sigma_z, dx, dy));
            }
            const float l = dn_lum(__ldg(&P.ev[0][q]));
            sw = sw + w;
            s1 = s1 + w * l;
            s2 = s2 + w * l * l;
        }
    }
    const float m1 = s1 / sw, m2 = s2 / sw;
    const float v = m2 - m1 * m1;
    float4 e = P.ev[0][p];
    e.w = v > 0.f ? v : 0.f;
    P.ev[1][p] = e;
}

// one a-trous pass with step 2^it: reads ev[src], writes ev[1 - src]; the last pass remodulates into out instead
__global__ void __launch_bounds__(DN_BX * DN_BY) k_dn_atrous(const __grid_constant__ dn_args P, int it, int src, int last) {
    const int i = blockIdx.x * DN_BX + threadIdx.x, j = blockIdx.y * DN_BY + threadIdx.y;
    if (i >= P.nx || j >= P.ny) return;
    const float4* __restrict__ ev = P.ev[src];
    const int p = j * P.nx + i;
    const bool hp = P.hit[p];
    const float4 fp = P.feat[p];
    const float4 ep = ev[p];
    // 3x3 binomial blur of the variance over the neighbours p may mix with: same hit class, weights w_n for hits
    float gs = 0.f, gw = 0.f;
    for (int dy = -1; dy <= 1; ++dy) {
        const int qj = j + dy;
        if (qj < 0 || qj >= P.ny) continue;
        for (int dx = -1; dx <= 1; ++dx) {
            const int qi = i + dx;
            if (qi < 0 || qi >= P.nx) continue;
            const int q = qj * P.nx + qi;
            if ((bool)__ldg(&P.hit[q]) != hp) continue;
            float w = (float)((2 - abs(dx)) * (2 - abs(dy)));
            if (q != p && hp) w = w * dn_normal_weight(fp, __ldg(&P.feat[q]), P.k);
            gs = gs + w * __ldg(&ev[q].w);
            gw = gw + w;
        }
    }
    const float2 gp = P.grad[p];
    const float lp = dn_lum(ep);
    const float dl_den = P.sigma_l * sqrtf(gs / gw) + DN_EPS_LUM;
    const float H[5] = {1.f / 16.f, 1.f / 4.f, 3.f / 8.f, 1.f / 4.f, 1.f / 16.f};
    const int step = 1 << it;
    float sw = 0.f, sv = 0.f, sx = 0.f, sy = 0.f, sz = 0.f;
#pragma unroll
    for (int b = -2; b <= 2; ++b) {
        const int dy = b * step, qj = j + dy;
        if (qj < 0 || qj >= P.ny) continue;
#pragma unroll
        for (int a = -2; a <= 2; ++a) {
            const int dx = a * step, qi = i + dx;
            if (qi < 0 || qi >= P.nx) continue;
            const int q = qj * P.nx + qi;
            if ((bool)__ldg(&P.hit[q]) != hp) continue;
            const float4 eq = __ldg(&ev[q]);
            float w;
            if (a == 0 && b == 0) {
                w = H[2] * H[2];
            } else {
                const float dl = fabsf(lp - dn_lum(eq)) / dl_den;
                if (hp) {
                    const float4 fq = __ldg(&P.feat[q]);
                    const float dz = dn_depth_distance(fp.w, fq.w, gp, P.sigma_z, dx, dy);
                    w = H[a + 2] * H[b + 2] * dn_normal_weight(fp, fq, P.k) * dn_exp_neg(dz + dl);
                } else {
                    w = H[a + 2] * H[b + 2] * dn_exp_neg(dl);
                }
            }
            sw = sw + w;
            sx = sx + w * eq.x;
            sy = sy + w * eq.y;
            sz = sz + w * eq.z;
            sv = sv + w * w * eq.w;
        }
    }
    if (last) {
        P.out[3 * p] = (sx / sw) * dn_albedo(P, p, 0);
        P.out[3 * p + 1] = (sy / sw) * dn_albedo(P, p, 1);
        P.out[3 * p + 2] = (sz / sw) * dn_albedo(P, p, 2);
    } else {
        P.ev[1 - src][p] = make_float4(sx / sw, sy / sw, sz / sw, sv / (sw * sw));
    }
}

// the epilogue of the sample loop, PSC/main.cpp:315-325, one thread per pixel; output row 0 = top row (j = ny-1)
__global__ void k_quantize(const float* __restrict__ sums, int nx, int ny, float inv_ns, int clamp255, int32_t* __restrict__ out) {
    const int q = blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= nx * ny) return;
    const int row = q / nx, i = q - row * nx, j = ny - 1 - row;
    const float* src = sums + 3ull * ((unsigned long long)j * nx + i);
#pragma unroll
    for (int c = 0; c < 3; ++c) {
        const float col = sqrtf(src[c] * inv_ns);      // col /= float(ns) multiplies by k = float(1.0/ns), PSC/vec3.h:134-141
        const double x = 255.99 * (double)col;          // int(255.99*col[c]): the product is a double
        // out of int range or NaN (a NaN sum without de_nan): x86's cvttsd2si, which the reference binary executes, returns
        // INT_MIN; CUDA's conversion would saturate / give 0
        int v = (x > -2147483649.0 && x < 2147483648.0) ? (int)x : (int)0x80000000;
        if (clamp255 && v > 255) v = 255;
        out[3ull * q + c] = v;
    }
}

// chunks > 1: the fixed-point sums of the subset's pixels become float sums (added to accum with RTNW_F_ACCUMULATE) and the
// plane is cleared for the next render
__global__ void k_finish_fixed(unsigned long long* __restrict__ fixed, int pixel_begin, int pixel_stride, int pixel_count,
                               int accumulate, float* __restrict__ accum) {
    const int q = blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= pixel_count) return;
    const unsigned long long at = 3ull * (unsigned long long)(pixel_begin + q * pixel_stride);
#pragma unroll
    for (int c = 0; c < 3; ++c) {
        const float v = from_fixed(fixed[at + c]);
        fixed[at + c] = 0ull;
        if (accumulate) accum[at + c] += v; else accum[at + c] = v;
    }
}

// FP32 issue peak of the device, measured: 8 independent FFMA chains per thread (the roofline denominator of bench.py)
__global__ void __launch_bounds__(256) k_fma_peak(float* out, int iters) {
    float a0 = threadIdx.x * 1e-3f, a1 = a0 + 1.f, a2 = a0 + 2.f, a3 = a0 + 3.f, a4 = a0 + 4.f, a5 = a0 + 5.f, a6 = a0 + 6.f, a7 = a0 + 7.f;
    const float m = 0.999f, c = 1e-3f;
    for (int i = 0; i < iters; ++i) {
        a0 = __fmaf_rn(a0, m, c); a1 = __fmaf_rn(a1, m, c); a2 = __fmaf_rn(a2, m, c); a3 = __fmaf_rn(a3, m, c);
        a4 = __fmaf_rn(a4, m, c); a5 = __fmaf_rn(a5, m, c); a6 = __fmaf_rn(a6, m, c); a7 = __fmaf_rn(a7, m, c);
    }
    if (a0 + a1 + a2 + a3 + a4 + a5 + a6 + a7 == 12345.678f) out[0] = a0;  // keeps the chains alive
}

// Self-test of the reciprocal shortcuts (rtnw_device.cuh, "IEEE quotients from a reciprocal"): every thread draws boxes,
// spheres and rays — scene-like values, origins exactly on face planes, zero / tiny / huge direction components, NaN and
// infinities, exponents over the whole float range — and compares hit_box<true> / hit_sphere_recip with the IEEE forms
// bit for bit; plus raw quotients inside the guard.  out: {box mismatches, sphere mismatches, quotient mismatches,
// boxes that took the reciprocal path, spheres tested with a positive discriminant, box hits}.
__device__ __forceinline__ float selftest_float(uint32_t bits, uint32_t mode) {
    const uint32_t sign = bits & 0x80000000u, man = bits & 0x7fffffu;
    switch (mode & 7u) {
        case 0: return __uint_as_float(sign | ((100u + ((bits >> 23) & 63u)) << 23) | (0x7fffffu - (man & 0xffu)));  // mantissa near all ones
        case 1: return __uint_as_float(sign | ((100u + ((bits >> 23) & 63u)) << 23) | (man & 0xffu));               // mantissa near 1.0
        case 2: return __uint_as_float(bits);                                                                        // any float at all
        case 3: return (bits & 1u) ? 0.0f : -0.0f;
        default: return ((float)(int32_t)bits) * (1000.0f / 2147483648.0f);                                          // scene-like
    }
}
__global__ void k_selftest_recip(uint64_t n, uint32_t seed, unsigned long long* out) {
    unsigned long long bad_box = 0, bad_sph = 0, bad_div = 0, fast_box = 0, disc_pos = 0, box_hits = 0;
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) {
        uint4 w[4];
        for (uint32_t j = 0; j < 4; ++j) w[j] = philox_block((uint32_t)i, (uint32_t)(i >> 32), j, 0x5e1f7e57u, seed, 0u);
        const uint32_t m = w[3].w;  // per-case mode word
        // ---- raw quotient inside the guard: d and q within 2^+-40 / 2^80 is implied by exponents 100..163 both
        {
            const float x = selftest_float(w[0].x, (m >> 0) & 1u ? 0u : 1u), d = selftest_float(w[0].y, (m >> 1) & 1u ? 0u : 1u);
            const float y = 1.0f / d;
            const float xx = ((m >> 2) & 15u) == 0u ? 0.0f * x : x, q = div_by_recip(xx, d, y), ref = xx / d;
            if (__float_as_uint(q) != __float_as_uint(ref) && !(q == 0.0f && ref == 0.0f)) ++bad_div;  // the sign of a zero quotient may differ
        }
        // ---- ray, box, sphere
        const uint32_t vmode = ((m >> 6) & 3u) == 0u ? 2u : 4u;          // a quarter of the cases: any float at all
        ray_t r;
        r.o = mk3(selftest_float(w[0].z, vmode), selftest_float(w[0].w, vmode), selftest_float(w[1].x, vmode));
        r.d = mk3(selftest_float(w[1].y, vmode), selftest_float(w[1].z, vmode), selftest_float(w[1].w, vmode));
        r.time = 0.f;
        if (((m >> 8) & 7u) == 0u) r.d.x = selftest_float(w[3].x, 3u);   // exact zeros
        if (((m >> 11) & 7u) == 0u) r.d.y *= 1e-30f;                     // below the guard
        if (((m >> 14) & 15u) == 0u) r.d.z *= 1e30f;                     // above the guard
        f3 p0 = mk3(selftest_float(w[2].x, vmode), selftest_float(w[2].y, vmode), selftest_float(w[2].z, vmode));
        f3 p1 = mk3(selftest_float(w[2].w, vmode), selftest_float(w[3].x, vmode), selftest_float(w[3].y, vmode));
        if (p0.x > p1.x) { const float t = p0.x; p0.x = p1.x; p1.x = t; }
        if (p0.y > p1.y) { const float t = p0.y; p0.y = p1.y; p1.y = t; }
        if (p0.z > p1.z) { const float t = p0.z; p0.z = p1.z; p1.z = t; }
        if (((m >> 18) & 3u) == 0u) r.o.y = p1.y;                        // the ray leaves a face of the box
        if (((m >> 20) & 7u) == 0u) r.o.x = p0.x;
        if (((m >> 23) & 1u) == 0u) {                                    // aim at the box so that hits are common
            const float u = u01(w[3].z), v = u01(w[3].w), q = u01(w[1].x ^ w[2].y);
            r.d = mk3(p0.x + u * (p1.x - p0.x), p0.y + v * (p1.y - p0.y), p0.z + q * (p1.z - p0.z)) - r.o;
        }
        const float t_lo = ((m >> 24) & 7u) == 0u ? 1e-12f : (((m >> 24) & 7u) == 1u ? 0.01f : 0.001f);
        const float t_hi = ((m >> 27) & 1u) ? FLT_MAX : fabsf(selftest_float(w[3].z, 4u));
        ray_recip rr;
        rr.inv = mk3(1.0f / r.d.x, 1.0f / r.d.y, 1.0f / r.d.z);
        const float a = dot(r.d, r.d);
        rr.inv_a = 1.0f / a;
        {
            float ta = 0.f, tb = 0.f; int fa = 0, fb = 0; bool ieee = true;
            const bool ha = hit_box<ARITH_RECIP>(p0, p1, r, rr, t_lo, t_hi, ta, fa, &ieee);
            const bool hb = hit_box<ARITH_IEEE>(p0, p1, r, rr, t_lo, t_hi, tb, fb);
            if (ha != hb || (ha && (__float_as_uint(ta) != __float_as_uint(tb) || fa != fb))) ++bad_box;
#ifdef RTNW_SELFTEST_PRINT
            if ((ha != hb || (ha && (__float_as_uint(ta) != __float_as_uint(tb) || fa != fb))) && bad_box <= 1 && blockIdx.x < 4 && threadIdx.x < 8)
                printf("box o=(%a %a %a) d=(%a %a %a) p0=(%a %a %a) p1=(%a %a %a) tlo=%a thi=%a | recip hit=%d t=%a f=%d ieee=%d | ref hit=%d t=%a f=%d\n",
                       r.o.x, r.o.y, r.o.z, r.d.x, r.d.y, r.d.z, p0.x, p0.y, p0.z, p1.x, p1.y, p1.z, t_lo, t_hi, (int)ha, ta, fa, (int)ieee, (int)hb, tb, fb);
#endif
            if (!ieee) ++fast_box;
            if (hb) ++box_hits;
        }
        {
            const f3 c = 0.5f * (p0 + p1);
            const float radius = 0.5f * fabsf(p1.x - p0.x);
            float ta = 0.f, tb = 0.f;
            const bool ha = hit_sphere_recip(c, radius, r, a, rr.inv_a, t_lo, t_hi, ta);
            const bool hb = hit_sphere(c, radius, r, a, t_lo, t_hi, tb);
            if (ha != hb || (ha && __float_as_uint(ta) != __float_as_uint(tb))) ++bad_sph;
            if (hb) ++disc_pos;
        }
    }
    if (bad_box) atomicAdd(&out[0], bad_box);
    if (bad_sph) atomicAdd(&out[1], bad_sph);
    if (bad_div) atomicAdd(&out[2], bad_div);
    atomicAdd(&out[3], fast_box);
    atomicAdd(&out[4], disc_pos);
    atomicAdd(&out[5], box_hits);
}

__global__ void k_eval_texture(const scene_view S, int tex, const float* __restrict__ uvp, size_t n, float* __restrict__ rgb) {
    const size_t q = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= n) return;
    const float* in = uvp + 5 * q;
    const f3 c = texture_value(S, tex, in[0], in[1], mk3(in[2], in[3], in[4]));
    rgb[3 * q] = c.x; rgb[3 * q + 1] = c.y; rgb[3 * q + 2] = c.z;
}

__global__ void k_eval_perlin(const scene_view S, int which, const float* __restrict__ xyz, size_t n, float* __restrict__ out) {
    const size_t q = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= n) return;
    const f3 p = mk3(xyz[3 * q], xyz[3 * q + 1], xyz[3 * q + 2]);
    out[q] = which == 0 ? perlin_noise(S, p) : perlin_turb(S, p);
}

__global__ void k_scatter(const scene_view S, const rtnw_ray* __restrict__ rays_in, const rtnw_hit* __restrict__ hits, size_t n,
                          uint64_t seed, rtnw_ray* __restrict__ out_sc, float* __restrict__ out_att, float* __restrict__ out_em,
                          int32_t* __restrict__ out_flag) {
    const size_t q = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= n) return;
    const rtnw_ray in = rays_in[q];
    const rtnw_hit hh = hits[q];
    ray_t r;
    r.o = mk3(in.origin[0], in.origin[1], in.origin[2]);
    r.d = mk3(in.direction[0], in.direction[1], in.direction[2]);
    r.time = in.time;
    surf_t s;
    s.p = mk3(hh.p[0], hh.p[1], hh.p[2]);
    s.n = mk3(hh.normal[0], hh.normal[1], hh.normal[2]);
    s.u = hh.u; s.v = hh.v; s.mat = hh.mat_id;
    rng_t g;
    g.begin((uint32_t)seed, (uint32_t)(seed >> 32), (uint32_t)q, 0u);
    const f3 em = material_emitted(S, s.mat, s.u, s.v, s.p);
    f3 att = mk3(0.f, 0.f, 0.f);
    ray_t sc;
    sc.o = att; sc.d = att; sc.time = 0.f;
    const bool ok = material_scatter(S, s.mat, r, s, g, att, sc);
    rtnw_ray o;
    memset(&o, 0, sizeof o);
    if (ok) {
        o.origin[0] = sc.o.x; o.origin[1] = sc.o.y; o.origin[2] = sc.o.z;
        o.direction[0] = sc.d.x; o.direction[1] = sc.d.y; o.direction[2] = sc.d.z;
        o.time = sc.time;
    } else {
        att = mk3(0.f, 0.f, 0.f);
    }
    o.key = (uint32_t)q;
    out_sc[q] = o;
    out_att[3 * q] = att.x; out_att[3 * q + 1] = att.y; out_att[3 * q + 2] = att.z;
    out_em[3 * q] = em.x; out_em[3 * q + 1] = em.y; out_em[3 * q + 2] = em.z;
    out_flag[q] = ok ? 1 : 0;
}

__global__ void k_camera_rays(const rtnw_camera cam, int nx, int ny, const int32_t* __restrict__ ij, const int32_t* __restrict__ sample,
                              size_t n, uint64_t seed, rtnw_ray* __restrict__ out) {
    const size_t q = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= n) return;
    const int i = ij[2 * q], j = ij[2 * q + 1];
    rng_t g;
    g.begin((uint32_t)seed, (uint32_t)(seed >> 32), (uint32_t)(j * nx + i), (uint32_t)sample[q]);
    ray_t r;
    camera_ray(cam, nx, ny, i, j, g, r);
    rtnw_ray o;
    o.origin[0] = r.o.x; o.origin[1] = r.o.y; o.origin[2] = r.o.z;
    o.direction[0] = r.d.x; o.direction[1] = r.d.y; o.direction[2] = r.d.z;
    o.time = r.time;
    o.key = (uint32_t)(j * nx + i);
    out[q] = o;
}

// camera::get_ray(s, t) for n (s, t) pairs, PSC/camera.h:41-47: the lens and shutter draws come from the path stream (seed, key_base + q, 0)
__global__ void k_camera_get_rays(const rtnw_camera cam, const float* __restrict__ st, size_t n, uint64_t seed, uint32_t key_base,
                                  rtnw_ray* __restrict__ out) {
    const size_t q = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= n) return;
    rng_t g;
    g.begin((uint32_t)seed, (uint32_t)(seed >> 32), key_base + (uint32_t)q, 0u);
    ray_t r;
    camera_get_ray(cam, st[2 * q], st[2 * q + 1], g, r);
    rtnw_ray o;
    o.origin[0] = r.o.x; o.origin[1] = r.o.y; o.origin[2] = r.o.z;
    o.direction[0] = r.d.x; o.direction[1] = r.d.y; o.direction[2] = r.d.z;
    o.time = r.time;
    o.key = key_base + (uint32_t)q;
    out[q] = o;
}

// rtnw_render_multi: the ranks' float sums added in rank order on device 0; src[r] may be peer memory read over NVLink
struct rank_planes { const float* src[RTNW_MAX_DEVICES]; int n; };
__global__ void k_sum_ranks(float* __restrict__ dst, const rank_planes P, size_t count) {
    const size_t stride = (size_t)gridDim.x * blockDim.x;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < count; i += stride) {
        float v = dst[i];
        for (int r = 1; r < P.n; ++r) v += P.src[r][i];
        dst[i] = v;
    }
}

// ================================================================================================ host side
namespace {

thread_local std::string g_err;
int fail(int code, const std::string& msg) {
    g_err = msg;
    return code;
}
#define CUDA_TRY(expr)                                                                                       \
    do {                                                                                                     \
        cudaError_t e_ = (expr);                                                                             \
        if (e_ != cudaSuccess)                                                                               \
            return fail(RTNW_ERR_CUDA, std::string(#expr) + ": " + cudaGetErrorString(e_));                  \
    } while (0)

struct dev_buf {  // RAII device allocation for the query entry points
    void* p = nullptr;
    ~dev_buf() { if (p) cudaFree(p); }
    cudaError_t alloc(size_t bytes) { return cudaMalloc(&p, bytes ? bytes : 1); }
    template <class T> T* as() { return static_cast<T*>(p); }
};

// Lays out n tables of sz[i] bytes back to back, each at a 256-byte aligned offset off[i]; returns the total size.
size_t layout256(const size_t* sz, int n, size_t* off) {
    size_t total = 0;
    for (int i = 0; i < n; ++i) {
        off[i] = total;
        total += (sz[i] + 255) & ~(size_t)255;
    }
    return total;
}

// The device buffers of one query call in one allocation.  add() declares a span of `bytes` with a host source (copied
// in), a host destination (copied out), both, or neither (device scratch) and returns its index.  copy_in allocates every
// span (layout256) and copies the sources in; copy_out copies the destinations out and waits for the stream.  The
// optional events are recorded before the copies in and after the copies out (the total_ms of rtnw_stats).
struct staging {
    static constexpr int MAX_SPANS = 10;
    size_t bytes[MAX_SPANS], off[MAX_SPANS];
    const void* src[MAX_SPANS];
    void* dst[MAX_SPANS];
    int n = 0;
    dev_buf d;

    int add(size_t size, const void* from = nullptr, void* to = nullptr) {
        bytes[n] = size;
        src[n] = from;
        dst[n] = to;
        return n++;
    }
    template <class T> T* at(int i) { return reinterpret_cast<T*>(d.as<unsigned char>() + off[i]); }
    cudaError_t copy_in(cudaStream_t st, cudaEvent_t start = nullptr) {
        cudaError_t e = d.alloc(layout256(bytes, n, off));
        if (e == cudaSuccess && start) e = cudaEventRecord(start, st);
        for (int i = 0; i < n && e == cudaSuccess; ++i)
            if (src[i]) e = cudaMemcpyAsync(at<void>(i), src[i], bytes[i], cudaMemcpyHostToDevice, st);
        return e;
    }
    cudaError_t copy_out(cudaStream_t st, cudaEvent_t done = nullptr) {
        cudaError_t e = cudaSuccess;
        for (int i = 0; i < n && e == cudaSuccess; ++i)
            if (dst[i]) e = cudaMemcpyAsync(dst[i], at<void>(i), bytes[i], cudaMemcpyDeviceToHost, st);
        if (e == cudaSuccess && done) e = cudaEventRecord(done, st);
        return e == cudaSuccess ? cudaStreamSynchronize(st) : e;
    }
};

// Makes *buf hold at least `count` elements of device memory: a smaller buffer is freed and replaced, its contents are
// not kept.  On failure *buf is null, *cap is 0 and the call fails with RTNW_ERR_NOMEM and `what`.
template <class T>
int grow(T** buf, size_t* cap, size_t count, const char* what) {
    if (*cap >= count) return RTNW_OK;
    if (*buf) cudaFree(*buf);
    *buf = nullptr;
    *cap = 0;
    if (cudaMalloc(buf, count * sizeof(T)) != cudaSuccess) {
        cudaGetLastError();
        return fail(RTNW_ERR_NOMEM, what);
    }
    *cap = count;
    return RTNW_OK;
}

// Launches a block-cooperative kernel whose dynamic shared memory is one SMEM.  That is more than the 48 KB a kernel gets
// by default, so the kernel opts in first.
template <class SMEM, class... P, class... A>
int launch_coop(void (*k)(P...), unsigned grid, cudaStream_t st, const A&... args) {
    CUDA_TRY(cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(SMEM)));
    k<<<grid, RTNW_BLOCK, sizeof(SMEM), st>>>(args...);
    CUDA_TRY(cudaGetLastError());
    return RTNW_OK;
}

// Calls f(count, fast) with the flags that select a traversal kernel's instantiation, RTNW_F_COUNTERS and RTNW_F_FAST_BVH,
// as std::bool_constant values, so that f can name the instantiation with decltype(count)::value.
template <class F>
int by_variant(uint32_t flags, F&& f) {
    using T = std::true_type;
    using N = std::false_type;
    const bool count = (flags & RTNW_F_COUNTERS) != 0;
    if (flags & RTNW_F_FAST_BVH) return count ? f(T(), T()) : f(N(), T());
    return count ? f(T(), N()) : f(N(), N());
}

}  // namespace

struct rtnw_ctx {
    int device = 0;
    cudaStream_t stream = nullptr;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    int sm_count = 0, clock_khz = 0, smem_optin = 0, l2_bytes = 0;
    float* accum = nullptr;          // device accumulation buffer of rtnw_render
    size_t accum_floats = 0;
    unsigned long long* fixed = nullptr;  // fixed-point plane of the sample-range split (zero between renders)
    size_t fixed_words = 0;
    unsigned long long* ctr = nullptr;       // 8 device counters
    unsigned long long* ctr_host = nullptr;  // their pinned host copy (filled asynchronously after every render)
    cudaEvent_t ev_t0 = nullptr, ev_t1 = nullptr;  // rtnw_render's total_ms
    int blocks_per_sm[4] = {0, 0, 0, 0};
    // freed scene slabs are kept for the next upload (cudaMalloc/cudaFree synchronise the device and can take
    // milliseconds to hundreds of milliseconds in a process that also hosts another allocator)
    void* spare_slab[2] = {nullptr, nullptr};
    size_t spare_bytes[2] = {0, 0};
};

struct rtnw_scene {
    scene_view view;
    void* slab = nullptr;  // one allocation holding every table
    size_t slab_bytes = 0;
};

namespace {

// ---- scene_desc -> record stream -----------------------------------------------------------------------------
struct stream_builder {
    const rtnw_scene_desc& d;
    std::vector<rec> recs;
    std::vector<int32_t> leaf;
    std::vector<uint32_t> rec_xf;  // per record: transform chain of its item
    uint32_t cur_item_xf = 0;
    std::string err;
    explicit stream_builder(const rtnw_scene_desc& desc) : d(desc) {}

    static float bits(int32_t v) { float f; std::memcpy(&f, &v, 4); return f; }
    static float ubits(uint32_t v) { float f; std::memcpy(&f, &v, 4); return f; }
    static int32_t as_int(float f) { int32_t v; std::memcpy(&v, &f, 4); return v; }
    static uint32_t as_uint(float f) { uint32_t v; std::memcpy(&v, &f, 4); return v; }

    bool bad(const std::string& m) { if (err.empty()) err = m; return false; }

    bool chain_ok(uint32_t chain) {
        if (chain == 0) return true;
        if (chain >= (uint32_t)d.n_xform_ops) return bad("transform chain index out of range");
        const uint32_t n = d.xforms[chain].kind >> 8;
        if (n == 0 || chain + n > (uint32_t)d.n_xform_ops) return bad("transform chain length out of range");
        for (uint32_t k = 0; k < n; ++k) {
            const uint32_t kk = d.xforms[chain + k].kind & 0xffu;
            if (kk != RTNW_XF_TRANSLATE && kk != RTNW_XF_ROTATE_Y) return bad("unknown transform op");
        }
        return true;
    }

    void push(float4 a, float bx, float by, uint32_t tag, int32_t w, int32_t leaf_id) {
        rec r;
        r.a = a;
        r.b = make_float4(bx, by, ubits(tag), bits(w));
        recs.push_back(r);
        leaf.push_back(leaf_id);
        rec_xf.push_back(cur_item_xf);
    }

    // Append the records of prim slots [first, first+count).  first_cont: narrowing flag of the first primitive;
    // the following primitives of the range always continue its scope (list semantics).
    // class of a prim slot for the run-specialised list scan (scan_run): 1 plain sphere, 2 plain moving sphere, 3 plain box, 0 other
    int run_class(int32_t s, int32_t end) const {
        const rtnw_prim& p = d.prims[s];
        if (RTNW_KX_XFORM(p.kx) != 0) return 0;
        switch (RTNW_KX_KIND(p.kx)) {
            case RTNW_PRIM_SPHERE: return 1;
            case RTNW_PRIM_MOVING_SPHERE: return (s + 1 < end && RTNW_KX_KIND(d.prims[s + 1].kx) == RTNW_PRIM_EXT) ? 2 : 0;
            case RTNW_PRIM_BOX: return 3;
            default: return 0;
        }
    }
    static constexpr int MIN_RUN = 8;  // primitives; shorter runs stay in the generic scan

    bool emit_prims(int32_t first, int32_t count, bool first_cont, bool boundary, bool allow_runs = false) {
        if (first < 0 || count < 0 || count > d.n_prim_slots - first) return bad("primitive range out of bounds");
        bool cont = first_cont;
        size_t last_head = (size_t)-1;  // the record a leaf scan tests last (a moving sphere / medium head, not its trailing records)
        int32_t run_end = first;        // slots below this one already belong to a run that has its header
        int32_t pad_spheres_until = first;  // plain spheres below this slot sit in a mixed sphere / moving-sphere run: padded to two records
        for (int32_t s = first; s < first + count; ++s) {
            if (allow_runs && s >= run_end) {  // does a run of plain spheres / (moving) spheres / boxes start here?
                const int c0 = run_class(s, first + count);
                if (c0) {
                    const bool sph = c0 <= 2;
                    bool pure = c0 == 1;
                    int32_t q = s, prims = 0, nrec = 0;
                    while (q < first + count) {
                        const int c = run_class(q, first + count);
                        if (!c || (c <= 2) != sph) break;
                        pure = pure && c == 1;
                        ++prims; nrec += c == 2 ? 2 : 1; q += c == 2 ? 2 : 1;
                    }
                    pad_spheres_until = first;
                    if (prims >= MIN_RUN) {
                        const uint32_t k = sph ? (pure ? K_RUN_SPHERE : K_RUN_SPHERELIKE) : K_RUN_BOX;
                        if (k == K_RUN_SPHERELIKE) { nrec = 2 * prims; pad_spheres_until = q; }  // every primitive of a mixed run takes two records
                        push(make_float4(bits(nrec), 0, 0, 0), 0, 0, RTNW_TAG(k, 0, 1, 0), 0, -1);
                    }
                    run_end = q;  // (short runs are not examined again)
                }
            }
            last_head = recs.size();
            const rtnw_prim& p = d.prims[s];
            const uint32_t kind = RTNW_KX_KIND(p.kx), flip = RTNW_KX_FLIP(p.kx), chain = RTNW_KX_XFORM(p.kx);
            const int32_t id = (d.prim_ids && !boundary) ? d.prim_ids[s] : -1;
            if (kind == RTNW_PRIM_EXT) return bad("stray continuation slot");
            if (!chain_ok(chain)) return false;
            if (chain >= (1u << 24)) return bad("transform chain index exceeds 24 bits");
            if (!boundary && (p.mat < 0 || p.mat >= d.n_materials)) return bad("material index out of range");
            switch (kind) {
                case RTNW_PRIM_SPHERE:
                    // in a mixed run a plain sphere is laid out like a moving one that does not move: shutter (0, 1), c1 = c0, so
                    // that center(time) = c0 + time * (c0 - c0) = c0 exactly and the run's loop needs no case distinction
                    push(make_float4(p.f[0], p.f[1], p.f[2], p.f[3]), 0, s < pad_spheres_until ? 1.f : 0.f, RTNW_TAG(K_SPHERE, flip, cont, chain), p.mat, id);
                    if (s < pad_spheres_until) push(make_float4(p.f[0], p.f[1], p.f[2], 0), 0, 0, RTNW_TAG(K_EXT, 0, 1, 0), -1, id);
                    break;
                case RTNW_PRIM_MOVING_SPHERE: {
                    if (s + 1 >= first + count || RTNW_KX_KIND(d.prims[s + 1].kx) != RTNW_PRIM_EXT)
                        return bad("moving sphere without its continuation slot");
                    const rtnw_prim& e = d.prims[s + 1];
                    push(make_float4(p.f[0], p.f[1], p.f[2], p.f[3]), p.f[4], p.f[5], RTNW_TAG(K_MSPHERE, flip, cont, chain), p.mat, id);
                    push(make_float4(e.f[0], e.f[1], e.f[2], 0), 0, 0, RTNW_TAG(K_EXT, 0, 1, 0), -1, id);
                    ++s;
                    break;
                }
                case RTNW_PRIM_RECT_XY:
                case RTNW_PRIM_RECT_XZ:
                case RTNW_PRIM_RECT_YZ: {
                    const uint32_t k = kind == RTNW_PRIM_RECT_XY ? K_RECT_XY : (kind == RTNW_PRIM_RECT_XZ ? K_RECT_XZ : K_RECT_YZ);
                    push(make_float4(p.f[0], p.f[1], p.f[2], p.f[3]), p.f[4], 0, RTNW_TAG(k, flip, cont, chain), p.mat, id);
                    break;
                }
                case RTNW_PRIM_BOX:
                    push(make_float4(p.f[0], p.f[1], p.f[2], p.f[3]), p.f[4], p.f[5], RTNW_TAG(K_BOX, flip, cont, chain), p.mat, id);
                    break;
                case RTNW_PRIM_MEDIUM: {
                    if (boundary) return bad("constant_medium as the boundary of a constant_medium");
                    const int32_t bfirst = as_int(p.f[1]), bcount = as_int(p.f[2]);
                    const size_t at = recs.size();
                    push(make_float4(p.f[0], p.f[3] /* leaf id bits */, 0, -(1.0f / p.f[0])), 0, 0, RTNW_TAG(K_MEDIUM, flip, cont, chain), p.mat, id);
                    if (!emit_prims(bfirst, bcount, true, true)) return false;
                    recs[at].a.z = bits((int32_t)(recs.size() - at - 1));
                    for (size_t q = at + 1; q < recs.size(); ++q) leaf[q] = id;
                    break;
                }
                default: return bad("unknown primitive kind");
            }
            cont = true;
        }
        if (!boundary && last_head != (size_t)-1) recs[last_head].b.z = ubits(as_uint(recs[last_head].b.z) | RTNW_TAG_LAST);
        return true;
    }

    // ---- gate tree (rtnw_device.cuh, "block-cooperative closest hit") ------------------------------------------
    struct gate_t { float bmin[3], bmax[3]; int32_t leaf0, leaf1; };
    struct bin_node { float bmin[3], bmax[3]; int left, right, gate; };  // binary SAH tree over gates; gate >= 0: leaf
    std::vector<gate_t> gates;          // all items
    std::vector<int2> gate_leaves;      // device table
    std::vector<float4> wnodes;         // device table, 8 float4 per wide node
    std::vector<uint8_t> node_seen;

    // bvh_node `idx` with own box [bmin,bmax]: its leaves go to the record stream in left-to-right order (the key's tie
    // rule relies on it); every leaf child becomes (part of) a gate guarded by THIS node's box.
    bool collect_gates(int32_t idx, const float* bmin, const float* bmax, int depth, std::vector<int>& mine, std::vector<int>& fmine) {
        if (idx < 0 || idx >= d.n_nodes) return bad("BVH node index out of range");
        if (depth > 4096) return bad("BVH deeper than 4096 levels (cycle?)");
        if (node_seen[idx]) return bad("BVH node referenced twice");
        node_seen[idx] = 1;
        const rtnw_bvh_node& n = d.nodes[idx];
        if (n.left == RTNW_REF_NONE) return bad("BVH node without a left child");
        const int32_t child[2] = {n.left, n.right};
        const int32_t cnt[2] = {n.lcount, n.rcount};
        const float* cmin[2] = {n.lmin, n.rmin};
        const float* cmax[2] = {n.lmax, n.rmax};
        gate_t g;
        for (int a = 0; a < 3; ++a) { g.bmin[a] = bmin[a]; g.bmax[a] = bmax[a]; }
        g.leaf0 = g.leaf1 = -1;
        for (int w = 0; w < 2; ++w) {
            if (child[w] == RTNW_REF_NONE) continue;
            if (child[w] >= 0) {
                if (!collect_gates(child[w], cmin[w], cmax[w], depth + 1, mine, fmine)) return false;
            } else {
                const size_t first = recs.size();
                if (!emit_prims(~child[w], cnt[w], false, false)) return false;
                if (recs.size() == first) return bad("empty BVH leaf");
                (g.leaf0 < 0 ? g.leaf0 : g.leaf1) = (int32_t)first;
                // RTNW_F_FAST_BVH: the leaf behind its OWN box (the reference's bounding_box of it, slightly padded: a primitive test
                // in float32 can accept a ray that a tight float32 slab test of its box rejects, within rounding of the silhouette)
                gate_t f;
                float side = 0.f, reach = 0.f;
                for (int a = 0; a < 3; ++a) {
                    side = std::fmax(side, cmax[w][a] - cmin[w][a]);
                    reach = std::fmax(reach, std::fmax(std::fabs(cmin[w][a]), std::fabs(cmax[w][a])));
                }
                const float pad = side * (1.0f / 1024.0f) + reach * (1.0f / 131072.0f);
                for (int a = 0; a < 3; ++a) { f.bmin[a] = cmin[w][a] - pad; f.bmax[a] = cmax[w][a] + pad; }
                f.leaf0 = (int32_t)first;
                f.leaf1 = -1;
                fmine.push_back((int)gates.size());
                gates.push_back(f);
                gate_leaves.push_back(make_int2(f.leaf0, -1));
            }
        }
        if (g.leaf0 >= 0) {
            mine.push_back((int)gates.size());
            gates.push_back(g);
            gate_leaves.push_back(make_int2(g.leaf0, g.leaf1));
        }
        return true;
    }

    static double half_area(const float* lo, const float* hi) {
        const double x = (double)hi[0] - lo[0], y = (double)hi[1] - lo[1], z = (double)hi[2] - lo[2];
        return x * y + y * z + z * x;
    }
    void bounds_of(const std::vector<int>& ids, size_t lo, size_t hi, float* bmin, float* bmax) const {
        for (int a = 0; a < 3; ++a) { bmin[a] = gates[ids[lo]].bmin[a]; bmax[a] = gates[ids[lo]].bmax[a]; }
        for (size_t q = lo + 1; q < hi; ++q)
            for (int a = 0; a < 3; ++a) {  // exact unions: the monotonicity argument needs nothing else
                bmin[a] = std::fmin(bmin[a], gates[ids[q]].bmin[a]);
                bmax[a] = std::fmax(bmax[a], gates[ids[q]].bmax[a]);
            }
    }
    // binary SAH split by full sweep over the three centroid orders (gate counts are small: <= #leaves)
    int build_binary(std::vector<int>& ids, size_t lo, size_t hi, std::vector<bin_node>& out) {
        const int me = (int)out.size();
        out.push_back(bin_node());
        bin_node nd;
        bounds_of(ids, lo, hi, nd.bmin, nd.bmax);
        nd.left = nd.right = -1;
        nd.gate = -1;
        if (hi - lo == 1) {
            nd.gate = ids[lo];
            out[me] = nd;
            return me;
        }
        double best_cost = 1e300;
        int best_axis = 0;
        size_t best_split = lo + (hi - lo) / 2;
        std::vector<double> right_area(hi - lo);
        for (int axis = 0; axis < 3; ++axis) {
            std::stable_sort(ids.begin() + lo, ids.begin() + hi, [&](int x, int y) {
                return gates[x].bmin[axis] + gates[x].bmax[axis] < gates[y].bmin[axis] + gates[y].bmax[axis];
            });
            float rmin[3], rmax[3];
            for (size_t q = hi; q-- > lo;) {
                if (q == hi - 1) { for (int a = 0; a < 3; ++a) { rmin[a] = gates[ids[q]].bmin[a]; rmax[a] = gates[ids[q]].bmax[a]; } }
                else for (int a = 0; a < 3; ++a) { rmin[a] = std::fmin(rmin[a], gates[ids[q]].bmin[a]); rmax[a] = std::fmax(rmax[a], gates[ids[q]].bmax[a]); }
                right_area[q - lo] = half_area(rmin, rmax);
            }
            float lmin[3], lmax[3];
            // keep both sides at least an eighth of the range: nested boxes would otherwise be peeled off one per level
            const size_t margin = (hi - lo) / 8;
            for (size_t q = lo; q + 1 < hi; ++q) {
                if (q == lo) { for (int a = 0; a < 3; ++a) { lmin[a] = gates[ids[q]].bmin[a]; lmax[a] = gates[ids[q]].bmax[a]; } }
                else for (int a = 0; a < 3; ++a) { lmin[a] = std::fmin(lmin[a], gates[ids[q]].bmin[a]); lmax[a] = std::fmax(lmax[a], gates[ids[q]].bmax[a]); }
                if (q + 1 - lo < margin || hi - q - 1 < margin) continue;
                const double cost = half_area(lmin, lmax) * (double)(q - lo + 1) + right_area[q + 1 - lo] * (double)(hi - q - 1);
                if (cost < best_cost) { best_cost = cost; best_axis = axis; best_split = q + 1; }
            }
        }
        std::stable_sort(ids.begin() + lo, ids.begin() + hi, [&](int x, int y) {
            return gates[x].bmin[best_axis] + gates[x].bmax[best_axis] < gates[y].bmin[best_axis] + gates[y].bmax[best_axis];
        });
        nd.left = build_binary(ids, lo, best_split, out);
        nd.right = build_binary(ids, best_split, hi, out);
        out[me] = nd;
        return me;
    }
    // Collapse binary trees into 4-wide nodes (repeatedly open the child with the largest box) and number the nodes of a
    // whole FOREST level by level: all roots first, then every tree's second level, and so on.  The traversal needs no
    // particular order; this one stays because every render measurement of the project was taken on the layout it gives.
    struct tree_t { std::vector<bin_node> bt; int broot = 0; size_t item_rec = 0; int root = 0, depth = 0; };
    void emit_forest(std::vector<tree_t>& forest) {
        struct pend { int tree, bnode, depth; size_t parent; int slot; };
        std::vector<pend> level, next;
        for (size_t t = 0; t < forest.size(); ++t) level.push_back(pend{(int)t, forest[t].broot, 0, (size_t)-1, 0});
        while (!level.empty()) {
            next.clear();
            for (const pend& p : level) {
                const std::vector<bin_node>& bt = forest[p.tree].bt;
                int kids[4], nk = 0;
                if (bt[p.bnode].gate >= 0) kids[nk++] = p.bnode;
                else { kids[nk++] = bt[p.bnode].left; kids[nk++] = bt[p.bnode].right; }
                while (nk < 4) {
                    int pick = -1;
                    double area = -1;
                    for (int q = 0; q < nk; ++q)
                        if (bt[kids[q]].gate < 0 && half_area(bt[kids[q]].bmin, bt[kids[q]].bmax) > area) { area = half_area(bt[kids[q]].bmin, bt[kids[q]].bmax); pick = q; }
                    if (pick < 0) break;
                    const int open = kids[pick];
                    kids[pick] = bt[open].left;
                    kids[nk++] = bt[open].right;
                }
                const size_t me = wnodes.size() / 8;
                wnodes.resize(wnodes.size() + 8, make_float4(0, 0, 0, 0));
                if (p.parent == (size_t)-1) forest[p.tree].root = (int)me;
                else (&wnodes[8 * p.parent + 6].x)[p.slot] = bits((int32_t)me);
                forest[p.tree].depth = std::max(forest[p.tree].depth, p.depth + 1);
                float v[6][4];
                int32_t ref[4];
                for (int q = 0; q < 4; ++q) {
                    ref[q] = RTNW_REF_NONE;
                    for (int a = 0; a < 6; ++a) v[a][q] = 0.f;
                }
                for (int q = 0; q < nk; ++q) {
                    const bin_node& c = bt[kids[q]];
                    for (int a = 0; a < 3; ++a) { v[a][q] = c.bmin[a]; v[3 + a][q] = c.bmax[a]; }
                    if (c.gate >= 0) ref[q] = ~c.gate;
                    else { ref[q] = 0; next.push_back(pend{p.tree, kids[q], p.depth + 1, me, q}); }  // patched when the child is numbered
                }
                for (int a = 0; a < 6; ++a) wnodes[8 * me + a] = make_float4(v[a][0], v[a][1], v[a][2], v[a][3]);
                wnodes[8 * me + 6] = make_float4(bits(ref[0]), bits(ref[1]), bits(ref[2]), bits(ref[3]));  // row 7 stays zero
            }
            level.swap(next);
        }
    }
    std::vector<tree_t> exact_forest, fast_forest;  // per BVH item: the gate tree (reference-exact traversal) and the tree over
                                                    // the leaves' own boxes (RTNW_F_FAST_BVH); numbered after the last item
    int32_t fast_base = 0;                          // first wide node of the fast forest

    // one BVH item: its leaves go to the record stream now, its two binary SAH trees are kept for emit_forest
    bool emit_bvh_item(const rtnw_item& it, size_t item_rec) {
        std::vector<int> mine, fmine;
        if (!collect_gates(it.first, it.bmin, it.bmax, 0, mine, fmine)) return false;
        if (mine.empty()) return bad("BVH without leaves");
        for (int pass = 0; pass < 2; ++pass) {
            std::vector<int>& ids = pass ? fmine : mine;
            std::vector<tree_t>& forest = pass ? fast_forest : exact_forest;
            forest.push_back(tree_t());
            tree_t& T = forest.back();
            T.item_rec = item_rec;
            T.bt.reserve(2 * ids.size());
            T.broot = build_binary(ids, 0, ids.size(), T.bt);
        }
        return true;
    }
    bool finish_forests() {
        emit_forest(exact_forest);
        fast_base = (int32_t)(wnodes.size() / 8);
        emit_forest(fast_forest);
        for (size_t t = 0; t < exact_forest.size(); ++t) {
            const tree_t &E = exact_forest[t], &F = fast_forest[t];
            if (2 * RTNW_BLOCK + 3 * std::max(E.depth, F.depth) + 8 > coop_smem<>::QN) return bad("gate tree deeper than the cooperative task stack can reserve for");
            recs[E.item_rec].a.y = bits(E.root);
            recs[E.item_rec].a.z = bits(E.depth);
            recs[E.item_rec].a.w = bits(F.root);   // RTNW_F_FAST_BVH: tree over the leaves' own boxes
            recs[E.item_rec].b.x = bits(F.depth);
        }
        return true;
    }

    bool run() {
        if (d.abi_version != RTNW_ABI_VERSION) return bad("scene_desc.abi_version does not match this library");
        if (d.n_items <= 0 || !d.items) return bad("scene has no items");
        if (d.n_nodes >= (1 << 24)) return bad("scene exceeds 2^24 BVH nodes");
        node_seen.assign((size_t)std::max(d.n_nodes, 1), 0);
        if (d.n_prim_slots < 0 || d.n_nodes < 0 || d.n_materials < 0 || d.n_textures < 0 || d.n_xform_ops < 1)
            return bad("negative table size (or missing identity transform op 0)");
        if ((d.n_prim_slots && !d.prims) || (d.n_nodes && !d.nodes) || (d.n_materials && !d.materials) ||
            (d.n_textures && !d.textures) || !d.xforms)
            return bad("null table pointer");
        if (!d.perlin_ranvec || !d.perlin_perm_x || !d.perlin_perm_y || !d.perlin_perm_z) return bad("null perlin table");
        for (int32_t t = 0; t < d.n_textures; ++t) {
            const rtnw_texture& x = d.textures[t];
            if (x.kind == RTNW_TEX_CHECKER) {
                if (x.i0 <= t || x.i1 <= t || x.i0 >= d.n_textures || x.i1 >= d.n_textures)
                    return bad("checker texture children must follow their parent in the table");
            } else if (x.kind == RTNW_TEX_IMAGE) {
                if (x.i0 < 0 || x.i1 <= 0 || x.i2 <= 0 || !d.images ||
                    (uint64_t)x.i0 + 3ull * (uint64_t)x.i1 * (uint64_t)x.i2 > d.image_bytes)
                    return bad("image texture outside the image pool");
            } else if (x.kind != RTNW_TEX_CONSTANT && x.kind != RTNW_TEX_NOISE && !(x.kind >= RTNW_TEX_NOISE_HASH && x.kind <= RTNW_TEX_NOISE_HERMITE)) {
                return bad("unknown texture kind");
            }
        }
        for (int32_t m = 0; m < d.n_materials; ++m) {
            const rtnw_material& x = d.materials[m];
            if (x.kind > RTNW_MAT_ISOTROPIC) return bad("unknown material kind");
            const bool needs_tex = x.kind == RTNW_MAT_LAMBERTIAN || x.kind == RTNW_MAT_DIFFUSE_LIGHT || x.kind == RTNW_MAT_ISOTROPIC;
            if (needs_tex && (x.tex < 0 || x.tex >= d.n_textures)) return bad("material texture index out of range");
        }
        for (int32_t i = 0; i < d.n_items; ++i) {
            const rtnw_item& it = d.items[i];
            if (!chain_ok(it.xform)) return false;
            if (it.xform >= (1u << 24)) return bad("transform chain index exceeds 24 bits");
            cur_item_xf = it.xform;
            const size_t at = recs.size();
            push(make_float4(0, 0, 0, 0), 0, 0, RTNW_TAG(K_ITEM, 0, 0, it.xform), (int32_t)it.kind, -1);
            if (it.kind == RTNW_ITEM_PRIMS) {
                if (!emit_prims(it.first, it.count, true, false, /*allow_runs=*/true)) return false;
            } else if (it.kind == RTNW_ITEM_BVH) {
                if (!emit_bvh_item(it, at)) return false;  // leaves -> record stream now; gates + trees -> side tables (finish_forests)
            } else {
                return bad("unknown item kind");
            }
            recs[at].a.x = bits((int32_t)recs.size());  // the next element of the top-level list (or K_END)
        }
        cur_item_xf = 0;
        push(make_float4(0, 0, 0, 0), 0, 0, RTNW_TAG(K_END, 0, 0, 0), 0, -1);
        if (!finish_forests()) return false;
        if (recs.size() >= (1u << 24) || gates.size() >= (1u << RTNW_IDX_BITS) || wnodes.size() / 8 >= (1u << RTNW_IDX_BITS)) return bad("scene exceeds the record / gate index range");
        if (gate_leaves.empty()) gate_leaves.push_back(make_int2(-1, -1));
        if (wnodes.empty()) wnodes.resize(8, make_float4(0, 0, 0, 0));
        return true;
    }
};

int check_ctx(rtnw_ctx* ctx) {
    if (!ctx) return fail(RTNW_ERR_INVALID, "null context");
    CUDA_TRY(cudaSetDevice(ctx->device));
    return RTNW_OK;
}

// k_render and k_aov set counter 4 when a block's traversal task stack overflowed: the frame is then incomplete
int check_task_stack(const rtnw_ctx* ctx) {
    if (ctx->ctr_host[4]) return fail(RTNW_ERR_UNSUPPORTED, "BVH task stack overflow: the tree is deeper than RTNW_QN/RTNW_BLOCK - 1 levels");
    return RTNW_OK;
}

// *stats (when given) = s, with kernel_ms between ctx->ev0 and ev1 and, when `total`, total_ms between ev_t0 and ev_t1
int report_stats(rtnw_ctx* ctx, rtnw_stats* stats, rtnw_stats s, bool total) {
    if (!stats) return RTNW_OK;
    CUDA_TRY(cudaEventElapsedTime(&s.kernel_ms, ctx->ev0, ctx->ev1));
    if (total) CUDA_TRY(cudaEventElapsedTime(&s.total_ms, ctx->ev_t0, ctx->ev_t1));
    *stats = s;
    return RTNW_OK;
}

// resident blocks per SM of k_render<COUNT, FAST> (cached per context)
template <bool COUNT, bool FAST>
int render_occupancy(rtnw_ctx* ctx, int* out) {
    int& bps = ctx->blocks_per_sm[(COUNT ? 1 : 0) + (FAST ? 2 : 0)];
    if (bps == 0) {
        CUDA_TRY(cudaFuncSetAttribute(k_render<COUNT, FAST>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(block_smem<FAST>)));
        CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&bps, k_render<COUNT, FAST>, RTNW_BLOCK, sizeof(block_smem<FAST>)));
        if (bps < 1) bps = 1;
    }
    *out = bps;
    return RTNW_OK;
}

template <bool COUNT, bool FAST>
int launch_render(rtnw_ctx* ctx, const render_args& a, cudaStream_t st) {
    int bps = 0;
    const int rc = render_occupancy<COUNT, FAST>(ctx, &bps);
    if (rc != RTNW_OK) return rc;
    int blocks = ctx->sm_count * bps;
    const long long warps_needed = ((long long)a.p.pixel_count * a.chunks + 31) / 32;
    const long long blocks_needed = (warps_needed * 32 + RTNW_BLOCK - 1) / RTNW_BLOCK;
    if (blocks_needed < blocks) blocks = (int)blocks_needed;
#ifdef RTNW_TUNING  // A/B builds only (scripts/ab_build.sh): the product library reads no environment on the launch path
    if (const char* e = getenv("RTNW_GRID_BLOCKS")) { const int v = atoi(e); if (v > 0) blocks = v; }
#endif
    k_render<COUNT, FAST><<<blocks, RTNW_BLOCK, sizeof(block_smem<FAST>), st>>>(a);
    CUDA_TRY(cudaGetLastError());
    return RTNW_OK;
}

// One thread owns one (pixel, sample range) work item at a time.  With whole pixels as items (one range) the kernel ends
// in a tail as long as the most expensive pixel — at 100 spp about 14 ms of 220, during which most of the device idles —
// and an image with fewer pixels than the device has resident threads (the reference's own 200x100 default is 20 000)
// never fills it.  So every pixel's samples are cut into contiguous ranges, handed out range-major; a range's partial
// sum is added to the pixel's 64-bit fixed-point sum (add_fixed) and k_finish_fixed turns the plane into floats
// (reproducible bit for bit; differs from the one-range float sum only by rounding).  Ranges are four samples long (more when
// there are more than ~110 samples per pixel) and the last ones shrink to 4, 2, 1, 1, because the kernel's tail is as long
// as the longest item still running when the items run out.  Measured on the bench workload: 453 (1 range) / 477 (2) /
// 490 (4) / 498 (16) Mpaths/s.
void pick_chunks(const rtnw_render_params& p, render_args& a) {
    int per_pixel = p.sample_count;  // most samples a pixel has in this call (ROTATE: sample_count is the frame's total over sample_stride ranks)
    if (p.flags & RTNW_F_ROTATE_SAMPLES) per_pixel = (p.sample_count + p.sample_stride - 1) / p.sample_stride;
    std::vector<int> sizes;
    int forced = std::min(p.sample_ranges, RTNW_MAX_CHUNKS);  // rtnw_render_params.sample_ranges: 0 = the schedule below
#ifdef RTNW_TUNING  // A/B builds only
    if (const char* e = getenv("RTNW_SAMPLE_CHUNKS")) forced = std::min(atoi(e), RTNW_MAX_CHUNKS);
#endif
    if (forced <= 0) {
        const int base = std::max(4, (per_pixel + 27) / 28);
        int rest = per_pixel;
        while (rest - base >= 8) { sizes.push_back(base); rest -= base; }
        while (rest > 0) { const int sz = std::max(1, rest / 2); sizes.push_back(sz); rest -= sz; }
    } else {  // equal ranges
        const int c = std::max(1, std::min(forced, per_pixel));
        for (int q = 0; q < c; ++q) sizes.push_back((int)((long long)(q + 1) * per_pixel / c - (long long)q * per_pixel / c));
    }
    a.chunks = (int)sizes.size();
    a.chunk_total = std::max(1, per_pixel);
    a.chunk_cum[0] = 0;
    for (int q = 0; q < a.chunks; ++q) a.chunk_cum[q + 1] = a.chunk_cum[q] + sizes[q];
}

int validate_params(const rtnw_render_params* p) {
    if (!p) return fail(RTNW_ERR_INVALID, "null render params");
    if (p->nx <= 0 || p->ny <= 0 || (long long)p->nx * p->ny > 0x7fffffffLL / 4) return fail(RTNW_ERR_INVALID, "bad image size");
    if (p->sample_count <= 0 || p->sample_stride <= 0 || p->sample_begin < 0) return fail(RTNW_ERR_INVALID, "bad sample range");
    if (p->max_depth < 0) return fail(RTNW_ERR_INVALID, "bad max_depth");
    if (p->background > RTNW_BG_SKY) return fail(RTNW_ERR_INVALID, "bad background");
    if (p->sample_ranges < 0) return fail(RTNW_ERR_INVALID, "bad sample_ranges");
    if (p->pixel_count < 0 || (p->pixel_count > 0 && (p->pixel_begin < 0 || p->pixel_stride < 1 ||
        (long long)p->pixel_begin + (long long)(p->pixel_count - 1) * p->pixel_stride >= (long long)p->nx * p->ny)))
        return fail(RTNW_ERR_INVALID, "bad pixel subset");
    return RTNW_OK;
}

// A render in two halves, so that one host thread can keep several devices busy (rtnw_render_multi): render_launch queues
// everything on stream st and returns; render_finish waits for it and fills stats (kernel_ms from CUDA events on st).
struct render_ticket {
    int chunks = 1;
    rtnw_render_params p;  // with the pixel subset filled in
    cudaStream_t st = nullptr;
};

int render_launch(rtnw_ctx* ctx, const rtnw_scene* scene, const rtnw_camera* cam, const rtnw_render_params* p, float* accum_dev,
                  cudaStream_t st, render_ticket* ticket) {
    render_args a;
    a.S = scene->view;
    a.cam = *cam;
    a.p = *p;
    if (a.p.pixel_count == 0) { a.p.pixel_begin = 0; a.p.pixel_stride = 1; a.p.pixel_count = p->nx * p->ny; }
    a.accum = accum_dev;
    a.ctr = ctx->ctr;
    int rc = RTNW_OK;
    pick_chunks(a.p, a);
    a.fixed = nullptr;
    const size_t plane = (size_t)p->nx * p->ny * 3;
    if (a.chunks > 1) {
        if (ctx->fixed_words < plane) {
            CUDA_TRY(cudaStreamSynchronize(st));
            rc = grow(&ctx->fixed, &ctx->fixed_words, plane, "cudaMalloc of the sample-range accumulation plane failed");
            if (rc != RTNW_OK) return rc;
            CUDA_TRY(cudaMemsetAsync(ctx->fixed, 0, plane * sizeof(unsigned long long), st));  // k_finish_fixed keeps it zero afterwards
        }
        a.fixed = ctx->fixed;
    }
    CUDA_TRY(cudaMemsetAsync(ctx->ctr, 0, 8 * sizeof(unsigned long long), st));
    CUDA_TRY(cudaEventRecord(ctx->ev0, st));
    rc = by_variant(p->flags, [&](auto count, auto fast) { return launch_render<decltype(count)::value, decltype(fast)::value>(ctx, a, st); });
    if (rc != RTNW_OK) return rc;
    if (a.chunks > 1) {
        k_finish_fixed<<<(a.p.pixel_count + 255) / 256, 256, 0, st>>>(a.fixed, a.p.pixel_begin, a.p.pixel_stride, a.p.pixel_count,
                                                                      (p->flags & RTNW_F_ACCUMULATE) ? 1 : 0, accum_dev);
        CUDA_TRY(cudaGetLastError());
    }
    CUDA_TRY(cudaEventRecord(ctx->ev1, st));
    CUDA_TRY(cudaMemcpyAsync(ctx->ctr_host, ctx->ctr, 8 * sizeof(unsigned long long), cudaMemcpyDeviceToHost, st));  // pinned: truly asynchronous
    ticket->chunks = a.chunks;
    ticket->p = a.p;
    ticket->st = st;
    return RTNW_OK;
}

uint64_t paths_of(const rtnw_render_params& p) {  // p: pixel subset filled in
    if (!(p.flags & RTNW_F_ROTATE_SAMPLES)) return (uint64_t)p.pixel_count * p.sample_count;
    uint64_t paths = 0;  // per pixel: the samples s = (begin - pixel) mod G + k*G below ns
    const int g = p.sample_stride;
    auto floordiv = [](long long x, long long y) { return x >= 0 ? x / y : -((-x + y - 1) / y); };
    for (int r = 0; r < g; ++r) {  // pixels whose index is r mod G
        const int b = ((p.sample_begin - r) % g + g) % g;
        const uint64_t per_pixel = b < p.sample_count ? (uint64_t)(p.sample_count - b + g - 1) / g : 0;
        uint64_t n_pix = 0;
        if (p.pixel_stride == 1) {  // integers in [begin, begin+count) congruent to r
            const long long lo = p.pixel_begin, hi = (long long)p.pixel_begin + p.pixel_count - 1;
            n_pix = (uint64_t)(floordiv(hi - r, g) - floordiv(lo - 1 - r, g));
        } else {
            for (long long k = 0; k < p.pixel_count; ++k) n_pix += ((p.pixel_begin + k * p.pixel_stride) % g) == r;
        }
        paths += per_pixel * n_pix;
    }
    return paths;
}

int render_finish(rtnw_ctx* ctx, const render_ticket& t, rtnw_stats* stats) {
    CUDA_TRY(cudaStreamSynchronize(t.st));
#ifdef RTNW_ROUND_STATS
    {
        unsigned long long rs[32];
        cudaMemcpyFromSymbol(rs, g_round_stats, sizeof rs);
        fprintf(stderr, "round_stats rounds %llu take/round %.1f drain/round %.1f n/round %.1f queued/round %.1f pure_gate_rounds %.3f busy<=64 %.3f <=128 %.3f <=192 %.3f >192 %.3f | "
                        "ray_rounds %llu rounds/ray_round %.1f cycles: hit %.3f (bvh items %.3f) shade %.3f of total; cycles/round by busy<=64 %.0f <=128 %.0f <=192 %.0f >192 %.0f; cycles/ray_round %.0f\n",
                rs[0], (double)rs[1] / rs[0], (double)rs[2] / rs[0], (double)rs[8] / rs[0], (double)rs[9] / rs[0], (double)rs[3] / rs[0],
                (double)rs[4] / rs[0], (double)rs[5] / rs[0], (double)rs[6] / rs[0], (double)rs[7] / rs[0], rs[10], (double)rs[0] / rs[10],
                (double)rs[11] / rs[12], (double)rs[14] / rs[12], (double)rs[13] / rs[12], (double)rs[15] / (rs[4] + 1), (double)rs[16] / (rs[5] + 1),
                (double)rs[17] / (rs[6] + 1), (double)rs[18] / (rs[7] + 1), (double)rs[12] / rs[10]);
        fprintf(stderr, "round_stats small: work<=32 %.3f of rounds, %.0f cycles each, %.3f of bvh cycles; work 33..64 %.3f of rounds, %.0f cycles each, %.3f of bvh cycles\n",
                (double)rs[19] / rs[0], (double)rs[20] / (rs[19] + 1), (double)rs[20] / rs[14], (double)rs[21] / rs[0], (double)rs[22] / (rs[21] + 1), (double)rs[22] / rs[14]);
        unsigned long long z[32] = {0};
        cudaMemcpyToSymbol(g_round_stats, z, sizeof z);
    }
#endif
    const int rc = check_task_stack(ctx);
    if (rc != RTNW_OK || !stats) return rc;
    const unsigned long long* h = ctx->ctr_host;
    rtnw_stats s = {};
    s.paths = paths_of(t.p);
    s.rays = h[1];
    s.box_tests = h[2];
    s.prim_tests = h[3];
    s.kernel_launches = t.chunks > 1 ? 2 : 1;
    s.sample_ranges = t.chunks;
    return report_stats(ctx, stats, s, false);
}

// render into a device buffer on stream st, synchronously
int render_core(rtnw_ctx* ctx, const rtnw_scene* scene, const rtnw_camera* cam, const rtnw_render_params* p, float* accum_dev,
                cudaStream_t st, rtnw_stats* stats) {
    render_ticket t;
    const int rc = render_launch(ctx, scene, cam, p, accum_dev, st, &t);
    if (rc != RTNW_OK) return rc;
    return render_finish(ctx, t, stats);
}

}  // namespace

extern "C" {

const char* rtnw_last_error(void) { return g_err.c_str(); }
int rtnw_abi_version(void) { return RTNW_ABI_VERSION; }

int rtnw_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
    int ok = 0;
    for (int i = 0; i < n; ++i) {
        int major = 0;
        if (cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, i) == cudaSuccess && major == 10) ++ok;
    }
    return ok;
}

int rtnw_ctx_create(int device, rtnw_ctx** out) {
    if (!out) return fail(RTNW_ERR_INVALID, "null out pointer");
    *out = nullptr;
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess || n == 0) {
        cudaGetLastError();
        return fail(RTNW_ERR_CUDA, "no CUDA device: this library has no CPU fallback");
    }
    if (device < 0 || device >= n) return fail(RTNW_ERR_INVALID, "device index out of range");
    int major = 0;
    CUDA_TRY(cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, device));
    if (major != 10) return fail(RTNW_ERR_CUDA, "device is not sm_100 (the library is built for sm_100a only)");
    CUDA_TRY(cudaSetDevice(device));
    rtnw_ctx* c = new rtnw_ctx();
    c->device = device;
    cudaDeviceGetAttribute(&c->sm_count, cudaDevAttrMultiProcessorCount, device);
    cudaDeviceGetAttribute(&c->clock_khz, cudaDevAttrClockRate, device);
    cudaDeviceGetAttribute(&c->smem_optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, device);
    cudaDeviceGetAttribute(&c->l2_bytes, cudaDevAttrL2CacheSize, device);
    // a BLOCKING stream: ordered with the legacy default stream (torch's default), so a caller's fills / reduces on stream 0
    // and the library's own launches cannot overtake each other
    cudaError_t e = cudaStreamCreateWithFlags(&c->stream, cudaStreamDefault);
    if (e == cudaSuccess) e = cudaEventCreate(&c->ev0);
    if (e == cudaSuccess) e = cudaEventCreate(&c->ev1);
    if (e == cudaSuccess) e = cudaEventCreate(&c->ev_t0);
    if (e == cudaSuccess) e = cudaEventCreate(&c->ev_t1);
    if (e == cudaSuccess) e = cudaMalloc(&c->ctr, 8 * sizeof(unsigned long long));
    if (e == cudaSuccess) e = cudaHostAlloc(&c->ctr_host, 8 * sizeof(unsigned long long), cudaHostAllocDefault);
    if (e != cudaSuccess) {
        rtnw_ctx_destroy(c);
        return fail(RTNW_ERR_CUDA, std::string("context setup: ") + cudaGetErrorString(e));
    }
    *out = c;
    return RTNW_OK;
}

int rtnw_ctx_destroy(rtnw_ctx* c) {
    if (!c) return RTNW_OK;
    cudaSetDevice(c->device);
    if (c->accum) cudaFree(c->accum);
    if (c->fixed) cudaFree(c->fixed);
    for (int q = 0; q < 2; ++q) if (c->spare_slab[q]) cudaFree(c->spare_slab[q]);
    if (c->ctr) cudaFree(c->ctr);
    if (c->ctr_host) cudaFreeHost(c->ctr_host);
    if (c->ev_t0) cudaEventDestroy(c->ev_t0);
    if (c->ev_t1) cudaEventDestroy(c->ev_t1);
    if (c->ev0) cudaEventDestroy(c->ev0);
    if (c->ev1) cudaEventDestroy(c->ev1);
    if (c->stream) cudaStreamDestroy(c->stream);
    delete c;
    return RTNW_OK;
}

int rtnw_ctx_info(rtnw_ctx* ctx, int32_t* sm_count, int32_t* clock_khz, int32_t* smem_optin, int32_t* l2_bytes) {
    if (!ctx) return fail(RTNW_ERR_INVALID, "null context");
    if (sm_count) *sm_count = ctx->sm_count;
    if (clock_khz) *clock_khz = ctx->clock_khz;
    if (smem_optin) *smem_optin = ctx->smem_optin;
    if (l2_bytes) *l2_bytes = ctx->l2_bytes;
    return RTNW_OK;
}

int rtnw_measure_fp32_peak(rtnw_ctx* ctx, float* tflops) {
    int rc = check_ctx(ctx);
    if (rc != RTNW_OK) return rc;
    if (!tflops) return fail(RTNW_ERR_INVALID, "null argument");
    staging g;
    const int sink = g.add(sizeof(float));
    CUDA_TRY(g.copy_in(ctx->stream));
    const int iters = 1 << 14, blocks = ctx->sm_count * 32;
    float best = 0.f;
    for (int rep = 0; rep < 4; ++rep) {  // first repetition warms the clocks up
        CUDA_TRY(cudaEventRecord(ctx->ev0, ctx->stream));
        k_fma_peak<<<blocks, 256, 0, ctx->stream>>>(g.at<float>(sink), iters);
        CUDA_TRY(cudaEventRecord(ctx->ev1, ctx->stream));
        CUDA_TRY(cudaStreamSynchronize(ctx->stream));
        float ms = 0.f;
        CUDA_TRY(cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev1));
        const float tf = 2.0f * 8.0f * (float)iters * 256.0f * (float)blocks / (ms * 1e-3f) / 1e12f;
        if (rep > 0 && tf > best) best = tf;
    }
    *tflops = best;
    return RTNW_OK;
}

int rtnw_selftest_recip(rtnw_ctx* ctx, uint64_t n, uint32_t seed, uint64_t out[6]) {
    int rc = check_ctx(ctx);
    if (rc != RTNW_OK) return rc;
    if (!out) return fail(RTNW_ERR_INVALID, "null argument");
    staging g;
    const int counts = g.add(6 * sizeof(unsigned long long), nullptr, out);
    CUDA_TRY(g.copy_in(ctx->stream));
    CUDA_TRY(cudaMemsetAsync(g.at<void>(counts), 0, 6 * sizeof(unsigned long long), ctx->stream));
    k_selftest_recip<<<ctx->sm_count * 8, 256, 0, ctx->stream>>>(n, seed, g.at<unsigned long long>(counts));
    CUDA_TRY(cudaGetLastError());
    CUDA_TRY(g.copy_out(ctx->stream));
    return RTNW_OK;
}

int64_t rtnw_scene_inspect(const rtnw_scene_desc* desc, int32_t table, void* buf, size_t cap_bytes) {
    if (!desc) return fail(RTNW_ERR_INVALID, "null scene_desc");
    stream_builder sb(*desc);
    if (!sb.run()) return fail(RTNW_ERR_INVALID, "scene_desc: " + sb.err);
    const void* src = nullptr;
    size_t bytes = 0;
    switch (table) {
        case 0: src = sb.recs.data(); bytes = sb.recs.size() * sizeof(rec); break;
        case 1: src = sb.leaf.data(); bytes = sb.leaf.size() * sizeof(int32_t); break;
        case 2: src = sb.gate_leaves.data(); bytes = sb.gate_leaves.size() * sizeof(int2); break;
        case 3: src = sb.wnodes.data(); bytes = sb.wnodes.size() * sizeof(float4); break;
        default: return fail(RTNW_ERR_INVALID, "unknown table");
    }
    if (buf && cap_bytes) std::memcpy(buf, src, std::min(cap_bytes, bytes));
    return (int64_t)bytes;
}

// The device image of a scene, built once on the host (no device needed): one slab with every table at a 256-byte
// aligned offset, in pinned memory when a CUDA driver is present (so an upload is a single asynchronous DMA).
enum prepared_table { T_RECS, T_LEAF, T_RXF, T_NODES, T_GATES, T_XF, T_MAT, T_TEX, T_RV, T_PERM, T_IMG, N_TABLES };
struct rtnw_prepared {
    uint8_t* host = nullptr;
    bool pinned = false;
    size_t bytes = 0;
    size_t off[N_TABLES] = {};  // byte offset of each table in the slab
    int32_t n_recs = 0, n_materials = 0, n_textures = 0, n_wnodes = 0, fast_node_base = 0;
};

int rtnw_prepared_free(rtnw_prepared* p) {
    if (!p) return RTNW_OK;
    if (p->host) { if (p->pinned) cudaFreeHost(p->host); else std::free(p->host); }
    delete p;
    return RTNW_OK;
}

int rtnw_scene_prepare(const rtnw_scene_desc* desc, rtnw_prepared** out) {
    if (!out) return fail(RTNW_ERR_INVALID, "null out pointer");
    *out = nullptr;
    if (!desc) return fail(RTNW_ERR_INVALID, "null scene_desc");
    stream_builder sb(*desc);
    if (!sb.run()) return fail(RTNW_ERR_INVALID, "scene_desc: " + sb.err);

    // perlin tables repacked for 128-bit gradient loads and byte permutations
    std::vector<float4> ranvec(256);
    std::vector<uint8_t> perm(768);
    for (int i = 0; i < 256; ++i) {
        ranvec[i] = make_float4(desc->perlin_ranvec[3 * i], desc->perlin_ranvec[3 * i + 1], desc->perlin_ranvec[3 * i + 2], 0.f);
        const int32_t px = desc->perlin_perm_x[i], py = desc->perlin_perm_y[i], pz = desc->perlin_perm_z[i];
        if ((px | py | pz) & ~255) return fail(RTNW_ERR_INVALID, "scene_desc: perlin permutation entry outside 0..255");
        perm[i] = (uint8_t)px; perm[256 + i] = (uint8_t)py; perm[512 + i] = (uint8_t)pz;
    }

    // one slab, every table 256-byte aligned; the image table has 16 bytes of slack after the pool
    const void* src[N_TABLES] = {sb.recs.data(), sb.leaf.data(), sb.rec_xf.data(), sb.wnodes.data(), sb.gate_leaves.data(),
                                 desc->xforms, desc->materials, desc->textures, ranvec.data(), perm.data(), desc->images};
    const size_t sz[N_TABLES] = {sb.recs.size() * sizeof(rec), sb.leaf.size() * sizeof(int32_t), sb.rec_xf.size() * sizeof(uint32_t),
                                 sb.wnodes.size() * sizeof(float4), sb.gate_leaves.size() * sizeof(int2),
                                 (size_t)desc->n_xform_ops * sizeof(rtnw_xform_op), (size_t)desc->n_materials * sizeof(rtnw_material),
                                 (size_t)desc->n_textures * sizeof(rtnw_texture), 256 * sizeof(float4), 768, (size_t)desc->image_bytes + 16};
    rtnw_prepared* P = new rtnw_prepared();
    P->bytes = layout256(sz, N_TABLES, P->off);
    void* pin = nullptr;
    if (cudaHostAlloc(&pin, P->bytes, cudaHostAllocDefault) == cudaSuccess) { P->host = static_cast<uint8_t*>(pin); P->pinned = true; }
    else { cudaGetLastError(); P->host = static_cast<uint8_t*>(std::malloc(P->bytes)); }
    if (!P->host) { delete P; return fail(RTNW_ERR_NOMEM, "cannot allocate the host image of the scene"); }
    std::memset(P->host, 0, P->bytes);
    for (int t = 0; t < N_TABLES; ++t) {
        const size_t bytes = t == T_IMG ? (size_t)desc->image_bytes : sz[t];
        if (bytes) std::memcpy(P->host + P->off[t], src[t], bytes);
    }
    P->n_recs = (int32_t)sb.recs.size();
    P->n_wnodes = (int32_t)(sb.wnodes.size() / 8);
    P->fast_node_base = sb.fast_base;
    P->n_materials = desc->n_materials;
    P->n_textures = desc->n_textures;
    *out = P;
    return RTNW_OK;
}

int64_t rtnw_prepared_bytes(const rtnw_prepared* p) { return p ? (int64_t)p->bytes : 0; }

int rtnw_scene_upload_prepared(rtnw_ctx* ctx, const rtnw_prepared* P, rtnw_scene** out) {
    if (!out) return fail(RTNW_ERR_INVALID, "null out pointer");
    *out = nullptr;
    if (!P) return fail(RTNW_ERR_INVALID, "null prepared scene");
    int rc = check_ctx(ctx);
    if (rc != RTNW_OK) return rc;
    const size_t off = P->bytes;
    rtnw_scene* s = new rtnw_scene();
    cudaError_t e = cudaSuccess;
    for (int q = 0; q < 2 && !s->slab; ++q)
        if (ctx->spare_slab[q] && ctx->spare_bytes[q] >= off) {
            s->slab = ctx->spare_slab[q];
            s->slab_bytes = ctx->spare_bytes[q];
            ctx->spare_slab[q] = nullptr;
            ctx->spare_bytes[q] = 0;
        }
    if (!s->slab) {
        e = cudaMalloc(&s->slab, off);
        s->slab_bytes = off;
    }
    // stream-ordered: the next render on this context's stream (or a stream ordered after it) sees the tables
    if (e == cudaSuccess) e = cudaMemcpyAsync(s->slab, P->host, off, cudaMemcpyHostToDevice, ctx->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
    if (e != cudaSuccess) {
        if (s->slab) cudaFree(s->slab);
        delete s;
        return fail(e == cudaErrorMemoryAllocation ? RTNW_ERR_NOMEM : RTNW_ERR_CUDA, std::string("scene upload: ") + cudaGetErrorString(e));
    }
    uint8_t* base = static_cast<uint8_t*>(s->slab);
    const size_t* o = P->off;
    s->view.recs = reinterpret_cast<const rec*>(base + o[T_RECS]);
    s->view.rec_leaf = reinterpret_cast<const int32_t*>(base + o[T_LEAF]);
    s->view.rec_xf = reinterpret_cast<const uint32_t*>(base + o[T_RXF]);
    s->view.wnodes = reinterpret_cast<const float4*>(base + o[T_NODES]);
    s->view.gates = reinterpret_cast<const int2*>(base + o[T_GATES]);
    s->view.xforms = reinterpret_cast<const rtnw_xform_op*>(base + o[T_XF]);
    s->view.materials = reinterpret_cast<const rtnw_material*>(base + o[T_MAT]);
    s->view.textures = reinterpret_cast<const rtnw_texture*>(base + o[T_TEX]);
    s->view.ranvec = reinterpret_cast<const float4*>(base + o[T_RV]);
    s->view.perm = base + o[T_PERM];
    s->view.images = base + o[T_IMG];
    s->view.n_recs = P->n_recs;
    s->view.n_wnodes = P->n_wnodes;
    s->view.fast_node_base = P->fast_node_base;
    s->view.n_materials = P->n_materials;
    s->view.n_textures = P->n_textures;
    *out = s;
    return RTNW_OK;
}

int rtnw_scene_upload(rtnw_ctx* ctx, const rtnw_scene_desc* desc, rtnw_scene** out) {
    if (!out) return fail(RTNW_ERR_INVALID, "null out pointer");
    *out = nullptr;
    int rc = check_ctx(ctx);
    if (rc != RTNW_OK) return rc;
    rtnw_prepared* P = nullptr;
    if ((rc = rtnw_scene_prepare(desc, &P)) != RTNW_OK) return rc;
    rc = rtnw_scene_upload_prepared(ctx, P, out);
    const std::string msg = g_err;
    rtnw_prepared_free(P);
    return rc == RTNW_OK ? RTNW_OK : fail(rc, msg);
}

int rtnw_scene_free(rtnw_ctx* ctx, rtnw_scene* scene) {
    if (!scene) return RTNW_OK;
    if (ctx) {
        cudaSetDevice(ctx->device);
        for (int q = 0; q < 2 && scene->slab; ++q)
            if (!ctx->spare_slab[q]) {
                ctx->spare_slab[q] = scene->slab;
                ctx->spare_bytes[q] = scene->slab_bytes;
                scene->slab = nullptr;
            }
    }
    if (scene->slab) cudaFree(scene->slab);
    delete scene;
    return RTNW_OK;
}

int rtnw_render_device(rtnw_ctx* ctx, const rtnw_scene* scene, const rtnw_camera* cam, const rtnw_render_params* params,
                       float* accum_rgb_dev, void* cuda_stream, rtnw_stats* stats) {
    int rc = check_ctx(ctx);
    if (rc != RTNW_OK) return rc;
    if (!scene || !cam || !accum_rgb_dev) return fail(RTNW_ERR_INVALID, "null argument");
    if ((rc = validate_params(params)) != RTNW_OK) return rc;
    cudaStream_t st = cuda_stream ? static_cast<cudaStream_t>(cuda_stream) : cudaStreamLegacy;  // NULL = the legacy default stream
    return render_core(ctx, scene, cam, params, accum_rgb_dev, st, stats);
}

int rtnw_render(rtnw_ctx* ctx, const rtnw_scene* scene, const rtnw_camera* cam, const rtnw_render_params* params,
                float* accum_rgb, rtnw_stats* stats) {
    int rc = check_ctx(ctx);
    if (rc != RTNW_OK) return rc;
    if (!scene || !cam || !accum_rgb) return fail(RTNW_ERR_INVALID, "null argument");
    if ((rc = validate_params(params)) != RTNW_OK) return rc;
    if (params->pixel_count != 0 || (params->flags & RTNW_F_ACCUMULATE))
        return fail(RTNW_ERR_INVALID, "pixel subsets / RTNW_F_ACCUMULATE need rtnw_render_device (the host entry point returns whole images)");
    const size_t floats = (size_t)params->nx * params->ny * 3;
    if ((rc = grow(&ctx->accum, &ctx->accum_floats, floats, "cannot allocate the accumulation buffer")) != RTNW_OK) return rc;
    CUDA_TRY(cudaEventRecord(ctx->ev_t0, ctx->stream));
    rc = render_core(ctx, scene, cam, params, ctx->accum, ctx->stream, stats);
    if (rc != RTNW_OK) return rc;
    CUDA_TRY(cudaMemcpyAsync(accum_rgb, ctx->accum, floats * sizeof(float), cudaMemcpyDeviceToHost, ctx->stream));
    CUDA_TRY(cudaEventRecord(ctx->ev_t1, ctx->stream));
    CUDA_TRY(cudaStreamSynchronize(ctx->stream));
    if (stats) CUDA_TRY(cudaEventElapsedTime(&stats->total_ms, ctx->ev_t0, ctx->ev_t1));
    return RTNW_OK;
}

int rtnw_plan_sample_ranges(const rtnw_render_params* params, int32_t* cum, int32_t cap) {
    const int rc = validate_params(params);
    if (rc != RTNW_OK) return rc;
    if (!cum || cap < 1) return fail(RTNW_ERR_INVALID, "null / empty output");
    render_args a;
    pick_chunks(*params, a);
    if (a.chunks > cap) return fail(RTNW_ERR_INVALID, "cap is smaller than the number of sample ranges");
    for (int q = 0; q <= a.chunks; ++q) cum[q] = a.chunk_cum[q];
    return a.chunks;
}

int rtnw_quantize_device(rtnw_ctx* ctx, const float* accum_rgb_dev, int32_t nx, int32_t ny, int32_t ns, int32_t clamp255, int32_t* rgb_out) {
    int rc = check_ctx(ctx);
    if (rc != RTNW_OK) return rc;
    if (!accum_rgb_dev || !rgb_out || nx <= 0 || ny <= 0 || ns <= 0) return fail(RTNW_ERR_INVALID, "bad quantize arguments");
    const size_t n = (size_t)nx * ny;
    staging g;  // the input is the caller's device buffer
    const int rgb = g.add(n * 3 * sizeof(int32_t), nullptr, rgb_out);
    CUDA_TRY(g.copy_in(ctx->stream));
    const float inv_ns = (float)(1.0 / (double)(float)ns);
    k_quantize<<<(unsigned)((n + 255) / 256), 256, 0, ctx->stream>>>(accum_rgb_dev, nx, ny, inv_ns, clamp255, g.at<int32_t>(rgb));
    CUDA_TRY(cudaGetLastError());
    CUDA_TRY(g.copy_out(ctx->stream));
    return RTNW_OK;
}

int rtnw_trace(rtnw_ctx* ctx, const rtnw_scene* scene, const rtnw_ray* rays, size_t n, float t_min, float t_max, uint32_t flags,
               uint64_t seed, rtnw_hit* out) {
    int rc = check_ctx(ctx);
    if (rc != RTNW_OK) return rc;
    if (!scene || (n && (!rays || !out))) return fail(RTNW_ERR_INVALID, "null argument");
    if (n == 0) return RTNW_OK;
    staging g;
    const int in = g.add(n * sizeof(rtnw_ray), rays), hit = g.add(n * sizeof(rtnw_hit), nullptr, out);
    CUDA_TRY(g.copy_in(ctx->stream));
    const unsigned grid = (unsigned)((n + RTNW_BLOCK - 1) / RTNW_BLOCK);
    rc = by_variant(flags, [&](auto, auto fast) {
        constexpr bool FAST = decltype(fast)::value;
        return launch_coop<block_smem<FAST>>(k_trace<FAST>, grid, ctx->stream, scene->view, g.at<const rtnw_ray>(in), n, t_min, t_max,
                                             seed, g.at<rtnw_hit>(hit));
    });
    if (rc != RTNW_OK) return rc;
    CUDA_TRY(g.copy_out(ctx->stream));
    return RTNW_OK;
}

int rtnw_render_aov(rtnw_ctx* ctx, const rtnw_scene* scene, const rtnw_camera* cam, const rtnw_render_params* params,
                    const rtnw_aov* out, rtnw_stats* stats) {
    int rc = check_ctx(ctx);
    if (rc != RTNW_OK) return rc;
    if (!scene || !cam || !out || !out->albedo || !out->normal || !out->depth || !out->hits || !out->prim_id)
        return fail(RTNW_ERR_INVALID, "null argument");
    if ((rc = validate_params(params)) != RTNW_OK) return rc;
    if (params->pixel_count != 0 || (params->flags & (RTNW_F_ACCUMULATE | RTNW_F_ROTATE_SAMPLES)))
        return fail(RTNW_ERR_INVALID, "rtnw_render_aov covers whole images: no pixel subset, RTNW_F_ACCUMULATE or RTNW_F_ROTATE_SAMPLES");
    const size_t n = (size_t)params->nx * params->ny;
    staging g;
    const int albedo = g.add(n * 3 * sizeof(float), nullptr, out->albedo), normal = g.add(n * 3 * sizeof(float), nullptr, out->normal);
    const int depth = g.add(n * sizeof(float), nullptr, out->depth), hits = g.add(n * sizeof(int32_t), nullptr, out->hits);
    const int prim_id = g.add(n * sizeof(int32_t), nullptr, out->prim_id);
    CUDA_TRY(g.copy_in(ctx->stream, ctx->ev_t0));
    aov_args a;
    a.S = scene->view;
    a.cam = *cam;
    a.p = *params;
    a.albedo = g.at<float>(albedo);
    a.normal = g.at<float>(normal);
    a.depth = g.at<float>(depth);
    a.hits = g.at<int32_t>(hits);
    a.prim_id = g.at<int32_t>(prim_id);
    a.ctr = ctx->ctr;
    const unsigned grid = (unsigned)((n + RTNW_BLOCK - 1) / RTNW_BLOCK);
    CUDA_TRY(cudaMemsetAsync(ctx->ctr, 0, 8 * sizeof(unsigned long long), ctx->stream));
    CUDA_TRY(cudaEventRecord(ctx->ev0, ctx->stream));
    rc = by_variant(params->flags, [&](auto, auto fast) {
        constexpr bool FAST = decltype(fast)::value;
        return launch_coop<aov_smem<FAST>>(k_aov<FAST>, grid, ctx->stream, a);
    });
    if (rc != RTNW_OK) return rc;
    CUDA_TRY(cudaEventRecord(ctx->ev1, ctx->stream));
    CUDA_TRY(cudaMemcpyAsync(ctx->ctr_host, ctx->ctr, 8 * sizeof(unsigned long long), cudaMemcpyDeviceToHost, ctx->stream));
    CUDA_TRY(g.copy_out(ctx->stream, ctx->ev_t1));
    if ((rc = check_task_stack(ctx)) != RTNW_OK) return rc;
    rtnw_stats s = {};
    s.paths = s.rays = (uint64_t)n * params->sample_count;
    s.kernel_launches = 1;
    s.sample_ranges = 1;
    return report_stats(ctx, stats, s, true);
}

int rtnw_eval_texture(rtnw_ctx* ctx, const rtnw_scene* scene, int32_t tex_id, const float* uvp, size_t n, float* rgb_out) {
    int rc = check_ctx(ctx);
    if (rc != RTNW_OK) return rc;
    if (!scene || (n && (!uvp || !rgb_out))) return fail(RTNW_ERR_INVALID, "null argument");
    if (tex_id < 0 || tex_id >= scene->view.n_textures) return fail(RTNW_ERR_INVALID, "texture index out of range");
    if (n == 0) return RTNW_OK;
    staging g;
    const int in = g.add(n * 5 * sizeof(float), uvp), rgb = g.add(n * 3 * sizeof(float), nullptr, rgb_out);
    CUDA_TRY(g.copy_in(ctx->stream));
    k_eval_texture<<<(unsigned)((n + 127) / 128), 128, 0, ctx->stream>>>(scene->view, tex_id, g.at<float>(in), n, g.at<float>(rgb));
    CUDA_TRY(cudaGetLastError());
    CUDA_TRY(g.copy_out(ctx->stream));
    return RTNW_OK;
}

int rtnw_denoise(rtnw_ctx* ctx, const float* color_sums, const rtnw_aov* features, int32_t nx, int32_t ny, int32_t ns,
                 const rtnw_denoise_params* dp, float* rgb_out, rtnw_stats* stats) {
    int rc = check_ctx(ctx);
    if (rc != RTNW_OK) return rc;
    if (!color_sums || !features || !features->albedo || !features->normal || !features->depth || !features->hits || !dp || !rgb_out)
        return fail(RTNW_ERR_INVALID, "null argument");
    if (nx <= 0 || ny <= 0 || (long long)nx * ny > 0x7fffffffLL / 4 || ns <= 0) return fail(RTNW_ERR_INVALID, "bad image size or sample count");
    if (dp->iterations < 1 || dp->iterations > 8) return fail(RTNW_ERR_INVALID, "iterations must be 1..8");
    if (dp->normal_power_log2 < 0 || dp->normal_power_log2 > 10) return fail(RTNW_ERR_INVALID, "normal_power_log2 must be 0..10");
    if (!(dp->sigma_luminance > 0.f) || !std::isfinite(dp->sigma_luminance) || !(dp->sigma_depth > 0.f) || !std::isfinite(dp->sigma_depth))
        return fail(RTNW_ERR_INVALID, "sigmas must be finite and > 0");
    const size_t n = (size_t)nx * ny;
    staging g;  // 101 bytes per pixel; the colour span is overwritten with the output
    const int color = g.add(12 * n, color_sums, rgb_out), albedo = g.add(12 * n, features->albedo), normal = g.add(12 * n, features->normal);
    const int depth = g.add(4 * n, features->depth), hits = g.add(4 * n, features->hits);
    const int ev0 = g.add(16 * n), ev1 = g.add(16 * n), feat = g.add(16 * n), grad = g.add(8 * n), hit = g.add(n);
    CUDA_TRY(g.copy_in(ctx->stream, ctx->ev_t0));
    dn_args a;
    a.nx = nx; a.ny = ny; a.k = dp->normal_power_log2;
    a.fns = (float)ns; a.sigma_l = dp->sigma_luminance; a.sigma_z = dp->sigma_depth;
    a.color = a.out = g.at<float>(color);
    a.albedo = g.at<float>(albedo);
    a.normal = g.at<float>(normal);
    a.depth = g.at<float>(depth);
    a.hits = g.at<int32_t>(hits);
    a.ev[0] = g.at<float4>(ev0);
    a.ev[1] = g.at<float4>(ev1);
    a.feat = g.at<float4>(feat);
    a.grad = g.at<float2>(grad);
    a.hit = g.at<unsigned char>(hit);
    const dim3 block(DN_BX, DN_BY), grid((unsigned)((nx + DN_BX - 1) / DN_BX), (unsigned)((ny + DN_BY - 1) / DN_BY));
    CUDA_TRY(cudaEventRecord(ctx->ev0, ctx->stream));
    k_dn_prepare<<<grid, block, 0, ctx->stream>>>(a);
    k_dn_variance<<<grid, block, 0, ctx->stream>>>(a);
    for (int it = 0; it < dp->iterations; ++it)  // k_dn_variance left (e, var) in ev[1]
        k_dn_atrous<<<grid, block, 0, ctx->stream>>>(a, it, it % 2 == 0 ? 1 : 0, it == dp->iterations - 1);
    CUDA_TRY(cudaGetLastError());
    CUDA_TRY(cudaEventRecord(ctx->ev1, ctx->stream));
    CUDA_TRY(g.copy_out(ctx->stream, ctx->ev_t1));
    rtnw_stats s = {};
    s.kernel_launches = dp->iterations + 2;
    return report_stats(ctx, stats, s, true);
}

int rtnw_eval_perlin(rtnw_ctx* ctx, const rtnw_scene* scene, int32_t which, const float* xyz, size_t n, float* out) {
    int rc = check_ctx(ctx);
    if (rc != RTNW_OK) return rc;
    if (!scene || (n && (!xyz || !out))) return fail(RTNW_ERR_INVALID, "null argument");
    if (which != 0 && which != 1) return fail(RTNW_ERR_INVALID, "which must be 0 (noise) or 1 (turb)");
    if (n == 0) return RTNW_OK;
    staging g;
    const int in = g.add(n * 3 * sizeof(float), xyz), val = g.add(n * sizeof(float), nullptr, out);
    CUDA_TRY(g.copy_in(ctx->stream));
    k_eval_perlin<<<(unsigned)((n + 127) / 128), 128, 0, ctx->stream>>>(scene->view, which, g.at<float>(in), n, g.at<float>(val));
    CUDA_TRY(cudaGetLastError());
    CUDA_TRY(g.copy_out(ctx->stream));
    return RTNW_OK;
}

int rtnw_scatter(rtnw_ctx* ctx, const rtnw_scene* scene, const rtnw_ray* rays_in, const rtnw_hit* hits, size_t n, uint64_t seed,
                 rtnw_ray* out_scattered, float* out_atten, float* out_emitted, int32_t* out_flag) {
    int rc = check_ctx(ctx);
    if (rc != RTNW_OK) return rc;
    if (!scene || (n && (!rays_in || !hits || !out_scattered || !out_atten || !out_emitted || !out_flag)))
        return fail(RTNW_ERR_INVALID, "null argument");
    for (size_t i = 0; i < n; ++i)
        if (hits[i].mat_id < 0 || hits[i].mat_id >= scene->view.n_materials) return fail(RTNW_ERR_INVALID, "hit.mat_id out of range");
    if (n == 0) return RTNW_OK;
    staging g;
    const int rays = g.add(n * sizeof(rtnw_ray), rays_in), hit = g.add(n * sizeof(rtnw_hit), hits);
    const int sc = g.add(n * sizeof(rtnw_ray), nullptr, out_scattered), att = g.add(n * 3 * sizeof(float), nullptr, out_atten);
    const int em = g.add(n * 3 * sizeof(float), nullptr, out_emitted), flag = g.add(n * sizeof(int32_t), nullptr, out_flag);
    CUDA_TRY(g.copy_in(ctx->stream));
    k_scatter<<<(unsigned)((n + 127) / 128), 128, 0, ctx->stream>>>(scene->view, g.at<rtnw_ray>(rays), g.at<rtnw_hit>(hit), n, seed,
                                                                    g.at<rtnw_ray>(sc), g.at<float>(att), g.at<float>(em),
                                                                    g.at<int32_t>(flag));
    CUDA_TRY(cudaGetLastError());
    CUDA_TRY(g.copy_out(ctx->stream));
    return RTNW_OK;
}

int rtnw_camera_rays(rtnw_ctx* ctx, const rtnw_camera* cam, int32_t nx, int32_t ny, const int32_t* ij, const int32_t* sample, size_t n,
                     uint64_t seed, rtnw_ray* rays_out) {
    int rc = check_ctx(ctx);
    if (rc != RTNW_OK) return rc;
    if (!cam || nx <= 0 || ny <= 0 || (n && (!ij || !sample || !rays_out))) return fail(RTNW_ERR_INVALID, "bad argument");
    if (n == 0) return RTNW_OK;
    staging g;
    const int pix = g.add(n * 2 * sizeof(int32_t), ij), smp = g.add(n * sizeof(int32_t), sample), ray = g.add(n * sizeof(rtnw_ray), nullptr, rays_out);
    CUDA_TRY(g.copy_in(ctx->stream));
    k_camera_rays<<<(unsigned)((n + 127) / 128), 128, 0, ctx->stream>>>(*cam, nx, ny, g.at<int32_t>(pix), g.at<int32_t>(smp), n, seed,
                                                                        g.at<rtnw_ray>(ray));
    CUDA_TRY(cudaGetLastError());
    CUDA_TRY(g.copy_out(ctx->stream));
    return RTNW_OK;
}

int rtnw_camera_get_rays(rtnw_ctx* ctx, const rtnw_camera* cam, const float* st, size_t n, uint64_t seed, uint32_t key_base,
                         rtnw_ray* rays_out) {
    int rc = check_ctx(ctx);
    if (rc != RTNW_OK) return rc;
    if (!cam || (n && (!st || !rays_out))) return fail(RTNW_ERR_INVALID, "bad argument");
    if (n == 0) return RTNW_OK;
    staging g;
    const int in = g.add(n * 2 * sizeof(float), st), ray = g.add(n * sizeof(rtnw_ray), nullptr, rays_out);
    CUDA_TRY(g.copy_in(ctx->stream));
    k_camera_get_rays<<<(unsigned)((n + 127) / 128), 128, 0, ctx->stream>>>(*cam, g.at<float>(in), n, seed, key_base, g.at<rtnw_ray>(ray));
    CUDA_TRY(cudaGetLastError());
    CUDA_TRY(g.copy_out(ctx->stream));
    return RTNW_OK;
}

// ---- N GPUs of one box behind one handle (SURVEY.md §8b): one host thread, one context + stream per device --------------
struct rtnw_multi {
    int n = 0;
    rtnw_ctx* ctx[RTNW_MAX_DEVICES] = {};
    float* accum[RTNW_MAX_DEVICES] = {};   // per device: nx*ny*3 sums of its share of the samples
    size_t accum_floats[RTNW_MAX_DEVICES] = {};
    cudaEvent_t done[RTNW_MAX_DEVICES] = {};
    bool peer[RTNW_MAX_DEVICES] = {};      // device 0 reads this rank's buffer directly (same device, or P2P over NVLink)
    float* stage = nullptr;                // device 0: copies of the buffers it cannot read directly
    size_t stage_floats = 0;
};
struct rtnw_multi_scene {
    int n = 0;
    rtnw_scene* scene[RTNW_MAX_DEVICES] = {};
};

int rtnw_ctx_destroy_multi(rtnw_multi* m) {
    if (!m) return RTNW_OK;
    for (int d = 0; d < m->n; ++d) {
        if (!m->ctx[d]) continue;
        cudaSetDevice(m->ctx[d]->device);
        if (m->accum[d]) cudaFree(m->accum[d]);
        if (m->done[d]) cudaEventDestroy(m->done[d]);
        if (d == 0 && m->stage) cudaFree(m->stage);
        rtnw_ctx_destroy(m->ctx[d]);
    }
    delete m;
    return RTNW_OK;
}

int rtnw_ctx_create_multi(const int* device_ids, int n, rtnw_multi** out) {
    if (!out) return fail(RTNW_ERR_INVALID, "null out pointer");
    *out = nullptr;
    if (!device_ids || n < 1 || n > RTNW_MAX_DEVICES) return fail(RTNW_ERR_INVALID, "bad device list");
    rtnw_multi* m = new rtnw_multi();
    m->n = n;
    for (int d = 0; d < n; ++d) {
        int rc = rtnw_ctx_create(device_ids[d], &m->ctx[d]);
        if (rc == RTNW_OK && cudaEventCreateWithFlags(&m->done[d], cudaEventDisableTiming) != cudaSuccess) rc = fail(RTNW_ERR_CUDA, "event creation failed");
        if (rc != RTNW_OK) { const std::string msg = g_err; rtnw_ctx_destroy_multi(m); return fail(rc, msg); }
    }
    // device 0 adds the other ranks' buffers: directly over NVLink where peer access exists, else through a staging copy
    const int dev0 = m->ctx[0]->device;
    for (int d = 0; d < n; ++d) {
        const int dev = m->ctx[d]->device;
        if (dev == dev0) { m->peer[d] = true; continue; }
        int can = 0;
        cudaDeviceCanAccessPeer(&can, dev0, dev);
        if (can) {
            cudaSetDevice(dev0);
            const cudaError_t e = cudaDeviceEnablePeerAccess(dev, 0);
            if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled) can = 0;
            cudaGetLastError();
        }
        m->peer[d] = can != 0;
    }
    *out = m;
    return RTNW_OK;
}

int rtnw_multi_device_count(const rtnw_multi* m) { return m ? m->n : 0; }

int rtnw_scene_free_multi(rtnw_multi* m, rtnw_multi_scene* ms) {
    if (!ms) return RTNW_OK;
    for (int d = 0; d < ms->n; ++d)
        if (ms->scene[d]) rtnw_scene_free(m && d < m->n ? m->ctx[d] : nullptr, ms->scene[d]);
    delete ms;
    return RTNW_OK;
}

int rtnw_scene_upload_multi(rtnw_multi* m, const rtnw_scene_desc* desc, rtnw_multi_scene** out) {
    if (!out) return fail(RTNW_ERR_INVALID, "null out pointer");
    *out = nullptr;
    if (!m) return fail(RTNW_ERR_INVALID, "null context");
    rtnw_prepared* P = nullptr;  // the device image is built once, then copied to every device
    int rc = rtnw_scene_prepare(desc, &P);
    if (rc != RTNW_OK) return rc;
    rtnw_multi_scene* ms = new rtnw_multi_scene();
    ms->n = m->n;
    for (int d = 0; d < m->n; ++d) {
        rc = rtnw_scene_upload_prepared(m->ctx[d], P, &ms->scene[d]);
        if (rc != RTNW_OK) { const std::string msg = g_err; rtnw_scene_free_multi(m, ms); rtnw_prepared_free(P); return fail(rc, msg); }
    }
    rtnw_prepared_free(P);
    *out = ms;
    return RTNW_OK;
}

int rtnw_render_multi(rtnw_multi* m, const rtnw_multi_scene* ms, const rtnw_camera* cam, const rtnw_render_params* params,
                      float* accum_rgb, rtnw_stats* stats) {
    if (!m || !ms || ms->n != m->n || !cam || !accum_rgb) return fail(RTNW_ERR_INVALID, "null argument");
    int rc = validate_params(params);
    if (rc != RTNW_OK) return rc;
    if (params->pixel_count != 0 || params->sample_begin != 0 || params->sample_stride != 1 ||
        (params->flags & (RTNW_F_ACCUMULATE | RTNW_F_ROTATE_SAMPLES)))
        return fail(RTNW_ERR_INVALID, "rtnw_render_multi renders whole frames: sample_begin 0, sample_stride 1, no pixel subset, no ACCUMULATE / ROTATE flags");
    const int n = m->n;
    const size_t floats = (size_t)params->nx * params->ny * 3;
    int need_stage = 0;
    for (int d = 1; d < n; ++d) need_stage += m->peer[d] ? 0 : 1;
    for (int d = 0; d < n; ++d) {
        CUDA_TRY(cudaSetDevice(m->ctx[d]->device));
        rc = grow(&m->accum[d], &m->accum_floats[d], floats, "cannot allocate the per-device accumulation buffers");
        if (rc != RTNW_OK) return rc;
    }
    if (need_stage) {
        CUDA_TRY(cudaSetDevice(m->ctx[0]->device));
        if ((rc = grow(&m->stage, &m->stage_floats, floats * need_stage, "cannot allocate the staging planes")) != RTNW_OK) return rc;
    }
    // every device renders its share of every pixel's samples (ownership rotates with the pixel index: even for any ns)
    render_ticket ticket[RTNW_MAX_DEVICES];
    CUDA_TRY(cudaSetDevice(m->ctx[0]->device));
    CUDA_TRY(cudaEventRecord(m->ctx[0]->ev_t0, m->ctx[0]->stream));
    for (int d = 0; d < n; ++d) {
        rtnw_ctx* c = m->ctx[d];
        CUDA_TRY(cudaSetDevice(c->device));
        rtnw_render_params p = *params;
        if (n > 1) { p.flags |= RTNW_F_ROTATE_SAMPLES; p.sample_begin = d; p.sample_stride = n; }
        rc = render_launch(c, ms->scene[d], cam, &p, m->accum[d], c->stream, &ticket[d]);
        if (rc != RTNW_OK) return rc;
        CUDA_TRY(cudaEventRecord(m->done[d], c->stream));
    }
    // one sum on device 0, in rank order (deterministic), then the frame goes to the host
    rtnw_ctx* c0 = m->ctx[0];
    CUDA_TRY(cudaSetDevice(c0->device));
    if (n > 1) {
        rank_planes P;
        P.n = n;
        int staged = 0;
        for (int d = 1; d < n; ++d) {
            CUDA_TRY(cudaStreamWaitEvent(c0->stream, m->done[d], 0));
            if (m->peer[d]) P.src[d] = m->accum[d];
            else {
                float* dst = m->stage + floats * (size_t)staged++;
                CUDA_TRY(cudaMemcpyPeerAsync(dst, c0->device, m->accum[d], m->ctx[d]->device, floats * sizeof(float), c0->stream));
                P.src[d] = dst;
            }
        }
        P.src[0] = m->accum[0];
        k_sum_ranks<<<c0->sm_count * 8, 256, 0, c0->stream>>>(m->accum[0], P, floats);
        CUDA_TRY(cudaGetLastError());
    }
    CUDA_TRY(cudaMemcpyAsync(accum_rgb, m->accum[0], floats * sizeof(float), cudaMemcpyDeviceToHost, c0->stream));
    CUDA_TRY(cudaEventRecord(c0->ev_t1, c0->stream));
    rtnw_stats total;
    std::memset(&total, 0, sizeof total);
    for (int d = 0; d < n; ++d) {
        CUDA_TRY(cudaSetDevice(m->ctx[d]->device));
        rtnw_stats st;
        rc = render_finish(m->ctx[d], ticket[d], &st);
        if (rc != RTNW_OK) return rc;
        total.paths += st.paths; total.rays += st.rays; total.box_tests += st.box_tests; total.prim_tests += st.prim_tests;
        total.kernel_ms = std::max(total.kernel_ms, st.kernel_ms);
        total.kernel_launches += st.kernel_launches;
        total.sample_ranges = std::max(total.sample_ranges, st.sample_ranges);
    }
    CUDA_TRY(cudaSetDevice(c0->device));
    CUDA_TRY(cudaStreamSynchronize(c0->stream));
    CUDA_TRY(cudaEventElapsedTime(&total.total_ms, c0->ev_t0, c0->ev_t1));
    if (n > 1) total.kernel_launches += 1;
    if (stats) *stats = total;
    return RTNW_OK;
}

}  // extern "C"
