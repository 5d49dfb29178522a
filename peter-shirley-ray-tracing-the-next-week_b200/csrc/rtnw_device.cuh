// rtnw_device.cuh — device functions of the B200 path tracer (sm_100a).
//
// Everything the reference evaluates per ray on the CPU (PSC/ = "Peter-Shirley-Project Code/" of the reference):
//   camera::get_ray                    PSC/camera.h:41-56
//   hitable_list::hit / bvh_node::hit  PSC/hitable_list.h:20-32, PSC/bvh.h:29-54, PSC/aabb.h:33-49 (+F2 origin fix)
//   sphere / moving_sphere / rects     PSC/sphere.h:25-52,92-118, PSC/aarect.h:50-100, PSC/box.h:36-38
//   translate / rotate_y / flip        PSC/hitable.h:39-150
//   constant_medium::hit               PSC/constant_medium.h:26-50
//   material::scatter / emitted        PSC/material.h:16-151
//   texture::value, perlin             PSC/texture.h, PSC/perlin.h, PSC/surface_texture.h
//   color / de_nan / sample loop       PSC/main.cpp:25-46,232-242,304-313
//
// Numerical contract: float32 with the reference's operation order, no FMA contraction (the TU is compiled with
// --fmad=false; IEEE div/sqrt are nvcc defaults), double only where the reference's C++ promotes to double.
// Consequently t / p / normal are bit-identical to the reference for every primitive; only libm calls
// (atan2f, asinf, sinf, log, pow) can differ by an ulp.
//
// Scene layout (DESIGN.md §3): ONE linear stream of 32-byte records, traversed front to back without a stack.
// BVH nodes are stored in preorder with a skip link; because the reference's bvh_node::hit hands both children
// the UN-narrowed [tmin,tmax] (PSC/bvh.h:34-35), the set of leaves it tests does not depend on traversal order,
// and "closest hit, ties to the right child" equals "scan leaves left to right, replace unless best_t < t".
#pragma once

#include <cuda_runtime.h>
#include <float.h>
#include <math.h>
#include <stdint.h>

#include "rtnw.h"

namespace rtnw_dev {

// ------------------------------------------------------------------------------------------------ records
enum rec_kind : uint32_t {
    K_SPHERE = 0, K_MSPHERE = 1, K_RECT_XY = 2, K_RECT_XZ = 3, K_RECT_YZ = 4, K_BOX = 5, K_MEDIUM = 6, K_EXT = 7,
    K_NODE = 8, K_ITEM = 9, K_END = 10,
    // run headers inside a list item (scan_run): the next a.x records are plain spheres / plain (moving) spheres / plain boxes
    // without a transform chain, scanned by a loop specialised for them — same records, same order, same narrowing
    K_RUN_SPHERE = 11, K_RUN_SPHERELIKE = 12, K_RUN_BOX = 13
};
#define RTNW_TAG_FLIP 16u
#define RTNW_TAG_CONT 32u  // same narrowing scope as the previous primitive (list semantics, PSC/hitable_list.h:23-29)
#define RTNW_TAG_LAST 64u  // last primitive of a BVH leaf: the leaf scan ends here without looking at the next record
#define RTNW_TAG(kind, flip, cont, xf) ((uint32_t)(kind) | ((flip) ? RTNW_TAG_FLIP : 0u) | ((cont) ? RTNW_TAG_CONT : 0u) | ((uint32_t)(xf) << 8))

struct __align__(16) rec {
    float4 a;  // geometry
    float4 b;  // b.x, b.y geometry; b.z = tag bits; b.w = int: material (prims) / skip index (nodes) / mode (items)
};

struct scene_view {
    const rec* recs;            // the stream; recs[0] is the first ITEM, the last record is K_END
    const int32_t* rec_leaf;    // per record: leaf id (parity output only)
    const rtnw_xform_op* xforms;
    const rtnw_material* materials;
    const rtnw_texture* textures;
    const uint8_t* images;
    const float4* ranvec;       // 256 gradients, PSC/perlin.h:82-87
    const uint8_t* perm;        // perm_x | perm_y | perm_z, 256 bytes each, PSC/perlin.h:99-106
    const uint32_t* rec_xf;     // per record: transform chain of the item it belongs to
    const float4* wnodes;       // gate tree, 8 float4 per 4-wide node: minx[4] miny[4] minz[4] maxx[4] maxy[4] maxz[4], then
                                // child refs (int4): >= 0 wide node, < 0 ~gate, RTNW_REF_NONE absent; last float4 unused
    const int2* gates;          // per gate: first records of the (one or two) leaves it guards, -1 = none
    int32_t n_recs, n_materials, n_textures;
    int32_t n_wnodes, fast_node_base;  // wide nodes in the table; first node of the RTNW_F_FAST_BVH forest (the exact forest starts at 0)
};

// ------------------------------------------------------------------------------------------------ vec3
struct f3 { float x, y, z; };
__device__ __forceinline__ f3 mk3(float x, float y, float z) { f3 r; r.x = x; r.y = y; r.z = z; return r; }
__device__ __forceinline__ f3 operator+(f3 a, f3 b) { return mk3(a.x + b.x, a.y + b.y, a.z + b.z); }
__device__ __forceinline__ f3 operator-(f3 a, f3 b) { return mk3(a.x - b.x, a.y - b.y, a.z - b.z); }
__device__ __forceinline__ f3 operator*(f3 a, f3 b) { return mk3(a.x * b.x, a.y * b.y, a.z * b.z); }
__device__ __forceinline__ f3 operator*(float t, f3 a) { return mk3(t * a.x, t * a.y, t * a.z); }
__device__ __forceinline__ f3 operator/(f3 a, float t) { return mk3(a.x / t, a.y / t, a.z / t); }  // PSC/vec3.h:82
__device__ __forceinline__ f3 operator-(f3 a) { return mk3(-a.x, -a.y, -a.z); }
__device__ __forceinline__ float dot(f3 a, f3 b) { return a.x * b.x + a.y * b.y + a.z * b.z; }  // ((x+y)+z), PSC/vec3.h:90
__device__ __forceinline__ float length(f3 a) { return sqrtf(dot(a, a)); }
__device__ __forceinline__ f3 unit_vector(f3 a) { return a / length(a); }

struct ray_t { f3 o, d; float time; };

// ------------------------------------------------------------------------------------------------ Philox4x32-10
// Replaces the process-global drand48 stream (DESIGN.md §4).  The reference oracle (oracle/ref_harness.cpp) is
// driven by the SAME generator, so GPU and reference consume identical numbers.
__device__ __forceinline__ void philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0, uint32_t k1,
                                              uint32_t& o0, uint32_t& o1, uint32_t& o2, uint32_t& o3) {
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        const uint32_t hi0 = __umulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
        const uint32_t hi1 = __umulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
        c0 = hi1 ^ c1 ^ k0;
        c1 = lo1;
        c2 = hi0 ^ c3 ^ k1;
        c3 = lo0;
        k0 += 0x9E3779B9u;
        k1 += 0xBB67AE85u;
    }
    o0 = c0; o1 = c1; o2 = c2; o3 = c3;
}
__device__ __forceinline__ float u01(uint32_t x) { return (float)(x >> 8) * (1.0f / 16777216.0f); }

// one copy of the 10 rounds in the binary (path seeding and medium draws call it)
__device__ __noinline__ uint4 philox_block(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0, uint32_t k1) {
    uint4 o;
    philox4x32_10(c0, c1, c2, c3, k0, k1, o.x, o.y, o.z, o.w);
    return o;
}

// The sequential stream of one path (DESIGN.md §4): Philox(counter = (0, 0, sample, pixel), key = seed) gives the 48-bit
// initial state, and the stream itself is the reference's own generator, the drand48 recurrence
// X <- (0x5DEECE66D * X + 0xB) mod 2^48 (glibc), of which a draw returns the top 24 bits as a float in [0,1).
// Counter-based where it matters (any path can be started anywhere, on any GPU), and a draw costs one 64-bit
// multiply-add instead of a quarter of a Philox block, with no data-dependent refill to diverge on.
struct rng_t {
    unsigned long long x;
    uint32_t sample;
    __device__ __forceinline__ void begin(uint32_t key0, uint32_t key1, uint32_t px, uint32_t s) {
        const uint4 o = philox_block(0u, 0u, s, px, key0, key1);
        x = ((unsigned long long)(o.y & 0xffffu) << 32) | (unsigned long long)o.x;
        sample = s;
    }
    __device__ __forceinline__ float draw() {
        x = (x * 0x5DEECE66Dull + 0xBull) & 0xffffffffffffull;
        return (float)(uint32_t)(x >> 24) * (1.0f / 16777216.0f);
    }
};
// keyed draw of a medium's free-flight number: independent of traversal order and of how often the leaf is tested
__device__ __forceinline__ float keyed_draw(uint32_t k0, uint32_t k1, uint32_t pixel, uint32_t sample, uint32_t depth, uint32_t leaf) {
    return u01(philox_block(leaf, 1u + depth, sample, pixel, k0, k1).x);
}

// PSC/material.h:41-47.  g++ evaluates `vec3(drand48(),drand48(),drand48())` right to left: first draw -> z.
__device__ __forceinline__ f3 random_in_unit_sphere(rng_t& g) {
    f3 p;
    do {
        const float dz = g.draw(), dy = g.draw(), dx = g.draw();
        p = 2.0f * mk3(dx, dy, dz) - mk3(1.f, 1.f, 1.f);
    } while (dot(p, p) >= 1.0f);
    return p;
}

// ------------------------------------------------------------------------------------------------ transforms
// PSC/hitable.h:66-74 (translate) and :128-150 (rotate_y); chains are applied to the ray first-to-last.
__device__ __forceinline__ void xform_ray(const rtnw_xform_op* __restrict__ ops, uint32_t chain, ray_t& r) {
    if (chain == 0) return;
    const uint32_t n = __ldg(&ops[chain].kind) >> 8;
    for (uint32_t k = 0; k < n; ++k) {
        const float4 op = __ldg(reinterpret_cast<const float4*>(ops + chain + k));
        if ((__float_as_uint(op.w) & 0xffu) == RTNW_XF_TRANSLATE) {
            r.o = r.o - mk3(op.x, op.y, op.z);
        } else {  // ROTATE_Y: op.x = sin, op.y = cos
            const float ox = op.y * r.o.x - op.x * r.o.z, oz = op.x * r.o.x + op.y * r.o.z;
            const float dx = op.y * r.d.x - op.x * r.d.z, dz = op.x * r.d.x + op.y * r.d.z;
            r.o.x = ox; r.o.z = oz; r.d.x = dx; r.d.z = dz;
        }
    }
}
// the hit is carried back out last-to-first
__device__ __forceinline__ void xform_hit_back(const rtnw_xform_op* __restrict__ ops, uint32_t chain, f3& p, f3& nrm) {
    if (chain == 0) return;
    const uint32_t n = __ldg(&ops[chain].kind) >> 8;
    for (int k = (int)n - 1; k >= 0; --k) {
        const float4 op = __ldg(reinterpret_cast<const float4*>(ops + chain + k));
        if ((__float_as_uint(op.w) & 0xffu) == RTNW_XF_TRANSLATE) {
            p = p + mk3(op.x, op.y, op.z);
        } else {
            const float px = op.y * p.x + op.x * p.z, pz = (-op.x) * p.x + op.y * p.z;
            const float nx = op.y * nrm.x + op.x * nrm.z, nz = (-op.x) * nrm.x + op.y * nrm.z;
            p.x = px; p.z = pz; nrm.x = nx; nrm.z = nz;
        }
    }
}

// ------------------------------------------------------------------------------------------------ primitives
// Each returns true and writes t when the reference's hit() would return true for (t_lo, t_hi).

// ---- IEEE quotients from a reciprocal the ray already carries
// A BVH item keeps RN(1/d) per axis for aabb::hit (PSC/aabb.h:38) and, since every sphere divides by it, RN(1/dot(d,d)).
// With y = RN(1/d):  q0 = RN(x*y) is within 2 ulp of x/d;  q1 = RN(q0 + RN(x - q0*d)*y) is faithful;  the residual
// r = x - q1*d of a faithful quotient is exact in one FMA, and RN(q1 + r*y) = RN(x/d) (Markstein's theorem) — the bits an
// IEEE division returns, in five dependent FMA-pipe instructions instead of MUFU.RCP + eight + a range check.  The theorem
// needs every intermediate in the normal range.  The callers' guard: |d| within 2^+-40 and |x| <= 2^80 (fmaxf skips a NaN
// x, whose quotient is the same canonical NaN either way) — then q*d and both residuals are finite, and they are normal
// unless |x/d| < 2^-31, a quotient no caller looks at beyond `t < t_lo` / `t <= t_lo` with t_lo >= 2^-30 (also required),
// which a wrong last bit or a wrong sign of zero cannot flip.  Outside the guard: the IEEE division.
// tests/test_gpu_parity.py::test_division_by_reciprocal compares 2^30 pairs (random, extreme mantissas, zeros) bit for bit.
// How a primitive test divides: the IEEE division, or the exact shortcut above (the leaf tests of a BVH item).
enum { ARITH_IEEE = 0, ARITH_RECIP = 1 };
struct ray_recip { f3 inv; float inv_a; };
__device__ __forceinline__ float div_by_recip(float x, float d, float y) {
    float q = x * y;
    q = fmaf(fmaf(-q, d, x), y, q);
    return fmaf(fmaf(-q, d, x), y, q);
}
#define RTNW_RECIP_DMIN 0x1p-40f
#define RTNW_RECIP_DMAX 0x1p40f
#define RTNW_RECIP_XMAX 0x1p80f
#define RTNW_RECIP_TLO 0x1p-30f
// PSC/sphere.h:25-52.  a = dot(d,d) is a pure function of the ray and is hoisted by the callers.
__device__ __forceinline__ bool hit_sphere(f3 c, float radius, const ray_t& r, float a, float t_lo, float t_hi, float& t) {
    const f3 oc = r.o - c;
    const float b = dot(oc, r.d);
    const float cc = dot(oc, oc) - radius * radius;
    const float disc = b * b - a * cc;
    if (disc > 0.f) {
        const float sq = sqrtf(disc);
        float temp = (-b - sq) / a;
        if (temp < t_hi && temp > t_lo) { t = temp; return true; }
        temp = (-b + sq) / a;
        if (temp < t_hi && temp > t_lo) { t = temp; return true; }
    }
    return false;
}
// the same with both roots divided through inv_a = RN(1/a)
__device__ __forceinline__ bool hit_sphere_recip(f3 c, float radius, const ray_t& r, float a, float inv_a, float t_lo, float t_hi, float& t) {
    const f3 oc = r.o - c;
    const float b = dot(oc, r.d);
    const float cc = dot(oc, oc) - radius * radius;
    const float disc = b * b - a * cc;
    if (disc > 0.f) {
        const float sq = sqrtf(disc);
        const float x0 = -b - sq, x1 = -b + sq;
        float q0 = div_by_recip(x0, a, inv_a), q1 = div_by_recip(x1, a, inv_a);
        if (!(a >= RTNW_RECIP_DMIN && a <= RTNW_RECIP_DMAX && fmaxf(fabsf(x0), fabsf(x1)) <= RTNW_RECIP_XMAX && t_lo >= RTNW_RECIP_TLO)) {
            q0 = x0 / a; q1 = x1 / a;
        }
        if (q0 < t_hi && q0 > t_lo) { t = q0; return true; }
        if (q1 < t_hi && q1 > t_lo) { t = q1; return true; }
    }
    return false;
}
// PSC/sphere.h:81-83
__device__ __forceinline__ f3 moving_center(f3 c0, f3 c1, float time0, float time1, float time) {
    return c0 + ((time - time0) / (time1 - time0)) * (c1 - c0);
}
// PSC/aarect.h:50-100: plane axis N, extent axes A,B; inclusive bounds; a NaN t passes, as in the reference.
template <int N, int A, int B>
__device__ __forceinline__ bool hit_rect(float a0, float a1, float b0, float b1, float k, const ray_t& r, float t_lo, float t_hi, float& t) {
    const float* o = &r.o.x;
    const float* d = &r.d.x;
    const float tt = (k - o[N]) / d[N];
    if (tt < t_lo || tt > t_hi) return false;
    const float a = o[A] + tt * d[A];
    const float b = o[B] + tt * d[B];
    if (a < a0 || a > a1 || b < b0 || b > b1) return false;
    t = tt;
    return true;
}
// PSC/box.h:23-38: inner list of six faces, order +z, -z, +y, -y, +x, -x, narrowing from t_hi.  The six plane distances
// and extent tests do not depend on the narrowing limit, so they are evaluated first (independent IEEE divisions that
// interleave); the list's sequential narrowing is then six compare/selects over the same predicates as hit_rect
// (a NaN t passes every comparison exactly as there).
template <int ARITH>
__device__ __forceinline__ bool hit_box(f3 p0, f3 p1, const ray_t& r, const ray_recip& rr, float t_lo, float t_hi, float& t, int& face,
                                        bool* took_ieee = nullptr) {
    float tt[6];
    bool in[6];
    const float x[6] = {p1.z - r.o.z, p0.z - r.o.z, p1.y - r.o.y, p0.y - r.o.y, p1.x - r.o.x, p0.x - r.o.x};
    bool ieee = true;
    if (ARITH == ARITH_RECIP) {
        tt[0] = div_by_recip(x[0], r.d.z, rr.inv.z); tt[1] = div_by_recip(x[1], r.d.z, rr.inv.z);
        tt[2] = div_by_recip(x[2], r.d.y, rr.inv.y); tt[3] = div_by_recip(x[3], r.d.y, rr.inv.y);
        tt[4] = div_by_recip(x[4], r.d.x, rr.inv.x); tt[5] = div_by_recip(x[5], r.d.x, rr.inv.x);
        const float dlo = fminf(fminf(fabsf(r.d.x), fabsf(r.d.y)), fabsf(r.d.z)), dhi = fmaxf(fmaxf(fabsf(r.d.x), fabsf(r.d.y)), fabsf(r.d.z));
        const float xhi = fmaxf(fmaxf(fmaxf(fabsf(x[0]), fabsf(x[1])), fmaxf(fabsf(x[2]), fabsf(x[3]))), fmaxf(fabsf(x[4]), fabsf(x[5])));
        ieee = !(dlo >= RTNW_RECIP_DMIN && dhi <= RTNW_RECIP_DMAX && xhi <= RTNW_RECIP_XMAX && t_lo >= RTNW_RECIP_TLO);
    }
    if (took_ieee) *took_ieee = ieee;
    if (ieee) {
        tt[0] = x[0] / r.d.z; tt[1] = x[1] / r.d.z;
        tt[2] = x[2] / r.d.y; tt[3] = x[3] / r.d.y;
        tt[4] = x[4] / r.d.x; tt[5] = x[5] / r.d.x;
    }
#pragma unroll
    for (int f = 0; f < 2; ++f) {  // xy faces
        const float a = r.o.x + tt[f] * r.d.x, b = r.o.y + tt[f] * r.d.y;
        in[f] = !(a < p0.x || a > p1.x || b < p0.y || b > p1.y);
    }
#pragma unroll
    for (int f = 2; f < 4; ++f) {  // xz faces
        const float a = r.o.x + tt[f] * r.d.x, b = r.o.z + tt[f] * r.d.z;
        in[f] = !(a < p0.x || a > p1.x || b < p0.z || b > p1.z);
    }
#pragma unroll
    for (int f = 4; f < 6; ++f) {  // yz faces
        const float a = r.o.y + tt[f] * r.d.y, b = r.o.z + tt[f] * r.d.z;
        in[f] = !(a < p0.y || a > p1.y || b < p0.z || b > p1.z);
    }
    bool any = false;
    float lim = t_hi;
#pragma unroll
    for (int f = 0; f < 6; ++f) {
        const bool hit = in[f] & !(tt[f] < t_lo || tt[f] > lim);
        if (hit) { any = true; lim = tt[f]; face = f; }
    }
    t = lim;
    return any;
}

// One surface primitive record (not a medium) against a ray given in the enclosing frame.  `a_frame` is dot(d,d)
// of that frame; a primitive with its own transform chain recomputes it from the transformed direction.
// Inlined at its four sites (list scan and gate task, each directly and as a medium boundary).  A single __noinline__
// copy shrinks k_render from 127 KB to 95 KB of SASS (the L1.5 I-cache holds 32 KB; ncu r9: icc hit rate 91 %) but was
// measured 4 % slower: the call's register shuffling costs more than the fetches it saves.
struct surf_hit_t { float t; int face; };  // face < 0: miss
template <int ARITH>
__device__ __forceinline__ surf_hit_t hit_surface_rec(const rec* __restrict__ recs, const rtnw_xform_op* __restrict__ xforms, int i, float4 A,
                                                      float4 B, ray_t r, float a, ray_recip rr, float t_lo, float t_hi) {
    const uint32_t tag = __float_as_uint(B.z);
    const uint32_t kind = tag & 15u;
    const uint32_t chain = tag >> 8;
    if (chain) {
        xform_ray(xforms, chain, r);
        a = dot(r.d, r.d);
        if (ARITH != ARITH_IEEE) { rr.inv = mk3(1.0f / r.d.x, 1.0f / r.d.y, 1.0f / r.d.z); rr.inv_a = 1.0f / a; }
    }
    surf_hit_t out;
    out.face = 0;
    out.t = 0.f;
    bool hit;
    switch (kind) {
        case K_SPHERE:
            hit = ARITH == ARITH_RECIP ? hit_sphere_recip(mk3(A.x, A.y, A.z), A.w, r, a, rr.inv_a, t_lo, t_hi, out.t)
                                       : hit_sphere(mk3(A.x, A.y, A.z), A.w, r, a, t_lo, t_hi, out.t);
            break;
        case K_MSPHERE: {
            const float4 A2 = __ldg(&recs[i + 1].a);
            const f3 c = moving_center(mk3(A.x, A.y, A.z), mk3(A2.x, A2.y, A2.z), B.x, B.y, r.time);
            hit = ARITH == ARITH_RECIP ? hit_sphere_recip(c, A.w, r, a, rr.inv_a, t_lo, t_hi, out.t)
                                       : hit_sphere(c, A.w, r, a, t_lo, t_hi, out.t);
            break;
        }
        case K_RECT_XY: hit = hit_rect<2, 0, 1>(A.x, A.y, A.z, A.w, B.x, r, t_lo, t_hi, out.t); break;
        case K_RECT_XZ: hit = hit_rect<1, 0, 2>(A.x, A.y, A.z, A.w, B.x, r, t_lo, t_hi, out.t); break;
        case K_RECT_YZ: hit = hit_rect<0, 1, 2>(A.x, A.y, A.z, A.w, B.x, r, t_lo, t_hi, out.t); break;
        case K_BOX: hit = hit_box<ARITH>(mk3(A.x, A.y, A.z), mk3(A.w, B.x, B.y), r, rr, t_lo, t_hi, out.t, out.face); break;
        default: hit = false; break;
    }
    if (!hit) out.face = -1;
    return out;
}
template <int ARITH = ARITH_IEEE>
__device__ __forceinline__ bool hit_surface(const scene_view& S, int i, float4 A, float4 B, uint32_t tag, const ray_t& r_frame,
                                            float a_frame, float t_lo, float t_hi, float& t, int& face, const ray_recip& rr = ray_recip()) {
    const surf_hit_t h = hit_surface_rec<ARITH>(S.recs, S.xforms, i, A, B, r_frame, a_frame, rr, t_lo, t_hi);
    t = h.t;
    face = h.face < 0 ? 0 : h.face;
    return h.face >= 0;
}

// boundary->hit(r, t_lo, t_hi, rec) of a constant_medium: list semantics over the nb boundary records that follow it
__device__ __forceinline__ bool hit_boundary(const scene_view& S, int first, int nb, const ray_t& r, float a, float t_lo, float t_hi, float& t) {
    bool any = false;
    float lim = t_hi;
#pragma unroll 1
    for (int i = first; i < first + nb; ++i) {
        const float4 A = __ldg(&S.recs[i].a), B = __ldg(&S.recs[i].b);
        const uint32_t tag = __float_as_uint(B.z);
        if ((tag & 15u) == K_EXT) continue;
        float tt; int face;
        if (hit_surface(S, i, A, B, tag, r, a, t_lo, lim, tt, face)) { any = true; lim = tt; }
    }
    t = lim;
    return any;
}

struct medium_key { uint32_t k0, k1, pixel, sample, depth; };

// PSC/constant_medium.h:26-50
__device__ __forceinline__ bool hit_medium(const scene_view& S, int i, float4 A, uint32_t tag, const ray_t& r_frame, float a_frame,
                                           float t_lo, float t_hi, const medium_key& mk, float& t) {
    ray_t r = r_frame;
    float a = a_frame;
    const uint32_t chain = tag >> 8;
    if (chain) { xform_ray(S.xforms, chain, r); a = dot(r.d, r.d); }
    const int nb = __float_as_int(A.z);
    float t1 = 0.f, t2 = 0.f;
    const float4 SA = __ldg(&S.recs[i + 1].a);
    if (nb == 1 && (__float_as_uint(__ldg(&S.recs[i + 1].b).z) & ~(uint32_t)(RTNW_TAG_FLIP | RTNW_TAG_CONT | RTNW_TAG_LAST)) == K_SPHERE) {
        // the boundary is one plain sphere (the media of final(), PSC/main.cpp:209-212): the two boundary->hit calls without
        // the boundary loop and the kind switch
        if (!hit_sphere(mk3(SA.x, SA.y, SA.z), SA.w, r, a, -FLT_MAX, FLT_MAX, t1)) return false;
        if (!hit_sphere(mk3(SA.x, SA.y, SA.z), SA.w, r, a, (float)((double)t1 + 0.0001), FLT_MAX, t2)) return false;
    } else {
#pragma unroll 1
        for (int pass = 0; pass < 2; ++pass) {  // rec1 over (-FLT_MAX, FLT_MAX), then rec2 over (rec1.t + 0.0001, FLT_MAX)
            float tt;
            if (!hit_boundary(S, i + 1, nb, r, a, pass ? (float)((double)t1 + 0.0001) : -FLT_MAX, FLT_MAX, tt)) return false;
            if (pass) t2 = tt; else t1 = tt;
        }
    }
    if (t1 < t_lo) t1 = t_lo;
    if (t2 > t_hi) t2 = t_hi;
    if (t1 >= t2) return false;
    if (t1 < 0.f) t1 = 0.f;
    const float len = sqrtf(a);  // r.direction().length(), same expression as dot(d,d)
    const float inside = (t2 - t1) * len;
    const float u = keyed_draw(mk.k0, mk.k1, mk.pixel, mk.sample, mk.depth, (uint32_t)__float_as_int(A.y));
    const float hit_distance = (float)((double)A.w * log((double)u));  // A.w = -(1 / density), rounded once on the host as PSC/constant_medium.h:42 does
    if (hit_distance < inside) {
        t = t1 + hit_distance / len;
        return true;
    }
    return false;
}

// ------------------------------------------------------------------------------------------------ closest hit
struct hit_t {
    float t;
    int rec;      // record index, -1 = miss
    int face;     // box face 0..5
    uint32_t xf;  // transform chain of the item the record was reached in
};

struct trav_counters { uint32_t box_tests, prim_tests; };

// The running closest hit of one query as a single 64-bit key, smaller = better:
//   bits 63..32  t, mapped so that unsigned order == float order
//   bits 31..3   (2^28-1) - record index: among equal t the LATER record of the stream wins, which is
//                bvh_node::hit's "right child unless left.t < right.t" (PSC/bvh.h:37-40) and the inclusive
//                narrowing of rectangles in a list (PSC/aarect.h:52)
//   bits  2..0   box face
// so candidates found by different threads combine with one atomicMin.
typedef unsigned long long hkey_t;
#define RTNW_KEY_NONE 0xffffffffffffffffull
__device__ __forceinline__ uint32_t float_order(float f) {
    const uint32_t b = __float_as_uint(f);
    return b ^ ((b >> 31) ? 0xffffffffu : 0x80000000u);
}
__device__ __forceinline__ float order_float(uint32_t u) {
    return __uint_as_float(u ^ ((u >> 31) ? 0x80000000u : 0xffffffffu));
}
__device__ __forceinline__ hkey_t make_key(float t, int rec, int face) {
    return ((hkey_t)float_order(t) << 32) | (hkey_t)(((0x0fffffffu - (uint32_t)rec) << 3) | (uint32_t)face);
}
__device__ __forceinline__ float key_t_or(hkey_t k, float t_max) { return k == RTNW_KEY_NONE ? t_max : order_float((uint32_t)(k >> 32)); }
__device__ __forceinline__ int key_rec(hkey_t k) { return (int)(0x0fffffffu - (((uint32_t)k) >> 3)); }
__device__ __forceinline__ int key_face(hkey_t k) { return (int)(((uint32_t)k) & 7u); }

// One primitive record (surface or medium) of a scope whose narrowing limit is `lim`; returns records consumed.
template <bool COUNT, int ARITH = ARITH_IEEE>
__device__ __forceinline__ int test_record(const scene_view& S, int i, float4 A, float4 B, const ray_t& r, float a, float t_min,
                                           float lim, const medium_key& mk, bool& hit, float& t, int& face, trav_counters& cnt,
                                           const ray_recip& rr = ray_recip()) {
    const uint32_t tag = __float_as_uint(B.z);
    const uint32_t kind = tag & 15u;
    if (COUNT) cnt.prim_tests++;
    face = 0;
    if (kind == K_MEDIUM) {
        hit = hit_medium(S, i, A, tag, r, a, t_min, lim, mk, t);
        return 1 + __float_as_int(A.z);
    }
    hit = hit_surface<ARITH>(S, i, A, B, tag, r, a, t_min, lim, t, face, rr);
    return kind == K_MSPHERE ? 2 : 1;
}

// A leaf of a bvh_node (one hitable, possibly a list of several primitives): tested with the UN-narrowed range the
// node received, narrowing only inside the leaf (PSC/bvh.h:34-35, PSC/hitable_list.h:23-29).  Returns its candidate key.
template <bool COUNT, int ARITH>
__device__ __forceinline__ hkey_t test_leaf(const scene_view& S, int first, float4 A, float4 B, const ray_t& r, float a, const ray_recip& rr,
                                            float t_min, float tmax0, const medium_key& mk, trav_counters& cnt) {
    hkey_t best = RTNW_KEY_NONE;
    float lim = tmax0;
    int i = first;  // A, B: record `first`, loaded by the caller (both leaves of a gate are fetched before either is tested)
    for (;;) {
        bool hit; float t; int face;
        const int step = test_record<COUNT, ARITH>(S, i, A, B, r, a, t_min, lim, mk, hit, t, face, cnt, rr);
        if (hit) { lim = t; best = make_key(t, i, face); }  // inside a list the later accepted hit always replaces
        if (__float_as_uint(B.z) & RTNW_TAG_LAST) break;
        i += step;
        A = __ldg(&S.recs[i].a); B = __ldg(&S.recs[i].b);
    }
    return best;
}

#ifdef RTNW_ROUND_STATS  // tuning aid (never defined in the product build): shape of the cooperative rounds
__device__ unsigned long long g_round_stats[32];
#define RTNW_STAT(i, v) atomicAdd(&g_round_stats[i], (unsigned long long)(v))
#else
#define RTNW_STAT(i, v) ((void)0)
#endif

// A run of same-kind plain records inside a list item (hitable_list::hit, PSC/hitable_list.h:20-32): the generic scan spends
// ~50 of its ~80 instructions per primitive on record decode, the kind switch and loop bookkeeping; all lanes of a warp
// scan the same record, so a loop that knows the kind needs one 128-bit load and the arithmetic of the test itself.
// Order, narrowing limit and the key of an accepted hit are exactly those of the generic scan.
template <bool COUNT, int RUN>
__device__ __forceinline__ void scan_run(const scene_view& S, int first, int nrec, const ray_t& r, float a, float t_min, float& lim,
                                         hkey_t& key, trav_counters& cnt) {
    const int end = first + nrec;
    if (RUN == K_RUN_SPHERE) {  // PSC/sphere.h:25-52, one record each
        // four spheres per step: the discriminants (the part every sphere pays) are four independent straight-line chains that
        // interleave; the roots and the narrowing, which only a sphere the ray's line meets needs, follow in record order
        int j = first;
#pragma unroll 1
        for (; j + 4 <= end; j += 4) {
            float bq[4], dq[4];
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                const float4 A = __ldg(&S.recs[j + q].a);
                const f3 oc = r.o - mk3(A.x, A.y, A.z);
                bq[q] = dot(oc, r.d);
                const float cc = dot(oc, oc) - A.w * A.w;
                dq[q] = bq[q] * bq[q] - a * cc;
            }
            if ((dq[0] > 0.f) | (dq[1] > 0.f) | (dq[2] > 0.f) | (dq[3] > 0.f)) {
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                    if (dq[q] > 0.f) {
                        const float sq = sqrtf(dq[q]);
                        float temp = (-bq[q] - sq) / a;
                        if (temp < lim && temp > t_min) { lim = temp; key = make_key(temp, j + q, 0); }
                        else {
                            temp = (-bq[q] + sq) / a;
                            if (temp < lim && temp > t_min) { lim = temp; key = make_key(temp, j + q, 0); }
                        }
                    }
                }
            }
        }
        for (; j < end; ++j) {
            const float4 A = __ldg(&S.recs[j].a);
            float t;
            if (hit_sphere(mk3(A.x, A.y, A.z), A.w, r, a, t_min, lim, t)) { lim = t; key = make_key(t, j, 0); }
        }
        if (COUNT) cnt.prim_tests += nrec;
    } else if (RUN == K_RUN_SPHERELIKE) {
        // spheres and moving spheres mixed (PSC/sphere.h:92-118).  Every primitive of such a run takes TWO records (the
        // upload pads a plain sphere with a continuation record), so record positions do not depend on kinds and four
        // primitives' centres and discriminants are computed as independent straight-line chains; a plain sphere is stored
        // as a moving sphere that does not move (shutter (0, 1), c1 = c0: its centre at any time is c0 exactly).
        int j = first;
#pragma unroll 1
        for (; j + 8 <= end; j += 8) {
            float bq[4], dq[4];
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                const float4 A = __ldg(&S.recs[j + 2 * q].a), B = __ldg(&S.recs[j + 2 * q].b), A2 = __ldg(&S.recs[j + 2 * q + 1].a);
                const f3 oc = r.o - moving_center(mk3(A.x, A.y, A.z), mk3(A2.x, A2.y, A2.z), B.x, B.y, r.time);  // a plain sphere: c0 + time * 0
                bq[q] = dot(oc, r.d);
                const float cc = dot(oc, oc) - A.w * A.w;
                dq[q] = bq[q] * bq[q] - a * cc;
            }
            if ((dq[0] > 0.f) | (dq[1] > 0.f) | (dq[2] > 0.f) | (dq[3] > 0.f)) {
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                    if (dq[q] > 0.f) {
                        const float sq = sqrtf(dq[q]);
                        float temp = (-bq[q] - sq) / a;
                        if (temp < lim && temp > t_min) { lim = temp; key = make_key(temp, j + 2 * q, 0); }
                        else {
                            temp = (-bq[q] + sq) / a;
                            if (temp < lim && temp > t_min) { lim = temp; key = make_key(temp, j + 2 * q, 0); }
                        }
                    }
                }
            }
        }
#pragma unroll 1
        for (; j < end; j += 2) {
            const float4 A = __ldg(&S.recs[j].a), B = __ldg(&S.recs[j].b);
            const float4 A2 = __ldg(&S.recs[j + 1].a);
            float t;
            if (hit_sphere(moving_center(mk3(A.x, A.y, A.z), mk3(A2.x, A2.y, A2.z), B.x, B.y, r.time), A.w, r, a, t_min, lim, t)) { lim = t; key = make_key(t, j, 0); }
        }
        if (COUNT) cnt.prim_tests += nrec >> 1;
    } else {  // K_RUN_BOX, PSC/box.h:23-38
#pragma unroll 2
        for (int j = first; j < end; ++j) {
            const float4 A = __ldg(&S.recs[j].a), B = __ldg(&S.recs[j].b);
            float t; int face = 0;
            if (hit_box<ARITH_IEEE>(mk3(A.x, A.y, A.z), mk3(A.w, B.x, B.y), r, ray_recip(), t_min, lim, t, face)) { lim = t; key = make_key(t, j, face); }
        }
        if (COUNT) cnt.prim_tests += nrec;
    }
}

// ---- block-cooperative closest hit --------------------------------------------------------------------------
// Every thread of the block owns one ray (or none).  All rays walk the same record stream, item by item:
//   * a list item (PSC/hitable_list.h:20-32) is scanned by each owner in lockstep: same records, same code, all lanes;
//   * a BVH item is traversed by the WHOLE BLOCK through a shared-memory task stack.
//
// Which leaves does the reference test?  bvh_node::hit hands both children the un-narrowed range (PSC/bvh.h:34-35), so
// a leaf is tested iff the own box of every bvh_node above it passes aabb::hit(r, tmin, tmax0).  A bvh_node's box is
// surrounding_box(left, right) (PSC/bvh.h:120, PSC/aabb.h:54-62), an exact fmin/fmax union, and every operation of the
// slab test (subtract, multiply by 1/d, swap, the NaN-ignoring min/max selects) is monotonic under IEEE rounding:
// a larger box yields a superset interval IN FLOATING POINT.  Hence "box of the leaf's parent passes" already implies
// that all ancestors pass, and the reference's leaf set is exactly { leaves whose parent ("gate") box passes }
// (checked numerically on all node pairs of the test scenes, DESIGN.md §3).  The hierarchy above the gates is only an
// index, so the upload builds its own: a 4-wide SAH tree over the gate boxes whose interior boxes are again exact unions
// (so, by the same monotonicity, they can never cull a passing gate), tested with the same aabb::hit arithmetic.
// Results are identical to the reference's tree; the number of box tests, tasks and rounds is a fraction of it.
//
// Tasks are uniform and any thread can take any of them: a node task (ray, wide node) tests the node's <= 4 child
// boxes and pushes the children that passed — wide nodes back on the stack, gates to the leaf queue; a gate task runs
// leaf->hit(r, tmin, tmax0) for the gate's one or two leaves.  Candidates are merged per ray with atomicMin on the
// 64-bit key.  The stack is served LIFO.  A popped task frees one slot and pushes at most four, so a round that pops
// `take` tasks needs 3*take free slots; `take` is BLOCK while there is room and shrinks as the stack fills, always
// leaving 3*depth slots in reserve: with take = 1 the traversal is a plain depth-first walk, which needs at most
// 3*(depth - d) slots above a task at depth d.  Hence the stack cannot overflow for a tree of any depth, and the usual
// case (room for everything) runs BLOCK tasks wide.
// The cooperating group is the whole block: every thread takes part in every round, and rounds are separated by
// __syncthreads.
#ifndef RTNW_BLOCK
#define RTNW_BLOCK 320      // x 2 blocks per SM at 96 registers: 640 rays in flight per SM (measured against 256 x 2 at 124
#endif                      // registers, 192 x 3, 288 x 2, 352 x 2, 384 x 2 and 256 x 3 at 80: DESIGN.md §6)
#ifndef RTNW_QN_MULT
#define RTNW_QN_MULT 12
#endif
#ifndef RTNW_QL_ABS
#define RTNW_QL_ABS 4096  // gate ring size (a power of two)
#endif
template <int FRAMES = 1>
struct coop_smem {
    static_assert(RTNW_BLOCK <= 512 && RTNW_BLOCK % 32 == 0 && FRAMES * RTNW_BLOCK <= 1024, "a task carries its (frame, owner) slot in 10 bits");
    static constexpr int QN = RTNW_QN_MULT * RTNW_BLOCK;   // node task stack
    static constexpr int QL = RTNW_QL_ABS;   // gate queue (circular, power of two); node work pauses while < 4*RTNW_BLOCK slots are free
    static constexpr int NFRAMES = FRAMES;
    static_assert((QL & (QL - 1)) == 0, "the gate ring must be a power of two");
    // the ray of owner `tid` in the frame of a BVH item lives at index frame * RTNW_BLOCK + tid ("virtual slot"; FRAMES = 2 only
    // in the RTNW_F_FAST_BVH kernels, which traverse two BVH items at once)
    float4 ray_o[FRAMES * RTNW_BLOCK];  // o.xyz in the item frame, w = tmax0 (closest_so_far when the item is entered)
    float4 ray_d[FRAMES * RTNW_BLOCK];  // d.xyz, w = dot(d,d)
    float4 ray_i[FRAMES * RTNW_BLOCK];  // 1/d, w = 1/dot(d,d)
    uint4 mkey[RTNW_BLOCK];    // pixel, sample, depth of the owner's path (keys the free-flight draw of media), w = the ray's time
    float4 acc[RTNW_BLOCK];    // k_render: the owner's work item — xyz = sum of its finished samples, w = next sample index k (int bits)
    int4 span[RTNW_BLOCK];     // k_render: the owner's work item — x = first sample of its pixel in this call (s_begin), y = end index
                               // of its range, z = pixel, w = range
    int bins[8];          // read by nothing; zeroed by coop_init only because deleting that store changes k_render's schedule
                          // (removing the field wants an A/B measurement of its own)
    int4 plan;            // the round's plan (take, base, node_threads, drain), computed by thread 0 alone
    hkey_t key[RTNW_BLOCK];
    uint32_t q[QN + QL];  // [0, QN): node task stack; [QN, QN + QL): gate ring (one array: a push is a single predicated store)
    int n[3];             // node stack height, one buffer per round (read r % 3, popped/pushed (r + 1) % 3, cleared (r + 2) % 3)
    unsigned lh[3];       // gate queue head (consumed), same rotation; counts up for the whole kernel, index = value % QL
    unsigned lt;          // gate queue tail (produced); never reset
    int overflow;         // a push did not fit (cannot happen for validated scenes); reported to the host
};
// task = virtual slot (frame * RTNW_BLOCK + owner, 10 bits) | signs of the ray's direction in that frame (3 bits) | wide node
// index or gate index (19 bits)
#define RTNW_IDX_BITS 19
#define RTNW_TASK(slot, idx) (((uint32_t)(slot) << 22) | (uint32_t)(idx))
#define RTNW_TASK_SLOT(task) ((int)((task) >> 22))
#define RTNW_TASK_IDX(task) ((task) & ((1u << RTNW_IDX_BITS) - 1u))
#define RTNW_TASK_SIGNS(task) ((task) & (7u << RTNW_IDX_BITS))

// once per kernel, before the first closest-hit query (followed by a __syncthreads).
// `threadIdx.x % RTNW_BLOCK` here and in the other cooperative functions is threadIdx.x, but ptxas does not fold the modulo,
// and writing threadIdx.x changes the schedule of every kernel: the form stays until an A/B measurement says otherwise.
template <class SM>
__device__ __forceinline__ void coop_init(SM& sm) {
    const int tid = threadIdx.x % RTNW_BLOCK;
    if (tid < 3) { sm.n[tid] = 0; sm.lh[tid] = 0u; }
    if (tid == 3) { sm.lt = 0u; sm.overflow = 0; }
    if (tid >= 8 && tid < 16) sm.bins[tid - 8] = 0;
}

// Closest hit of the block's rays against the BVH item whose gate tree has root `root`.  Owners have already written
// their ray to sm.ray_* / sm.mkey and their running key to sm.key.  Called by all threads.
//
// One loop of rounds, two barriers per round.  In a round the first ceil(take/32) warps each take one node task per
// lane from the top of the stack; the remaining warps take one queued gate per lane (leaf->hit for its leaves), so
// thin node rounds are filled with leaf work instead of idling at the barrier; when the stack is empty all warps
// drain the gate queue.
template <bool COUNT, bool FAST, class SM>
__device__ __forceinline__ void coop_bvh_item(const scene_view& S, SM& sm, int nf, int root0, int root1, int tree_depth, bool active,
                                              float t_min, uint32_t k0, uint32_t k1, trav_counters& cnt, int& r3) {
    constexpr unsigned FULL = 0xffffffffu;
    constexpr int QN = SM::QN, QL = SM::QL;
    const int tid = threadIdx.x % RTNW_BLOCK;
    const unsigned lane = tid & 31u, lt_mask = (1u << lane) - 1u;
#ifdef RTNW_ROUND_STATS
    int stat_busy = 0, stat_small = 0; long long stat_c = 0; const long long stat_c0 = clock64();
#endif
    // The rounds of ALL items of a kernel form one sequence r = 0, 1, 2, ... (r3 = r % 3 lives in a register of every
    // thread).  Round r reads n[r3] / lh[r3], writes the popped state to buffer r3 + 1 and clears n[r3 + 2] — the buffer
    // the round before it read, which nobody looks at any more.  An item ends in a round that finds both queues empty;
    // the next item's root tasks then go to n[r3 + 1], cleared one round earlier, so entering an item needs no reset and no
    // barrier of its own: a thread still reading n[r3] / lh[r3] / lt of the final round never sees them change.
    if (tid == 0) sm.lh[r3] = sm.lt;  // empty ring; lh[r3] was last read three rounds ago
    {   // one task per ray and frame: the root of the gate tree of each of the nf (1 or 2) items traversed together
        const unsigned b = __ballot_sync(FULL, active);
        int base = 0;
        if (lane == 0 && b) base = atomicAdd(&sm.n[r3], __popc(b) * nf);
        base = __shfl_sync(FULL, base, 0);
        if (active) {
#pragma unroll
            for (int f = 0; f < SM::NFRAMES; ++f) {
                if (f < nf) {
                    const int v = f * RTNW_BLOCK + tid;
                    const float4 ri = sm.ray_i[v];  // written by this thread: which plane of a slab the ray meets first
                    const uint32_t sg = (ri.x < 0.f ? 1u : 0u) | (ri.y < 0.f ? 2u : 0u) | (ri.z < 0.f ? 4u : 0u);
                    sm.q[base + __popc(b & lt_mask) * nf + f] = RTNW_TASK(v, f ? root1 : root0) | (sg << RTNW_IDX_BITS);
                }
            }
        }
    }
    __syncthreads();
#pragma unroll 1
    for (;;) {
        const int nxt = r3 == 2 ? 0 : r3 + 1, prv = r3 == 0 ? 2 : r3 - 1;
        const int n = sm.n[r3];
        const unsigned lh = sm.lh[r3], ltail = sm.lt;
        const int queued = (int)(ltail - lh);
        if (tid == 0) sm.n[prv] = 0;
        if (n == 0 && queued == 0) { r3 = nxt; break; }
        // The round's plan is computed by ONE thread and read by the others after the barrier they wait at anyway: the
        // ~50 instructions of it cost issue slots in one warp instead of all ten (they were 14 % of all instructions).
        if (tid == 0) {
            const int room_ = (QN - n - 3 * tree_depth) / 3;
            const int take_ = (queued > QL - 4 * RTNW_BLOCK) ? 0 : min(min(n, RTNW_BLOCK), max(room_, 1));
            const int nt_ = (take_ + 31) & ~31;
            const int drain_ = min(queued, FAST ? RTNW_BLOCK - nt_ : (RTNW_BLOCK - nt_) >> 1);  // exact mode: two lanes per gate, one per leaf
            sm.plan = make_int4(take_, n - take_, nt_, drain_);
            sm.n[nxt] = n - take_; sm.lh[nxt] = lh + (unsigned)drain_;  // pop both
        }
        __syncthreads();
        const int4 pl = sm.plan;
        const int take = pl.x, base = pl.y, node_threads = pl.z, drain = pl.w;
        constexpr int LPG = FAST ? 1 : 2, LSH = FAST ? 0 : 1;  // lanes per gate: the fast mode's gates guard ONE leaf each
        uint32_t task = 0;
        if (tid < take) task = sm.q[base + tid];
        else if (tid >= node_threads && tid - node_threads < LPG * drain) task = sm.q[QN + ((lh + (unsigned)((tid - node_threads) >> LSH)) & (QL - 1))];
#ifdef RTNW_ROUND_STATS
        if (tid == 0) {
            RTNW_STAT(0, 1); RTNW_STAT(1, take); RTNW_STAT(2, drain); RTNW_STAT(8, n); RTNW_STAT(9, queued);
            if (take == 0) RTNW_STAT(3, 1);
            const int busy = node_threads + LPG * drain;
            RTNW_STAT(busy <= 64 ? 4 : busy <= 128 ? 5 : busy <= 192 ? 6 : 7, 1);
            stat_busy = busy; stat_c = clock64(); stat_small = n + LPG * queued <= 32 ? 1 : (n + LPG * queued <= 64 ? 2 : 0);
        }
#endif
        const int slot = RTNW_TASK_SLOT(task);  // virtual slot: the ray in its item's frame
        const int own = (SM::NFRAMES > 1 && slot >= RTNW_BLOCK) ? slot - RTNW_BLOCK : slot;  // the thread that owns the ray (key, medium key)
        if (tid < node_threads) {
            // ---- node warps: test the <= 4 child boxes of one wide node per lane, push what passed.  Straight-line code
            // (no short-circuit): the four slab tests are independent and interleave; a lane of the last node warp
            // without a task reads node 0 / slot 0 and masks its results.
            const bool live = tid < take;
            // The children this round pushes go to the stack slots this round pops ([base, base + take), stack discipline): every
            // node warp must have READ its task before any of them pushes.  They all read right after the plan barrier and push
            // hundreds of cycles later, so the order held by itself except about once in 10^8 warp-rounds, when a starved warp's
            // read came after another warp's push (found as 1 differing path in ~5 % of 1000x1000 frames).  A barrier among
            // the node warps alone, where they are still in step, makes it a guarantee.
            if (node_threads > 32) asm volatile("bar.sync 1, %0;" ::"r"(node_threads) : "memory");
            const float4* N = S.wnodes + 8 * (size_t)(live ? RTNW_TASK_IDX(task) : 0u);
            const float4 rf = __ldg(N + 6);
            const float4 ro = sm.ray_o[slot], ri = sm.ray_i[slot];
            const f3 o = mk3(ro.x, ro.y, ro.z), inv = mk3(ri.x, ri.y, ri.z);
            const int ref[4] = {__float_as_int(rf.x), __float_as_int(rf.y), __float_as_int(rf.z), __float_as_int(rf.w)};
            // RTNW_F_FAST_BVH: boxes are tested against the ray's closest hit SO FAR (any value read is a valid upper bound:
            // the key only ever decreases) instead of the un-narrowed range the reference hands down
            const float t_hi = FAST ? fminf(ro.w, key_t_or(sm.key[own], ro.w)) : ro.w;
            bool pass[4];
            // aabb::hit's swap of (t0, t1) when invD < 0 (PSC/aabb.h:41-42) picks, per axis, which of the min / max planes is met
            // first; the ray's three signs travel in the task word, so the near and far planes of the four boxes are simply
            // LOADED from the right rows of the node instead of selected value by value (24 selects per task).
            // aabb::hit (PSC/aabb.h:33-49, with r.origin(): F2): `tmin = t0 > tmin ? t0 : tmin` is fmaxf(t0, tmin) whenever tmin
            // is not NaN (a NaN t0, from 0 * inf, is ignored by both), likewise fminf for tmax; tmin starts finite, and a NaN
            // tmax (closest_so_far after a NaN rectangle hit) makes the reference accept every box, which the last term reproduces.
            const unsigned sg = task >> RTNW_IDX_BITS;
            const float4 nx4 = __ldg(N + ((sg & 1u) ? 3 : 0)), fx4 = __ldg(N + ((sg & 1u) ? 0 : 3));
            const float4 ny4 = __ldg(N + ((sg & 2u) ? 4 : 1)), fy4 = __ldg(N + ((sg & 2u) ? 1 : 4));
            const float4 nz4 = __ldg(N + ((sg & 4u) ? 5 : 2)), fz4 = __ldg(N + ((sg & 4u) ? 2 : 5));
#define RTNW_SLAB(c) (!(fminf(fminf(fminf((fx4.c - o.x) * inv.x, t_hi), (fy4.c - o.y) * inv.y), (fz4.c - o.z) * inv.z) <= \
                        fmaxf(fmaxf(fmaxf((nx4.c - o.x) * inv.x, t_min), (ny4.c - o.y) * inv.y), (nz4.c - o.z) * inv.z)) || (t_hi != t_hi))
            pass[0] = live & (ref[0] != RTNW_REF_NONE) & RTNW_SLAB(x);
            pass[1] = live & (ref[1] != RTNW_REF_NONE) & RTNW_SLAB(y);
            pass[2] = live & (ref[2] != RTNW_REF_NONE) & RTNW_SLAB(z);
            pass[3] = live & (ref[3] != RTNW_REF_NONE) & RTNW_SLAB(w);
#undef RTNW_SLAB
            if (COUNT && live) cnt.box_tests += (ref[0] != RTNW_REF_NONE) + (ref[1] != RTNW_REF_NONE) + (ref[2] != RTNW_REF_NONE) + (ref[3] != RTNW_REF_NONE);
            // warp-aggregated appends: wide nodes back onto the stack, gates to the gate ring
            unsigned bn[4], bl[4];
            int tn = 0, tl = 0;
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                bn[j] = __ballot_sync(FULL, pass[j] & (ref[j] >= 0));
                bl[j] = __ballot_sync(FULL, pass[j] & (ref[j] < 0));
                tn += __popc(bn[j]); tl += __popc(bl[j]);
            }
            int base_n = 0;
            unsigned base_l = 0;
            if (lane == 0) {
                if (tn) base_n = atomicAdd(&sm.n[nxt], tn);
                if (tl) base_l = atomicAdd(&sm.lt, (unsigned)tl);
            }
            base_n = __shfl_sync(FULL, base_n, 0);
            base_l = __shfl_sync(FULL, base_l, 0);
            const bool ring_ok = (int)(base_l + (unsigned)tl - lh) <= QL;  // never laps the unconsumed part of the ring
            bool ok = true;
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const bool isn = ref[j] >= 0;
                const int at_n = base_n + __popc(bn[j] & lt_mask);
                const int at_l = QN + (int)((base_l + (unsigned)__popc(bl[j] & lt_mask)) & (unsigned)(QL - 1));
                const bool fits = isn ? at_n < QN : ring_ok;
                if (pass[j] & fits) sm.q[isn ? at_n : at_l] = RTNW_TASK(slot, isn ? ref[j] : ~ref[j]) | RTNW_TASK_SIGNS(task);
                ok &= !pass[j] | fits;
                base_n += __popc(bn[j]); base_l += (unsigned)__popc(bl[j]);
            }
            if (!ok) sm.overflow = 1;
        } else if (tid - node_threads < LPG * drain) {
            // ---- gate lanes: leaf->hit(r, tmin, tmax0) for the one or two leaves the gate guards, one lane per leaf (a leaf
            // test is about as long as a node task; a round lasts as long as its slowest lane)
            const int2 g = __ldg(&S.gates[RTNW_TASK_IDX(task)]);
            const int leaf = (!FAST && (tid & 1)) ? g.y : g.x;  // node_threads is even: lane parity = leaf of the gate
            hkey_t k = RTNW_KEY_NONE;
            if (leaf >= 0) {
                const float4 A0 = __ldg(&S.recs[leaf].a), B0 = __ldg(&S.recs[leaf].b);
                const float4 ro = sm.ray_o[slot], rd = sm.ray_d[slot], ri = sm.ray_i[slot];
                const uint4 mq = sm.mkey[own];
                ray_t r; r.o = mk3(ro.x, ro.y, ro.z); r.d = mk3(rd.x, rd.y, rd.z); r.time = __uint_as_float(mq.w);
                ray_recip rr; rr.inv = mk3(ri.x, ri.y, ri.z); rr.inv_a = ri.w;
                medium_key mk; mk.k0 = k0; mk.k1 = k1; mk.pixel = mq.x; mk.sample = mq.y; mk.depth = mq.z;
                const float t_hi = FAST ? fminf(ro.w, key_t_or(sm.key[own], ro.w)) : ro.w;
                // nearly every leaf is ONE plain box or sphere record (no transform chain, not a list, not a medium): those skip
                // the record loop and the kind switch of the general leaf test — the same hit function, the same key
                const uint32_t plain = __float_as_uint(B0.z) & ~(uint32_t)RTNW_TAG_FLIP;
                if (plain == (K_BOX | RTNW_TAG_LAST)) {
                    float t; int face = 0;
                    if (COUNT) cnt.prim_tests++;
                    if (hit_box<ARITH_RECIP>(mk3(A0.x, A0.y, A0.z), mk3(A0.w, B0.x, B0.y), r, rr, t_min, t_hi, t, face)) k = make_key(t, leaf, face);
                } else if (plain == (K_SPHERE | RTNW_TAG_LAST)) {
                    float t;
                    if (COUNT) cnt.prim_tests++;
                    if (hit_sphere_recip(mk3(A0.x, A0.y, A0.z), A0.w, r, rd.w, rr.inv_a, t_min, t_hi, t)) k = make_key(t, leaf, 0);
                } else {
                    k = test_leaf<COUNT, ARITH_RECIP>(S, leaf, A0, B0, r, rd.w, rr, t_min, t_hi, mk, cnt);
                }
            }
            if (k != RTNW_KEY_NONE) atomicMin(&sm.key[own], k);
        }
        __syncthreads();
        r3 = nxt;
#ifdef RTNW_ROUND_STATS
        if (tid == 0) { const long long d = clock64() - stat_c; RTNW_STAT(stat_busy <= 64 ? 15 : stat_busy <= 128 ? 16 : stat_busy <= 192 ? 17 : 18, d); if (stat_small == 1) { RTNW_STAT(19, 1); RTNW_STAT(20, d); } else if (stat_small == 2) { RTNW_STAT(21, 1); RTNW_STAT(22, d); } }
#endif
    }
#ifdef RTNW_ROUND_STATS
    if (tid == 0) RTNW_STAT(14, clock64() - stat_c0);
#endif
}

// world->hit(r, t_min, t_max, rec) (PSC/main.cpp:27) for the rays of the block.  Must be called by all threads; a
// thread without a ray passes active = false and still works on the other threads' BVH tasks.
// One element of the top-level list that is a plain list of primitives: scanned by each owner in lockstep.
template <bool COUNT>
__device__ __forceinline__ void scan_list_item(const scene_view& S, int i, int next, const ray_t& r, float a, float t_min, float best_t,
                                               const medium_key& mk, hkey_t& key, trav_counters& cnt) {
    float lim = best_t;
#pragma unroll 1
    for (int j = i + 1; j < next;) {
        const float4 A = __ldg(&S.recs[j].a), B = __ldg(&S.recs[j].b);
        const uint32_t rk = __float_as_uint(B.z) & 15u;
        if (rk >= K_RUN_SPHERE) {  // a run header (uniform over the block): the specialised loop takes the next A.x records
            const int nrec = __float_as_int(A.x);
            if (rk == K_RUN_SPHERE) scan_run<COUNT, K_RUN_SPHERE>(S, j + 1, nrec, r, a, t_min, lim, key, cnt);
            else if (rk == K_RUN_SPHERELIKE) scan_run<COUNT, K_RUN_SPHERELIKE>(S, j + 1, nrec, r, a, t_min, lim, key, cnt);
            else scan_run<COUNT, K_RUN_BOX>(S, j + 1, nrec, r, a, t_min, lim, key, cnt);
            j += 1 + nrec;
            continue;
        }
        // plain records (no transform chain) skip the record dispatch: same test, same narrowing, same key
        const uint32_t plain = __float_as_uint(B.z) & ~(uint32_t)(RTNW_TAG_FLIP | RTNW_TAG_CONT | RTNW_TAG_LAST);
        if (plain == K_SPHERE) {
            float t;
            if (COUNT) cnt.prim_tests++;
            if (hit_sphere(mk3(A.x, A.y, A.z), A.w, r, a, t_min, lim, t)) { lim = t; key = make_key(t, j, 0); }
            ++j;
            continue;
        }
        if (plain >= K_RECT_XY && plain <= K_RECT_YZ) {
            float t;
            if (COUNT) cnt.prim_tests++;
            const bool hit = plain == K_RECT_XY   ? hit_rect<2, 0, 1>(A.x, A.y, A.z, A.w, B.x, r, t_min, lim, t)
                             : plain == K_RECT_XZ ? hit_rect<1, 0, 2>(A.x, A.y, A.z, A.w, B.x, r, t_min, lim, t)
                                                  : hit_rect<0, 1, 2>(A.x, A.y, A.z, A.w, B.x, r, t_min, lim, t);
            if (hit) { lim = t; key = make_key(t, j, 0); }
            ++j;
            continue;
        }
        if (plain == K_MSPHERE) {
            float t;
            if (COUNT) cnt.prim_tests++;
            const float4 A2 = __ldg(&S.recs[j + 1].a);
            if (hit_sphere(moving_center(mk3(A.x, A.y, A.z), mk3(A2.x, A2.y, A2.z), B.x, B.y, r.time), A.w, r, a, t_min, lim, t)) { lim = t; key = make_key(t, j, 0); }
            j += 2;
            continue;
        }
        bool hit; float t; int face;
        const int step = test_record<COUNT>(S, j, A, B, r, a, t_min, lim, mk, hit, t, face, cnt);
        if (hit) { lim = t; key = make_key(t, j, face); }  // list narrowing: an accepted hit is the new closest
        j += step;
    }
}

template <bool COUNT, bool FAST, class SM>
__device__ __forceinline__ hkey_t coop_closest_hit(const scene_view& S, SM& sm, const ray_t& wr, bool active,
                                                   float t_min, float t_max, const medium_key& mk, trav_counters& cnt, int& r3) {
    const int tid = threadIdx.x % RTNW_BLOCK;
    sm.key[tid] = RTNW_KEY_NONE;
    sm.mkey[tid] = make_uint4(mk.pixel, mk.sample, mk.depth, __float_as_uint(wr.time));
    if (!FAST) {
        int i = 0;
        for (;;) {  // the elements of the top-level hitable_list, in order (PSC/hitable_list.h:24-30); uniform over the block
            const float4 IA = __ldg(&S.recs[i].a), IB = __ldg(&S.recs[i].b);
            const uint32_t tag = __float_as_uint(IB.z);
            if ((tag & 15u) != K_ITEM) break;  // K_END
            const int next = __float_as_int(IA.x);
            hkey_t key = sm.key[tid];
            const float best_t = key_t_or(key, t_max);  // closest_so_far: the t_max this element receives
            ray_t r = wr;
            xform_ray(S.xforms, tag >> 8, r);
            const float a = dot(r.d, r.d);
            if (__float_as_int(IB.w) == RTNW_ITEM_BVH) {
                sm.ray_o[tid] = make_float4(r.o.x, r.o.y, r.o.z, best_t);
                sm.ray_d[tid] = make_float4(r.d.x, r.d.y, r.d.z, a);
                sm.ray_i[tid] = make_float4(1.0f / r.d.x, 1.0f / r.d.y, 1.0f / r.d.z, 1.0f / a);
                coop_bvh_item<COUNT, false, SM>(S, sm, 1, __float_as_int(IA.y), 0, __float_as_int(IA.z), active, t_min, mk.k0, mk.k1, cnt, r3);
            } else if (active) {
                scan_list_item<COUNT>(S, i, next, r, a, t_min, best_t, mk, key, cnt);
                sm.key[tid] = key;
            }
            i = next;
        }
    } else {
        // RTNW_F_FAST_BVH.  The closest hit does not depend on the order in which the elements of the list are examined
        // (except among candidates of equal t), only the reference's TEST SET does: an element is handed the closest hit of
        // the elements before it as its t_max.  The fast mode gives that up: first every plain element (narrowing as usual),
        // then the BVH elements TWO AT A TIME in one cooperative traversal, each ray present once per item frame — half the
        // rounds of the latency chain for a scene with two BVHs — and boxes / leaves tested against the running closest hit.
        for (int i = 0;;) {
            const float4 IA = __ldg(&S.recs[i].a), IB = __ldg(&S.recs[i].b);
            const uint32_t tag = __float_as_uint(IB.z);
            if ((tag & 15u) != K_ITEM) break;
            const int next = __float_as_int(IA.x);
            if (__float_as_int(IB.w) != RTNW_ITEM_BVH && active) {
                hkey_t key = sm.key[tid];
                ray_t r = wr;
                xform_ray(S.xforms, tag >> 8, r);
                scan_list_item<COUNT>(S, i, next, r, dot(r.d, r.d), t_min, key_t_or(key, t_max), mk, key, cnt);
                sm.key[tid] = key;
            }
            i = next;
        }
        int nf = 0, root0 = 0, root1 = 0, depth = 0;
        for (int i = 0;;) {
            const float4 IA = __ldg(&S.recs[i].a), IB = __ldg(&S.recs[i].b);
            const uint32_t tag = __float_as_uint(IB.z);
            const bool end = (tag & 15u) != K_ITEM;
            if (!end && __float_as_int(IB.w) == RTNW_ITEM_BVH) {
                ray_t r = wr;
                xform_ray(S.xforms, tag >> 8, r);
                const int v = nf * RTNW_BLOCK + tid;
                sm.ray_o[v] = make_float4(r.o.x, r.o.y, r.o.z, key_t_or(sm.key[tid], t_max));
                const float a = dot(r.d, r.d);
                sm.ray_d[v] = make_float4(r.d.x, r.d.y, r.d.z, a);
                sm.ray_i[v] = make_float4(1.0f / r.d.x, 1.0f / r.d.y, 1.0f / r.d.z, 1.0f / a);
                if (nf == 0) root0 = __float_as_int(IA.w); else root1 = __float_as_int(IA.w);  // the trees over the leaves' own boxes
                depth = max(depth, __float_as_int(IB.x));
                ++nf;
            }
            if (nf == SM::NFRAMES || (end && nf > 0)) {
                coop_bvh_item<COUNT, true, SM>(S, sm, nf, root0, root1, depth, active, t_min, mk.k0, mk.k1, cnt, r3);
                nf = 0; depth = 0;
            }
            if (end) break;
            i = __float_as_int(IA.x);
        }
    }
    __syncthreads();  // nobody may overwrite sm.key before every owner has read its result
    const hkey_t out = sm.key[tid];
    __syncthreads();
    return out;
}

__device__ __forceinline__ void key_to_hit(const scene_view& S, hkey_t key, float t_max, hit_t& h) {
    if (key == RTNW_KEY_NONE) { h.rec = -1; h.t = t_max; h.face = 0; h.xf = 0; return; }
    h.rec = key_rec(key);
    h.face = key_face(key);
    h.t = order_float((uint32_t)(key >> 32));
    h.xf = __ldg(&S.rec_xf[h.rec]);
}

// PSC/hitable.h:14-19
__device__ __forceinline__ void get_sphere_uv(f3 p, float& u, float& v) {
    const float phi = atan2f(p.z, p.x);
    const float theta = asinf(p.y);
    u = (float)(1.0 - ((double)phi + M_PI) / (2.0 * M_PI));
    v = (float)(((double)theta + M_PI / 2.0) / M_PI);
}

struct surf_t { f3 p, n; float u, v; int mat; };

// Rebuild the hit_record of the winning record: p / normal / uv are pure functions of (ray, primitive, t), so the
// traversal only tracks (t, record) and the record is evaluated once here.
// want_uv: the spherical (u,v) of PSC/hitable.h:14-19 costs an atan2f, an asinf and two double divisions, and only
// image_texture::value reads u,v; the renderer asks for it only when the hit material's texture is an image.
__device__ __forceinline__ void finish_hit(const scene_view& S, const ray_t& wr, hit_t& h, surf_t& s, bool want_uv = true) {
    const float4 A = __ldg(&S.recs[h.rec].a), B = __ldg(&S.recs[h.rec].b);
    const uint32_t tag = __float_as_uint(B.z);
    const uint32_t kind = tag & 15u, chain = tag >> 8;
    ray_t r = wr;
    xform_ray(S.xforms, h.xf, r);
    xform_ray(S.xforms, chain, r);
    const float t = h.t;
    s.p = r.o + t * r.d;  // ray::point_at_parameter, PSC/ray.h:18
    s.u = 0.f; s.v = 0.f;  // the reference leaves u,v unwritten for moving spheres and media (SURVEY F5)
    s.mat = __float_as_int(B.w);
    bool flip = (tag & RTNW_TAG_FLIP) != 0;
    switch (kind) {
        case K_SPHERE: {
            s.n = (s.p - mk3(A.x, A.y, A.z)) / A.w;
            if (want_uv) get_sphere_uv(s.n, s.u, s.v);
            break;
        }
        case K_MSPHERE: {
            const float4 A2 = __ldg(&S.recs[h.rec + 1].a);
            const f3 c = moving_center(mk3(A.x, A.y, A.z), mk3(A2.x, A2.y, A2.z), B.x, B.y, r.time);
            s.n = (s.p - c) / A.w;
            break;
        }
        case K_RECT_XY: s.u = (s.p.x - A.x) / (A.y - A.x); s.v = (s.p.y - A.z) / (A.w - A.z); s.n = mk3(0, 0, 1); break;
        case K_RECT_XZ: s.u = (s.p.x - A.x) / (A.y - A.x); s.v = (s.p.z - A.z) / (A.w - A.z); s.n = mk3(0, 1, 0); break;
        case K_RECT_YZ: s.u = (s.p.y - A.x) / (A.y - A.x); s.v = (s.p.z - A.z) / (A.w - A.z); s.n = mk3(1, 0, 0); break;
        case K_BOX: {
            const f3 p0 = mk3(A.x, A.y, A.z), p1 = mk3(A.w, B.x, B.y);
            const int axis = h.face >> 1;  // 0: xy faces, 1: xz faces, 2: yz faces
            if (axis == 0) { s.u = (s.p.x - p0.x) / (p1.x - p0.x); s.v = (s.p.y - p0.y) / (p1.y - p0.y); s.n = mk3(0, 0, 1); }
            else if (axis == 1) { s.u = (s.p.x - p0.x) / (p1.x - p0.x); s.v = (s.p.z - p0.z) / (p1.z - p0.z); s.n = mk3(0, 1, 0); }
            else { s.u = (s.p.y - p0.y) / (p1.y - p0.y); s.v = (s.p.z - p0.z) / (p1.z - p0.z); s.n = mk3(1, 0, 0); }
            if (h.face & 1) flip = !flip;  // faces 1,3,5 are flip_normals(rect), PSC/box.h:29-33
            break;
        }
        default: s.n = mk3(1, 0, 0); break;  // K_MEDIUM: "arbitrary", PSC/constant_medium.h:44
    }
    if (flip) s.n = -s.n;
    xform_hit_back(S.xforms, chain, s.p, s.n);
    xform_hit_back(S.xforms, h.xf, s.p, s.n);
}

// ------------------------------------------------------------------------------------------------ textures
// PSC/perlin.h:25-61.  noise() smooths u,v,w and perlin_interp smooths them again (and uses the smoothed u in
// weight_v) — reproduced as written.
__device__ __forceinline__ float perlin_noise(const scene_view& S, f3 p) {
    const float fx = floorf(p.x), fy = floorf(p.y), fz = floorf(p.z);
    float u = p.x - fx, v = p.y - fy, w = p.z - fz;
    u = u * u * (3.f - 2.f * u);
    v = v * v * (3.f - 2.f * v);
    w = w * w * (3.f - 2.f * w);
    const int i = (int)fx, j = (int)fy, k = (int)fz;
    const float uu = u * u * (3.f - 2.f * u);
    const float vv = v * v * (3.f - 2.f * v);
    const float ww = w * w * (3.f - 2.f * w);
    uint32_t hx[2], hy[2], hz[2];
#pragma unroll
    for (int d = 0; d < 2; ++d) {
        hx[d] = __ldg(&S.perm[(i + d) & 255]);
        hy[d] = __ldg(&S.perm[256 + ((j + d) & 255)]);
        hz[d] = __ldg(&S.perm[512 + ((k + d) & 255)]);
    }
    float accum = 0.f;
#pragma unroll
    for (int di = 0; di < 2; ++di)
#pragma unroll
        for (int dj = 0; dj < 2; ++dj)
#pragma unroll
            for (int dk = 0; dk < 2; ++dk) {
                const float4 c = __ldg(&S.ranvec[hx[di] ^ hy[dj] ^ hz[dk]]);
                const f3 weight_v = mk3(u - (float)di, v - (float)dj, w - (float)dk);
                accum += ((float)di * uu + (float)(1 - di) * (1.f - uu)) *
                         ((float)dj * vv + (float)(1 - dj) * (1.f - vv)) *
                         ((float)dk * ww + (float)(1 - dk) * (1.f - ww)) * dot(mk3(c.x, c.y, c.z), weight_v);
            }
    return accum;
}
// PSC/perlin.h:64-74
__device__ __forceinline__ float perlin_turb(const scene_view& S, f3 p) {
    float accum = 0.f, weight = 1.0f;
    f3 q = p;
#pragma unroll 1
    for (int o = 0; o < 7; ++o) {
        accum += weight * perlin_noise(S, q);
        weight *= 0.5f;
        q = 2.f * q;
    }
    return fabsf(accum);
}

// README.md:516-630: the Chapter 4 noise functions that preceded perlin.h's shipped form (RTNW_TEX_NOISE_HASH / _TRILINEAR /
// _HERMITE); `ranfloat[i]` is S.ranvec[i].x.  Operation order as in the reference's trilinear_interp (PSC/perlin.h:11-23).
__device__ __forceinline__ float readme_noise(const scene_view& S, uint32_t kind, f3 p) {
    if (kind == RTNW_TEX_NOISE_HASH) {
        const int i = (int)(4.f * p.x) & 255, j = (int)(4.f * p.y) & 255, k = (int)(4.f * p.z) & 255;
        return __ldg(&S.ranvec[__ldg(&S.perm[i]) ^ __ldg(&S.perm[256 + j]) ^ __ldg(&S.perm[512 + k])]).x;
    }
    const float fx = floorf(p.x), fy = floorf(p.y), fz = floorf(p.z);
    float u = p.x - fx, v = p.y - fy, w = p.z - fz;
    if (kind == RTNW_TEX_NOISE_HERMITE) {
        u = u * u * (3.f - 2.f * u);
        v = v * v * (3.f - 2.f * v);
        w = w * w * (3.f - 2.f * w);
    }
    const int i = (int)fx, j = (int)fy, k = (int)fz;
    float accum = 0.f;
#pragma unroll
    for (int di = 0; di < 2; ++di)
#pragma unroll
        for (int dj = 0; dj < 2; ++dj)
#pragma unroll
            for (int dk = 0; dk < 2; ++dk) {
                const float c = __ldg(&S.ranvec[__ldg(&S.perm[(i + di) & 255]) ^ __ldg(&S.perm[256 + ((j + dj) & 255)]) ^ __ldg(&S.perm[512 + ((k + dk) & 255)])]).x;
                accum += ((float)di * u + (float)(1 - di) * (1.f - u)) * ((float)dj * v + (float)(1 - dj) * (1.f - v)) *
                         ((float)dk * w + (float)(1 - dk) * (1.f - w)) * c;
            }
    return accum;
}

// texture::value(u, v, p): PSC/texture.h:22-56, PSC/surface_texture.h:19-30
__device__ __forceinline__ f3 texture_value(const scene_view& S, int tex, float u, float v, f3 p) {
    for (;;) {
        const float4 t0 = __ldg(reinterpret_cast<const float4*>(S.textures + tex));      // kind, i0, i1, i2
        const float4 t1 = __ldg(reinterpret_cast<const float4*>(S.textures + tex) + 1);  // c[3], pad
        const uint32_t kind = __float_as_uint(t0.x);
        if (kind == RTNW_TEX_CONSTANT) return mk3(t1.x, t1.y, t1.z);
        if (kind == RTNW_TEX_CHECKER) {
            const float sines = sinf(10.f * p.x) * sinf(10.f * p.y) * sinf(10.f * p.z);
            tex = sines < 0.f ? __float_as_int(t0.z) /* odd */ : __float_as_int(t0.y) /* even */;
            continue;
        }
        if (kind >= RTNW_TEX_NOISE_HASH) {
            const float n = readme_noise(S, kind, p);
            return mk3(n, n, n);  // vec3(1,1,1) * noise(p)
        }
        if (kind == RTNW_TEX_NOISE) {
            const float scale = t1.x;
            const float s = 1.f + sinf(scale * p.x + 5.f * perlin_turb(S, scale * p));
            return mk3(0.5f * s, 0.5f * s, 0.5f * s);  // vec3(1,1,1)*0.5 = (0.5,0.5,0.5) exactly, then * s
        }
        // image: nearest texel, flipped u and v
        const int off = __float_as_int(t0.y), nx = __float_as_int(t0.z), ny = __float_as_int(t0.w);
        if (__float_as_uint(t1.w) & RTNW_TEXF_BILINEAR) {  // option (not in the reference): blend the four texels around (u, v)
            const float fx = (1.f - u) * (float)nx - 0.5f, fy = (1.f - v) * (float)ny - 0.5f;
            const float x0 = floorf(fx), y0 = floorf(fy);
            const float wx = fx - x0, wy = fy - y0;
            const int i0 = min(max((int)x0, 0), nx - 1), i1 = min(max((int)x0 + 1, 0), nx - 1);
            const int j0 = min(max((int)y0, 0), ny - 1), j1 = min(max((int)y0 + 1, 0), ny - 1);
            f3 c[4];
            const int ii[4] = {i0, i1, i0, i1}, jj[4] = {j0, j0, j1, j1};
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                const uint8_t* px = S.images + off + 3 * ii[q] + 3 * nx * jj[q];
                c[q] = mk3((float)__ldg(px) / 255.0f, (float)__ldg(px + 1) / 255.0f, (float)__ldg(px + 2) / 255.0f);
            }
            const f3 top = (1.f - wx) * c[0] + wx * c[1], bot = (1.f - wx) * c[2] + wx * c[3];
            return (1.f - wy) * top + wy * bot;
        }
        int i = (int)((1.f - u) * (float)nx);
        int j = (int)((double)((1.f - v) * (float)ny) - 0.001);
        if (i < 0) i = 0;
        if (j < 0) j = 0;
        if (i > nx - 1) i = nx - 1;
        if (j > ny - 1) j = ny - 1;
        const uint8_t* px = S.images + off + 3 * i + 3 * nx * j;
        return mk3((float)__ldg(px) / 255.0f, (float)__ldg(px + 1) / 255.0f, (float)__ldg(px + 2) / 255.0f);
    }
}

// ------------------------------------------------------------------------------------------------ materials
// PSC/material.h:16-20: float r0; the return expression is evaluated in double (pow(float,int) promotes)
__device__ __forceinline__ float schlick(float cosine, float ref_idx) {
    float r0 = (1.f - ref_idx) / (1.f + ref_idx);
    r0 = r0 * r0;
    const double x = (double)(1.f - cosine);
    const double x2 = x * x;
    return (float)((double)r0 + (double)(1.f - r0) * (x2 * x2 * x));
}
// PSC/material.h:23-33
__device__ __forceinline__ bool refract(f3 v, f3 n, float ni_over_nt, f3& refracted) {
    const f3 uv = unit_vector(v);
    const float dt = dot(uv, n);
    const float disc = 1.0f - ni_over_nt * ni_over_nt * (1.f - dt * dt);
    if (disc > 0.f) {
        refracted = ni_over_nt * (uv - dt * n) - sqrtf(disc) * n;
        return true;
    }
    return false;
}
__device__ __forceinline__ f3 reflect(f3 v, f3 n) { return v - (2.f * dot(v, n)) * n; }  // PSC/material.h:36-38

// material::emitted(u,v,p), PSC/material.h:56-57,134-136
__device__ __forceinline__ f3 material_emitted(const scene_view& S, int mat, float u, float v, f3 p) {
    const float4 m0 = __ldg(reinterpret_cast<const float4*>(S.materials + mat));
    if (__float_as_uint(m0.x) != RTNW_MAT_DIFFUSE_LIGHT) return mk3(0.f, 0.f, 0.f);
    return texture_value(S, __float_as_int(m0.y), u, v, p);
}
// material::scatter(r_in, rec, attenuation, scattered), PSC/material.h:64-149.  lambertian, metal and isotropic each
// draw exactly one random_in_unit_sphere() and nothing else, and two of them end with one texture lookup, so both are
// evaluated at a single site (draw order inside each material is unchanged: reflect() and value() draw nothing).
__device__ __forceinline__ bool material_scatter(const scene_view& S, int mat, const ray_t& r_in, const surf_t& s, rng_t& g,
                                                 f3& attenuation, ray_t& scattered) {
    const float4 m0 = __ldg(reinterpret_cast<const float4*>(S.materials + mat));      // kind, tex, f, pad
    const uint32_t kind = __float_as_uint(m0.x);
    if (kind == RTNW_MAT_DIFFUSE_LIGHT) return false;
    scattered.o = s.p;
    if (kind == RTNW_MAT_DIELECTRIC) {
        const float ref_idx = m0.z;
        f3 outward_normal;
        const f3 reflected = reflect(r_in.d, s.n);
        float ni_over_nt, reflect_prob, cosine;
        attenuation = mk3(1.f, 1.f, 1.f);
        f3 refracted = mk3(0.f, 0.f, 0.f);
        const float dn = dot(r_in.d, s.n);
        if (dn > 0.f) {
            outward_normal = -s.n;
            ni_over_nt = ref_idx;
            cosine = dn / length(r_in.d);
            cosine = sqrtf(1.f - ref_idx * ref_idx * (1.f - cosine * cosine));
        } else {
            outward_normal = s.n;
            ni_over_nt = 1.0f / ref_idx;
            cosine = -dn / length(r_in.d);
        }
        if (refract(r_in.d, outward_normal, ni_over_nt, refracted)) reflect_prob = schlick(cosine, ref_idx);
        else reflect_prob = 1.0f;
        scattered.time = 0.f;
        scattered.d = (g.draw() < reflect_prob) ? reflected : refracted;
        return true;
    }
    const f3 rs = random_in_unit_sphere(g);
    if (kind == RTNW_MAT_METAL) {
        const float4 m1 = __ldg(reinterpret_cast<const float4*>(S.materials + mat) + 1);  // albedo
        const f3 reflected = reflect(unit_vector(r_in.d), s.n);
        scattered.d = reflected + m0.z * rs;
        scattered.time = 0.f;
        attenuation = mk3(m1.x, m1.y, m1.z);
        return dot(scattered.d, s.n) > 0.f;
    }
    if (kind == RTNW_MAT_LAMBERTIAN) {
        const f3 target = s.p + s.n + rs;
        scattered.d = target - s.p;
        scattered.time = r_in.time;
    } else {  // isotropic
        scattered.d = rs;
        scattered.time = 0.f;
    }
    attenuation = texture_value(S, __float_as_int(m0.y), s.u, s.v, s.p);
    return true;
}

// ------------------------------------------------------------------------------------------------ light sampling
// RTNW_F_LIGHT_SAMPLING (include/rtnw.h): a light of the table is two float4, a = {a0, a1, b0, b1} (rectangle) or {cx, cy, cz, r}
// (sphere), b = {plane offset k, area, kind bits, record bits}.  tests/light_oracle.c restates these functions draw for draw.
__device__ __forceinline__ f3 cross(f3 a, f3 b) { return mk3(a.y * b.z - a.z * b.y, a.z * b.x - a.x * b.z, a.x * b.y - a.y * b.x); }

// p_k(e): the solid-angle density with which light k samples the unit direction e from p; 0 where the ray (p, e) misses it
template <int N, int A, int B>
__device__ __forceinline__ float rect_pdf(float4 la, float4 lb, f3 p, f3 e) {
    const float* o = &p.x;
    const float* d = &e.x;
    const float t = (lb.x - o[N]) / d[N];
    if (!(t > 0.f)) return 0.f;
    const float a = o[A] + t * d[A], b = o[B] + t * d[B];
    if (a < la.x || a > la.y || b < la.z || b > la.w) return 0.f;
    return t * t / (fabsf(d[N]) * lb.y);
}
__device__ __forceinline__ float light_pdf(const float4* __restrict__ lights, int k, f3 p, f3 e) {
    const float4 la = __ldg(&lights[2 * k]), lb = __ldg(&lights[2 * k + 1]);
    switch (__float_as_int(lb.z)) {
        case RTNW_PRIM_RECT_XY: return rect_pdf<2, 0, 1>(la, lb, p, e);
        case RTNW_PRIM_RECT_XZ: return rect_pdf<1, 0, 2>(la, lb, p, e);
        case RTNW_PRIM_RECT_YZ: return rect_pdf<0, 1, 2>(la, lb, p, e);
        default: {  // sphere: uniform in the cone it subtends
            const f3 oc = mk3(la.x, la.y, la.z) - p;
            const float d2 = dot(oc, oc), r2 = la.w * la.w;
            if (!(d2 > r2)) return 0.f;
            const float cmax = sqrtf(1.f - r2 / d2);
            if (!(dot(e, unit_vector(oc)) >= cmax)) return 0.f;
            return 1.f / (6.28318531f * (1.f - cmax));
        }
    }
}
// a unit direction towards light k from p for the draws (u1, u2); false when p is inside or on a sphere light
__device__ __forceinline__ bool sample_light(const float4* __restrict__ lights, int k, f3 p, float u1, float u2, f3& d) {
    const float4 la = __ldg(&lights[2 * k]), lb = __ldg(&lights[2 * k + 1]);
    const int kind = __float_as_int(lb.z);
    if (kind != RTNW_PRIM_SPHERE) {
        const float a = la.x + u1 * (la.y - la.x), b = la.z + u2 * (la.w - la.z);
        const f3 q = kind == RTNW_PRIM_RECT_XY ? mk3(a, b, lb.x) : (kind == RTNW_PRIM_RECT_XZ ? mk3(a, lb.x, b) : mk3(lb.x, a, b));
        d = unit_vector(q - p);  // unit length like the sphere's: the scattered ray's t_min stays a distance of ~0.001, as in the reference branch
        return true;
    }
    const f3 oc = mk3(la.x, la.y, la.z) - p;
    const float d2 = dot(oc, oc), r2 = la.w * la.w;
    if (!(d2 > r2)) return false;
    const float cmax = sqrtf(1.f - r2 / d2);
    const float z = 1.f + u2 * (cmax - 1.f), phi = 6.28318531f * u1, s = sqrtf(1.f - z * z);
    const f3 w = unit_vector(oc);
    const f3 v = unit_vector(cross(w, fabsf(w.x) > 0.9f ? mk3(0.f, 1.f, 0.f) : mk3(1.f, 0.f, 0.f)));
    const f3 u = cross(w, v);
    d = (cosf(phi) * s) * u + (sinf(phi) * s) * v + z * w;
    return true;
}
// the same with the next two draws of the path's stream
__device__ __forceinline__ bool sample_light(const float4* __restrict__ lights, int k, f3 p, rng_t& g, f3& d) {
    const float u1 = g.draw(), u2 = g.draw();
    return sample_light(lights, k, p, u1, u2, d);
}
// material_scatter with the one-sample light mixture for lambertian and isotropic bounces (n_lights > 0, RTNW_F_EMIT on)
__device__ __forceinline__ bool mixture_scatter(const scene_view& S, const float4* __restrict__ lights, int n_lights, int mat,
                                                const ray_t& r_in, const surf_t& s, rng_t& g, f3& attenuation, ray_t& scattered) {
    const float4 m0 = __ldg(reinterpret_cast<const float4*>(S.materials + mat));
    const uint32_t kind = __float_as_uint(m0.x);
    const bool mix = kind == RTNW_MAT_LAMBERTIAN || kind == RTNW_MAT_ISOTROPIC;
    const float u = mix ? g.draw() : 1.f;
    if (u < 0.5f) {  // light branch
        const int k = min((int)(2.f * u * (float)n_lights), n_lights - 1);
        if (!sample_light(lights, k, s.p, g, scattered.d)) return false;
        scattered.o = s.p;
        scattered.time = kind == RTNW_MAT_LAMBERTIAN ? r_in.time : 0.f;
        attenuation = texture_value(S, __float_as_int(m0.y), s.u, s.v, s.p);
    } else if (!material_scatter(S, mat, r_in, s, g, attenuation, scattered)) {
        return false;
    }
    if (!mix) return true;
    const f3 e = unit_vector(scattered.d);
    float p_ref = 0.0795774715f;  // isotropic: 1 / (4 pi)
    if (kind == RTNW_MAT_LAMBERTIAN) {
        const float c = dot(e, s.n);
        if (!(c > 0.f)) return false;
        p_ref = c * c * c * 0.636619772f;  // (2 / pi) cos^3
    }
    float sum = 0.f;
#pragma unroll 1
    for (int k = 0; k < n_lights; ++k) sum += light_pdf(lights, k, s.p, e);
    const float w = p_ref / (0.5f * p_ref + 0.5f * (sum / (float)n_lights));
    attenuation = w * attenuation;
    return true;
}

// ------------------------------------------------------------------------------------------------ next-event estimation
// RTNW_F_NEXT_EVENT (include/rtnw.h), restated operation for operation by tests/nee_oracle.c.
// p_ref(e) of a lambertian (normal n) or isotropic vertex for the unit direction e
__device__ __forceinline__ float ref_density(bool lambertian, f3 n, f3 e) {
    if (!lambertian) return 0.0795774715f;  // 1 / (4 pi)
    const float c = dot(e, n);
    return c > 0.f ? c * c * c * 0.636619772f : 0.f;  // (2 / pi) cos^3
}
// p_L(e): the mean of the lights' densities, summed in table order
__device__ __forceinline__ float lights_density(const float4* __restrict__ lights, int n_lights, f3 p, f3 e) {
    float sum = 0.f;
#pragma unroll 1
    for (int k = 0; k < n_lights; ++k) sum += light_pdf(lights, k, p, e);
    return sum / (float)n_lights;
}
// is record rec one of the light table's (n_lights <= RTNW_MAX_LIGHTS)
__device__ __forceinline__ bool is_light_record(const float4* __restrict__ lights, int n_lights, int rec) {
#pragma unroll 1
    for (int k = 0; k < n_lights; ++k)
        if (__float_as_int(__ldg(&lights[2 * k + 1]).w) == rec) return true;
    return false;
}

// ------------------------------------------------------------------------------------------------ camera
// PSC/main.cpp:305-306 + PSC/camera.h:41-56.  Draw order of the path's sequential stream: jitter u, jitter v,
// disk (first draw -> y, second -> x, g++ right-to-left), time.
// camera::get_ray(s, t), PSC/camera.h:41-56
__device__ __forceinline__ void camera_get_ray(const rtnw_camera& c, float s, float t, rng_t& g, ray_t& r) {
    float px, py;
    do {
        const float dy = g.draw(), dx = g.draw();
        px = 2.0f * dx - 1.f; py = 2.0f * dy - 1.f;
    } while (px * px + py * py + 0.f >= 1.0f);
    const float rdx = c.lens_radius * px, rdy = c.lens_radius * py;
    const f3 cu = mk3(c.u[0], c.u[1], c.u[2]), cv = mk3(c.v[0], c.v[1], c.v[2]);
    const f3 offset = rdx * cu + rdy * cv;
    const float time = (float)((double)c.time0 + (double)g.draw() * (double)(c.time1 - c.time0));
    const f3 org = mk3(c.origin[0], c.origin[1], c.origin[2]);
    const f3 llc = mk3(c.lower_left_corner[0], c.lower_left_corner[1], c.lower_left_corner[2]);
    const f3 hor = mk3(c.horizontal[0], c.horizontal[1], c.horizontal[2]);
    const f3 ver = mk3(c.vertical[0], c.vertical[1], c.vertical[2]);
    r.o = org + offset;
    r.d = llc + s * hor + t * ver - org - offset;
    r.time = time;
}
__device__ __forceinline__ void camera_ray(const rtnw_camera& c, int nx, int ny, int i, int j, rng_t& g, ray_t& r) {
    const float s = ((float)i + g.draw()) / (float)nx;  // float(i + drand48()): the double sum is exact, one rounding
    const float t = ((float)j + g.draw()) / (float)ny;
    camera_get_ray(c, s, t, g, r);
}

// TNW/Chapter01_Motion Blur.cpp:29-31
__device__ __forceinline__ f3 sky_color(f3 d) {
    const f3 ud = unit_vector(d);
    const float t = 0.5f * (ud.y + 1.0f);
    return (1.0f - t) * mk3(1.f, 1.f, 1.f) + t * mk3(0.5f, 0.7f, 1.0f);
}

}  // namespace rtnw_dev
