/*
 * rtnw.h — C-ABI of the B200-native replacement for the per-pixel path-tracing sample loop of
 * EStormLynn/Peter-Shirley-Ray-Tracing-the-next-week.
 *
 * The reference has no FFI: its seam is the C++ object API (`hitable`, `material`, `texture`, `camera`)
 * plus the sample loop in `Peter-Shirley-Project Code/main.cpp:299-332` (PSC/ below).  This header is the
 * boundary a maintainer binds instead of that loop:
 *
 *   host C++ scene graph (same class names/ctors as the PSC headers)  --flatten-->  rtnw_scene_desc (SoA tables)
 *   rtnw_scene_upload()  -> tables resident in HBM
 *   rtnw_render()        -> replaces PSC/main.cpp:304-313 for every (i,j,s); returns float RGB sums
 *   rtnw_trace()         -> replaces one `world->hit(r,tmin,tmax,rec)` (PSC/main.cpp:27) per ray, for parity
 *
 * Plain pointers and sizes only; no C++/torch types.  Every call returns RTNW_OK (0) or a negative status and
 * never throws across the boundary; rtnw_last_error() gives a thread-local message.
 * There is no CPU fallback: every compute entry point fails with RTNW_ERR_CUDA when no sm_100 device is usable.
 */
#ifndef RTNW_H_
#define RTNW_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define RTNW_ABI_VERSION 5

enum rtnw_status {
    RTNW_OK = 0,
    RTNW_ERR_INVALID = -1,     /* bad argument / malformed tables            */
    RTNW_ERR_CUDA = -2,        /* CUDA runtime error or no usable device     */
    RTNW_ERR_UNSUPPORTED = -3, /* scene nesting the flattened form cannot express */
    RTNW_ERR_NOMEM = -4
};

/* ------------------------------------------------------------------------------------------------
 * Flattened scene tables.  All records are 16-byte multiples so the device reads them with 128-bit loads.
 * ---------------------------------------------------------------------------------------------- */

/* Primitive kinds (one 32-byte slot each; a moving sphere takes two consecutive slots). */
enum rtnw_prim_kind {
    RTNW_PRIM_SPHERE = 0,        /* PSC/sphere.h:10-58     f = {cx,cy,cz,r}                                */
    RTNW_PRIM_MOVING_SPHERE = 1, /* PSC/sphere.h:61-118    f = {c0x,c0y,c0z,r,t0,t1}; next slot f={c1x,c1y,c1z} */
    RTNW_PRIM_RECT_XY = 2,       /* PSC/aarect.h:11-22     f = {x0,x1,y0,y1,k}                             */
    RTNW_PRIM_RECT_XZ = 3,       /* PSC/aarect.h:24-34     f = {x0,x1,z0,z1,k}                             */
    RTNW_PRIM_RECT_YZ = 4,       /* PSC/aarect.h:36-46     f = {y0,y1,z0,z1,k}                             */
    RTNW_PRIM_BOX = 5,           /* PSC/box.h:11-38        f = {p0x,p0y,p0z,p1x,p1y,p1z}; six faces in the reference's order */
    RTNW_PRIM_MEDIUM = 6,        /* PSC/constant_medium.h  f[0]=density, f[1],f[2] = int32 bit patterns: first boundary slot, slot count */
    RTNW_PRIM_EXT = 7            /* continuation slot of the previous primitive                              */
};

/* kx word: bits 0-2 kind, bit 3 flip_normals parity (PSC/hitable.h:39-54), bits 4-31 xform chain (index of its
 * first op in the xform table; 0 = identity). */
#define RTNW_KX(kind, flip, xform) ((uint32_t)(kind) | ((uint32_t)((flip) & 1) << 3) | ((uint32_t)(xform) << 4))
#define RTNW_KX_KIND(kx) ((kx) & 7u)
#define RTNW_KX_FLIP(kx) (((kx) >> 3) & 1u)
#define RTNW_KX_XFORM(kx) ((kx) >> 4)

typedef struct rtnw_prim {
    float f[6];
    uint32_t kx;  /* RTNW_KX(kind, flip, xform) */
    int32_t mat;  /* material index (phase function for a medium); -1 for boundary-only / EXT slots */
} rtnw_prim; /* 32 B */

/* Transform chain ops, applied to the ray first-to-last and to the hit last-to-first
 * (PSC/hitable.h:57-83 translate, :85-150 rotate_y).  Op 0 of the table is a reserved identity. */
enum rtnw_xform_kind { RTNW_XF_END = 0, RTNW_XF_TRANSLATE = 1, RTNW_XF_ROTATE_Y = 2 };
typedef struct rtnw_xform_op {
    float a, b, c;   /* TRANSLATE: offset xyz; ROTATE_Y: a = sin_theta, b = cos_theta */
    uint32_t kind;   /* bits 0-7 rtnw_xform_kind; bits 8-31 (first op of a chain only) number of ops in the chain */
} rtnw_xform_op; /* 16 B */

/* BVH node = one reference bvh_node (PSC/bvh.h:11-54) holding BOTH children's boxes, so that entering a child
 * is decided by that child's own aabb::hit exactly as in the reference (leaves are never box-tested there).
 * Child ref >= 0: index of an internal node. ref < 0 and != RTNW_REF_NONE: leaf, first prim slot = ~ref,
 * slot count in lcount/rcount (list semantics inside the range).  RTNW_REF_NONE: absent (n==1 nodes, where the
 * reference sets left == right, PSC/bvh.h:106-108). */
#define RTNW_REF_NONE INT32_MIN
typedef struct rtnw_bvh_node {
    float lmin[3]; int32_t left;
    float lmax[3]; int32_t right;
    float rmin[3]; int32_t lcount;
    float rmax[3]; int32_t rcount;
} rtnw_bvh_node; /* 64 B */

/* World sequence: the top-level hitable_list (PSC/hitable_list.h:20-32) after inlining nested lists.
 * Items are evaluated in order with the narrowing closest_so_far of the reference's list. */
enum rtnw_item_kind { RTNW_ITEM_PRIMS = 0, RTNW_ITEM_BVH = 1 };
typedef struct rtnw_item {
    uint32_t kind;    /* rtnw_item_kind */
    uint32_t xform;   /* chain applied before entering the item (e.g. translate(rotate_y(bvh_node))) */
    int32_t first;    /* PRIMS: first prim slot; BVH: root node index */
    int32_t count;    /* PRIMS: slot count; BVH: number of nodes in this tree */
    float bmin[3]; uint32_t flip; /* BVH: root box (the root bvh_node's own box); flip parity pushed to prims already (informational) */
    float bmax[3]; uint32_t pad;
} rtnw_item; /* 48 B */

enum rtnw_material_kind {
    RTNW_MAT_LAMBERTIAN = 0,   /* PSC/material.h:61-72   tex = albedo texture */
    RTNW_MAT_METAL = 1,        /* PSC/material.h:74-85   albedo rgb, f = fuzz (already clamped to <= 1) */
    RTNW_MAT_DIELECTRIC = 2,   /* PSC/material.h:87-123  f = ref_idx */
    RTNW_MAT_DIFFUSE_LIGHT = 3,/* PSC/material.h:126-139 tex = emit texture */
    RTNW_MAT_ISOTROPIC = 4     /* PSC/material.h:142-151 tex = albedo texture */
};
typedef struct rtnw_material {
    uint32_t kind; int32_t tex; float f; uint32_t pad0;
    float albedo[3]; uint32_t pad1;
} rtnw_material; /* 32 B */

enum rtnw_texture_kind {
    RTNW_TEX_CONSTANT = 0, /* PSC/texture.h:16-28   c = color */
    RTNW_TEX_CHECKER = 1,  /* PSC/texture.h:30-45   i0 = even texture, i1 = odd texture */
    RTNW_TEX_NOISE = 2,    /* PSC/texture.h:47-59   c[0] = scale */
    RTNW_TEX_IMAGE = 3,    /* PSC/surface_texture.h i0 = byte offset into the image pool, i1 = nx, i2 = ny (RGB8) */
    /* The three intermediate noise textures of the reference's Chapter 4 (README.md:516-630; the sources of the shipped
     * "Chapter04_Perlin noise_noise*.ppm"): value = (1,1,1) * noise(p) over a table of 256 FLOATS, which a scene using them
     * passes in perlin_ranvec[3*i] (the x components; README.md:536-542 `ranfloat`): */
    RTNW_TEX_NOISE_HASH = 4,      /* README.md:516-524   ranfloat[perm_x[int(4x)&255] ^ perm_y[..] ^ perm_z[..]]           */
    RTNW_TEX_NOISE_TRILINEAR = 5, /* README.md:599-611   trilinear interpolation of the eight lattice values (PSC/perlin.h:11-23) */
    RTNW_TEX_NOISE_HERMITE = 6    /* README.md:619-630   the same with Hermite-smoothed u, v, w                               */
};
/* rtnw_texture.flags of an image texture: sample the four texels around (u, v) and blend them (texel centres at i + 0.5, edges
 * clamped) instead of the reference's nearest-texel lookup (PSC/surface_texture.h:19-30).  Not in the reference: an option. */
#define RTNW_TEXF_BILINEAR 1u
typedef struct rtnw_texture {
    uint32_t kind; int32_t i0, i1, i2;
    float c[3]; uint32_t flags;
} rtnw_texture; /* 32 B */

/* Borrowed host pointers; rtnw_scene_upload copies everything, the caller may free afterwards. */
typedef struct rtnw_scene_desc {
    uint32_t abi_version;          /* RTNW_ABI_VERSION */
    int32_t n_items;      const rtnw_item* items;
    int32_t n_nodes;      const rtnw_bvh_node* nodes;
    int32_t n_prim_slots; const rtnw_prim* prims;
    const int32_t* prim_ids;       /* per slot: leaf id (creation-order index of the leaf handed to the list/BVH); parity only */
    int32_t n_xform_ops;  const rtnw_xform_op* xforms;
    int32_t n_materials;  const rtnw_material* materials;
    int32_t n_textures;   const rtnw_texture* textures;
    uint64_t image_bytes; const uint8_t* images;
    const float* perlin_ranvec;    /* 256 x 3 floats, PSC/perlin.h:82-87 */
    const int32_t* perlin_perm_x;  /* 256 each, PSC/perlin.h:99-106 */
    const int32_t* perlin_perm_y;
    const int32_t* perlin_perm_z;
} rtnw_scene_desc;

/* camera — the fields PSC/camera.h:21-39 computes, passed through verbatim. */
typedef struct rtnw_camera {
    float origin[3];
    float lower_left_corner[3];
    float horizontal[3];
    float vertical[3];
    float u[3], v[3], w[3];
    float lens_radius;
    float time0, time1;
} rtnw_camera;

enum rtnw_background { RTNW_BG_BLACK = 0 /* PSC/main.cpp:44 */, RTNW_BG_SKY = 1 /* TNW/Chapter01_Motion Blur.cpp:29-31 */ };

/* render flags */
#define RTNW_F_DE_NAN        1u  /* per-sample NaN->0, PSC/main.cpp:232-242,311 */
#define RTNW_F_EMIT          2u  /* add material emitted(), PSC/main.cpp:33 (off only for the Ch01/Ch03 snapshots) */
#define RTNW_F_FAST_BVH      4u  /* fast traversal mode (default off = reference-exact): BVH boxes and leaves are tested against the
                                    ray's closest hit so far instead of the un-narrowed range bvh_node::hit hands down (PSC/bvh.h:34-35).
                                    Fewer box / primitive tests; the closest hit is the same except among candidates whose t is equal
                                    or within rounding of each other, where another of them may win */
#define RTNW_F_COUNTERS      8u  /* fill the optional work counters in rtnw_stats */
#define RTNW_F_ACCUMULATE   16u  /* add this call's pixel sums to accum_rgb instead of overwriting (rtnw_render_device only) */
#define RTNW_F_ROTATE_SAMPLES 32u /* multi-GPU split that is even for any ns: sample_count is the TOTAL number of samples ns of
                                    the frame, and for pixel p this call renders the samples s in [0, ns) with
                                    s = (sample_begin - p) mod sample_stride, + k*sample_stride: rank g of G passes
                                    sample_begin = g, sample_stride = G; each pixel gets floor or ceil(ns/G) samples per rank */

typedef struct rtnw_render_params {
    int32_t nx, ny;
    int32_t sample_begin;   /* this call renders samples s = sample_begin + k*sample_stride, k in [0, sample_count) */
    int32_t sample_count;
    int32_t sample_stride;  /* multi-GPU spp split: rank g of G uses begin=g, stride=G */
    int32_t max_depth;      /* 50, PSC/main.cpp:34 */
    float t_min;            /* 0.001, PSC/main.cpp:27 (0.0 / 0.01 in the chapter snapshots) */
    float t_max;            /* MAXFLOAT */
    uint32_t background;    /* rtnw_background */
    uint32_t flags;         /* RTNW_F_* */
    uint64_t seed;          /* Philox key; the sample stream of a path is a function of (seed, pixel, sample) only */
    /* pixel subset of this call: pixels p = pixel_begin + k*pixel_stride, k in [0, pixel_count); p = j*nx + i.
     * pixel_count == 0 means every pixel (begin 0, stride 1).  Pixels outside the subset are left untouched.  Used by
     * the multi-GPU split for the samples that do not divide evenly among the ranks. */
    int32_t pixel_begin, pixel_stride, pixel_count;
    /* 0 = the library's schedule (rtnw_plan_sample_ranges); N > 0 = cut every pixel's samples into N equal ranges (1 = one
     * work item per pixel).  Only the float summation order depends on it. */
    int32_t sample_ranges;
} rtnw_render_params;

typedef struct rtnw_stats {
    uint64_t paths;        /* (i,j,s) samples, PSC/main.cpp:304 */
    uint64_t rays;         /* top-level closest-hit queries, PSC/main.cpp:27 */
    uint64_t box_tests;    /* RTNW_F_COUNTERS only */
    uint64_t prim_tests;   /* RTNW_F_COUNTERS only */
    float kernel_ms;       /* device time of the render kernel(s), CUDA events */
    float total_ms;        /* including copies done inside the call */
    int32_t kernel_launches; /* k_render, + k_finish_fixed when the samples of a pixel were cut into more than one range */
    int32_t sample_ranges;   /* (pixel, sample range) work items per pixel of this call; their partial sums are added in 64-bit fixed point (order independent) */
} rtnw_stats;

typedef struct rtnw_ray {
    float origin[3];
    float direction[3];
    float time;
    uint32_t key;          /* stream id for media free-flight draws in rtnw_trace (Philox pixel slot) */
} rtnw_ray; /* 32 B */

typedef struct rtnw_hit {
    int32_t prim_id;       /* leaf id, -1 = miss */
    int32_t sub_id;        /* box face 0..5 (reference order, PSC/box.h:28-33), else 0 */
    float t;
    float p[3];
    float normal[3];
    float u, v;
    int32_t mat_id;
} rtnw_hit; /* 48 B */

typedef struct rtnw_ctx rtnw_ctx;       /* one GPU + its stream */
typedef struct rtnw_scene rtnw_scene;   /* device-resident copy of a scene_desc */

const char* rtnw_last_error(void);
int rtnw_abi_version(void);
/* number of CUDA devices with compute capability 10.x; 0 if none (never an error) */
int rtnw_device_count(void);

int rtnw_ctx_create(int device, rtnw_ctx** out);
int rtnw_ctx_destroy(rtnw_ctx* ctx);
/* copy the device properties the roofline needs: sm_count, clock kHz, smem per block optin, l2 bytes */
int rtnw_ctx_info(rtnw_ctx* ctx, int32_t* sm_count, int32_t* clock_khz, int32_t* smem_optin, int32_t* l2_bytes);

/* measured FP32 peak of the device in TFLOP/s (independent FFMA chains, FMA = 2 flops): the denominator of the
 * FP32-issue roofline the path is reported against (SURVEY.md §8d; not part of the reference) */
int rtnw_measure_fp32_peak(rtnw_ctx* ctx, float* tflops);

/* device self-test of the kernels' division shortcut (IEEE quotients computed from the reciprocal a ray already carries for
 * aabb::hit, PSC/aabb.h:38, instead of a second division): n random boxes / spheres / rays, including zeros, infinities, NaN
 * and the whole exponent range, each tested through the shortcut and through the plain IEEE form.  out = {box mismatches,
 * sphere mismatches, raw quotient mismatches, boxes that took the shortcut, sphere hits, box hits}; the first three must be 0.
 * Not part of the reference. */
int rtnw_selftest_recip(rtnw_ctx* ctx, uint64_t n, uint32_t seed, uint64_t out[6]);

int rtnw_scene_upload(rtnw_ctx* ctx, const rtnw_scene_desc* desc, rtnw_scene** out);

/* rtnw_scene_upload in two steps, for callers that upload the same scene repeatedly or to several devices: rtnw_scene_prepare
 * turns the tables into the device image once on the host (validation, record stream, gate tree — no device needed; the image
 * lives in pinned memory when a CUDA driver is present), rtnw_scene_upload_prepared is then one host->device copy of it.
 * rtnw_scene_upload(ctx, desc) == prepare + upload_prepared + free. */
typedef struct rtnw_prepared rtnw_prepared;
int rtnw_scene_prepare(const rtnw_scene_desc* desc, rtnw_prepared** out);
int64_t rtnw_prepared_bytes(const rtnw_prepared* p);   /* size of the device image = bytes one upload copies */
int rtnw_scene_upload_prepared(rtnw_ctx* ctx, const rtnw_prepared* prepared, rtnw_scene** out);
int rtnw_prepared_free(rtnw_prepared* p);

/* The device tables rtnw_scene_upload derives from `desc`, built on the host WITHOUT a device and copied out for
 * inspection (the invariants the traversal's exactness rests on are checked on the CPU from these, tests/test_device_tables.py).
 * table: 0 = record stream (32 B each: 8 floats, [6] = tag bits, [7] = int), 1 = per-record leaf id (int32),
 * 2 = gates (2 x int32: first records of the one or two leaves, -1 = none), 3 = gate tree (128 B per 4-wide node:
 * minx[4] miny[4] minz[4] maxx[4] maxy[4] maxz[4] ref[4] pad[4]; ref >= 0 wide node, < 0 ~gate, INT32_MIN absent).
 * Copies min(cap_bytes, size) bytes into buf (may be NULL) and returns the table's size in bytes, or a negative status. */
int64_t rtnw_scene_inspect(const rtnw_scene_desc* desc, int32_t table, void* buf, size_t cap_bytes);
int rtnw_scene_free(rtnw_ctx* ctx, rtnw_scene* scene);

/* Replaces PSC/main.cpp:304-313 over all pixels.  accum_rgb (host, nx*ny*3 floats, index (j*nx+i)*3+c with the
 * reference's j, i.e. j=0 is the bottom row) receives per-pixel SUMS over this call's samples; the host epilogue
 * (PSC/main.cpp:315-330) divides by ns, applies sqrt gamma and quantises.  Device->host copy is inside the call. */
int rtnw_render(rtnw_ctx* ctx, const rtnw_scene* scene, const rtnw_camera* cam, const rtnw_render_params* params,
                float* accum_rgb, rtnw_stats* stats);

/* Same, but accum_rgb_dev is DEVICE memory owned by the caller (e.g. a torch tensor that is then reduced with
 * NCCL); the buffer is overwritten.  The call is STREAM-ORDERED on cuda_stream (a cudaStream_t): work queued there before the
 * call (fills, a previous reduce) completes first.  NULL = the CUDA legacy default stream, which is torch's default stream.
 * Synchronous on return. */
int rtnw_render_device(rtnw_ctx* ctx, const rtnw_scene* scene, const rtnw_camera* cam,
                       const rtnw_render_params* params, float* accum_rgb_dev, void* cuda_stream, rtnw_stats* stats);

/* How rtnw_render / rtnw_render_device cut the samples of a pixel into (pixel, sample range) work items for `params`
 * (host arithmetic only, no device needed).  Writes n+1 cumulative boundaries cum[0..n] (cum[0] = 0, cum[n] = total,
 * total = the most samples a pixel has in the call) and returns n (<= cap), or a negative status.  Range c of a pixel
 * with m <= total samples covers its samples k in [cum[c]*m/total, cum[c+1]*m/total): the ranges of every pixel are
 * disjoint and cover all of its samples; their partial sums are added exactly, in 64-bit fixed point (rtnw_stats.sample_ranges = n). */
int rtnw_plan_sample_ranges(const rtnw_render_params* params, int32_t* cum, int32_t cap);

/* Output stage on the device, PSC/main.cpp:315-325: col = sums/ns (vec3::operator/=: multiply by float(1.0/ns)), sqrt gamma,
 * int(255.99*c) in double, optional clamp to 255.  accum_rgb_dev = nx*ny*3 float sums in DEVICE memory (e.g. the buffer
 * rtnw_render_device filled and NCCL reduced); rgb_out = nx*ny*3 int32 in HOST memory, in the reference's output order
 * (top row first).  Identical to rtnw_host_quantize on the same sums. */
int rtnw_quantize_device(rtnw_ctx* ctx, const float* accum_rgb_dev, int32_t nx, int32_t ny, int32_t ns, int32_t clamp255,
                         int32_t* rgb_out);

/* Deterministic closest-hit query: one `world->hit(r, t_min, t_max, rec)` per ray (PSC/main.cpp:27).  Host buffers.
 * flags: RTNW_F_FAST_BVH or 0.  Media draw their free-flight number from Philox(seed; medium leaf id, depth 0, sample 0, pixel = ray.key),
 * so results do not depend on traversal order. */
int rtnw_trace(rtnw_ctx* ctx, const rtnw_scene* scene, const rtnw_ray* rays, size_t n, float t_min, float t_max,
               uint32_t flags, uint64_t seed, rtnw_hit* out);

/* First-hit feature buffers (AOVs) of a frame: the per-pixel inputs a denoiser takes next to the noisy colour, plus depth
 * for compositing and a leaf id for picking.  For pixel p = j*nx + i and sample s = sample_begin + k*sample_stride,
 * k < sample_count, the AOV ray is exactly the first ray rtnw_render traces for (p, s) with the same camera and seed: the
 * path stream (seed, p, s), camera::get_ray with the pixel jitter, and one closest hit over [t_min, t_max] whose media draw
 * with the key (p, s, depth 0).  So the first hit of every AOV sample is the first vertex of that render path.
 * Per sample, in sample order k = 0, 1, ... (plain float additions, no atomics: the buffers are bit-reproducible):
 *   albedo  (nx*ny*3 sums)  hit: the attenuation scatter() returns — lambertian / isotropic texture value, metal albedo,
 *                           dielectric (1,1,1) — or, for diffuse_light, its emitted texture value clamped to 1 per channel;
 *                           miss: the sky colour with RTNW_BG_SKY, 0 with a black background
 *   normal  (nx*ny*3 sums)  hit: the hit_record normal (after the transform chain and flip_normals; (1,0,0) in a medium)
 *   depth   (nx*ny sums)    hit: t * sqrtf(d.x*d.x + d.y*d.y + d.z*d.z) of the camera ray direction d (distance from its origin)
 *   hits    (nx*ny int32)   number of samples that hit
 *   prim_id (nx*ny int32)   leaf id of the hit of the call's first sample (k = 0), -1 if it missed
 * These are sums like rtnw_render's: divide albedo by sample_count, normal and depth by hits.  Index order is rtnw_render's
 * ((j*nx + i)*3 + c, j = 0 the bottom row).  Honours nx, ny, sample_begin/count/stride, t_min, t_max, background, seed
 * and RTNW_F_FAST_BVH; accepts and ignores the other flags, max_depth and sample_ranges; rejects a pixel subset,
 * RTNW_F_ACCUMULATE and RTNW_F_ROTATE_SAMPLES (RTNW_ERR_INVALID).  Host buffers; stats: paths = rays = nx*ny*sample_count. */
typedef struct rtnw_aov {        /* host buffers, all required */
    float* albedo; float* normal; float* depth; int32_t* hits; int32_t* prim_id;
} rtnw_aov;
int rtnw_render_aov(rtnw_ctx* ctx, const rtnw_scene* scene, const rtnw_camera* cam,
                    const rtnw_render_params* params, const rtnw_aov* out, rtnw_stats* stats);

/* Feature-guided denoiser of a frame: spatial-only SVGF (Schied et al. 2017 without the temporal part), i.e. the edge-avoiding
 * a-trous wavelet filter of Dammertz et al. 2010 with a variance-guided luminance weight, on the GPU.  Inputs are the colour
 * sums of rtnw_render and the rtnw_aov sums of rtnw_render_aov for the same params (ns = their sample_count); prim_id is not
 * read and may be NULL.  rgb_out receives the denoised MEAN colour (nx*ny*3, not sums).  All buffers are host buffers in the
 * library's index order ((j*nx + i)*3 + c, j = 0 the bottom row).  Every step is float32 in a fixed order: the result is
 * bit-reproducible and equals its C restatement (tests/denoise_oracle.c).
 *   inputs   c = colour/ns, a = albedo/ns; a pixel is a hit pixel when hits > 0, and then n = normal/hits normalised (0 if its
 *            length is 0) and z = depth/hits.  Demodulation: a' = max(a, 1e-3) per channel, irradiance e = c / a',
 *            luminance l = 0.2126 e.r + 0.7152 e.g + 0.0722 e.b.  (A sky miss pixel has c ~ a, e ~ 1; a black miss stays 0.)
 *   gradient (|dz/dx|, |dz/dy|) by central differences over hit neighbours, one-sided next to a miss or the border, else 0.
 *   weight   of tap q at offset (dx, dy) from p: 0 if exactly one of p, q is a hit pixel, else
 *            h(dx) h(dy) w_n exp(-(d_z + d_l)) with h the B3 spline [1/16 1/4 3/8 1/4 1/16] on the pass's step,
 *            w_n = max(0, n_p.n_q)^(2^normal_power_log2), d_z = |z_p - z_q| / (sigma_depth (|dz/dx|_p |dx| + |dz/dy|_p |dy|)
 *            + 1e-3 z_p), d_l = |l_p - l_q| / (sigma_luminance sqrt(g(var)_p) + 1e-4); for two miss pixels w_n = 1, d_z = 0.
 *            g is the 3x3 binomial blur of the variance over the taps p may mix with (same hit class, weights x w_n for hits).
 *            The centre tap weighs exactly h(0)^2.  Taps outside the image are skipped; taps are summed row by row, then
 *            left to right.  exp(-x) is the library's own: range reduction to 2^-f, f in [0, 1), a degree-6 polynomial, and
 *            the exponent bits; within 1e-5 relative of exp, exactly 1 at 0 and 0 from 88 up.
 *   variance of l before the first pass: over 7x7 with weights w_n exp(-d_z) (1 at the centre), max(mu2 - mu1^2, 0).
 *   passes   i = 0 .. iterations-1 with step 2^i: e' = sum w e_q / sum w, var' = sum w^2 var_q / (sum w)^2; then out = e' a'.
 * Rejects (RTNW_ERR_INVALID, the context stays usable) a null colour, albedo, normal, depth or hits buffer or params, nx, ny or
 * ns <= 0, parameters outside their ranges, and a sigma that is not finite and > 0.  stats: kernel_ms = the denoise kernels,
 * total_ms = with the copies, kernel_launches = iterations + 2; the other fields 0.  Device memory: 101 bytes per pixel. */
typedef struct rtnw_denoise_params {
    int32_t iterations;         /* a-trous passes, step 2^i; 1..8 (5) */
    float sigma_luminance;      /* (4) */
    float sigma_depth;          /* (1) */
    int32_t normal_power_log2;  /* w_n = max(0, n_p.n_q)^(2^k); 0..10 (7 = 128) */
} rtnw_denoise_params;
#define RTNW_DENOISE_DEFAULTS {5, 4.0f, 1.0f, 7}
int rtnw_denoise(rtnw_ctx* ctx, const float* color_sums, const rtnw_aov* features, int32_t nx, int32_t ny, int32_t ns,
                 const rtnw_denoise_params* dp, float* rgb_out, rtnw_stats* stats);

/* texture::value(u,v,p) for n points; uvp = n x 5 floats {u,v,px,py,pz}; rgb_out = n x 3 (PSC/texture.h, surface_texture.h) */
int rtnw_eval_texture(rtnw_ctx* ctx, const rtnw_scene* scene, int32_t tex_id, const float* uvp, size_t n, float* rgb_out);
/* perlin::noise (which=0) / perlin::turb depth 7 (which=1) at n points xyz (PSC/perlin.h:43-74) */
int rtnw_eval_perlin(rtnw_ctx* ctx, const rtnw_scene* scene, int32_t which, const float* xyz, size_t n, float* out);

/* material::emitted + material::scatter for n (ray, hit) pairs; hit[i].mat_id selects the material.
 * Random draws come from the path stream (seed, pixel=i, sample=0) starting at its first draw (DESIGN.md §4).
 * out_scattered[i] = scattered ray; out_atten = n x 3; out_emitted = n x 3; out_flag[i] = scatter's return value. */
int rtnw_scatter(rtnw_ctx* ctx, const rtnw_scene* scene, const rtnw_ray* rays_in, const rtnw_hit* hits, size_t n,
                 uint64_t seed, rtnw_ray* out_scattered, float* out_atten, float* out_emitted, int32_t* out_flag);

/* camera::get_ray for n samples (PSC/camera.h:41-56 + the jitter of PSC/main.cpp:305-306):
 * ij = n x 2 int32 {i, j}; sample s = sample index; rays_out[n]. Draw order as in rtnw_render. */
int rtnw_camera_rays(rtnw_ctx* ctx, const rtnw_camera* cam, int32_t nx, int32_t ny, const int32_t* ij,
                     const int32_t* sample, size_t n, uint64_t seed, rtnw_ray* rays_out);

/* camera::get_ray(s, t) itself (PSC/camera.h:41-47) for n pairs: st = n x 2 floats {s, t}.  The lens-disk and shutter-time
 * draws of pair q come from the path stream (seed, pixel slot key_base + q, sample 0).  Serves the drop-in `camera::get_ray`. */
int rtnw_camera_get_rays(rtnw_ctx* ctx, const rtnw_camera* cam, const float* st, size_t n, uint64_t seed, uint32_t key_base,
                         rtnw_ray* rays_out);

/* ------------------------------------------------------------------------------------------------
 * N GPUs of one box behind one handle, driven by one host thread (one context + stream per device).  The frame's samples
 * are split over the devices (device g of G renders, for pixel p, the samples s = (g - p) mod G + k*G: even for any ns),
 * each device sums into its own buffer, and device 0 adds the buffers in rank order — reading its peers' memory directly
 * over NVLink where peer access exists, through a staging copy otherwise — before the one device->host copy of the frame.
 * The same device id may be listed more than once (two contexts on one GPU; used by the single-GPU tests).
 * ---------------------------------------------------------------------------------------------- */
typedef struct rtnw_multi rtnw_multi;
typedef struct rtnw_multi_scene rtnw_multi_scene;
int rtnw_ctx_create_multi(const int* device_ids, int n, rtnw_multi** out);   /* n <= 16 */
int rtnw_ctx_destroy_multi(rtnw_multi* m);
int rtnw_multi_device_count(const rtnw_multi* m);
int rtnw_scene_upload_multi(rtnw_multi* m, const rtnw_scene_desc* desc, rtnw_multi_scene** out);   /* to every device */
int rtnw_scene_free_multi(rtnw_multi* m, rtnw_multi_scene* scene);
/* Like rtnw_render (host buffer of per-pixel sums, whole frames only: sample_begin 0, sample_stride 1, no pixel subset).
 * stats: paths / rays / tests summed over the devices, kernel_ms = the slowest device, total_ms = launch to frame on the host. */
int rtnw_render_multi(rtnw_multi* m, const rtnw_multi_scene* scene, const rtnw_camera* cam, const rtnw_render_params* params,
                      float* accum_rgb, rtnw_stats* stats);

#ifdef __cplusplus
}
#endif
#endif /* RTNW_H_ */
