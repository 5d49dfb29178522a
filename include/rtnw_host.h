/*
 * rtnw_host.h — C-ABI of the host scene library (librtnw_host.so): the chapter scene builders of the reference
 * (`Peter-Shirley-Project Code/main.cpp:49-230`, written against the drop-in C++ scene API) flattened into the
 * tables of rtnw.h, plus the host epilogue of the sample loop (PSC/main.cpp:315-330).  No ray arithmetic happens
 * in this library.  Used by tests/bench through ctypes and by the C++ driver `rtnw_main`.
 */
#ifndef RTNW_HOST_H_
#define RTNW_HOST_H_

#include "rtnw.h"

#ifdef __cplusplus
extern "C" {
#endif

typedef struct rtnw_host_scene rtnw_host_scene;

/* The settings each chapter's main() hard-codes (SURVEY.md §3.4, §8d). */
typedef struct rtnw_host_view {
    int32_t nx, ny, ns;
    float t_min;
    uint32_t background;  /* rtnw_background */
    uint32_t flags;       /* RTNW_F_EMIT | RTNW_F_DE_NAN as the chapter has them */
} rtnw_host_view;

const char* rtnw_host_last_error(void);

/* Build a named scene with the process-global drand48 stream reset to its never-seeded state, the perlin tables
 * drawn first (1533 draws, as the reference's static initialisers do, PSC/perlin.h:108-111), then the builder.
 * Names: "ch01_random", "two_perlin", "cornell_box", "cornell_smoke", "final", "final_northstar",
 * "simple_light", "two_spheres", "earth", "random_scene", "test", "perlin_v1" / "perlin_v2" / "perlin_v3" (the Chapter 4 noise
 * drafts of README.md:516-630), "stress_shells" and "twin_bvh" (test fixtures, not reference scenes); suffix "+bvh" wraps the flat top-level list in one
 * bvh_node(list, n, 0, 1) (PSC/bvh.h:97-121), e.g. "final+bvh"; suffix ":ch01" / ":ch03" / ":ch07" / ":ch08" selects the camera and
 * integrator settings of that chapter snapshot's main() (t_min 0.0 / 0.01, aperture 0.1, its image size, no de_nan), e.g.
 * "cornell_smoke:ch08" is TNW/Chapter08_Volume.cpp as shipped. */
int rtnw_host_scene_build(const char* name, rtnw_host_scene** out);
void rtnw_host_scene_free(rtnw_host_scene* s);
const rtnw_scene_desc* rtnw_host_scene_desc(const rtnw_host_scene* s);
int32_t rtnw_host_scene_leaf_count(const rtnw_host_scene* s);
/* the chapter's camera for an nx x ny image (aspect = nx/ny as in PSC/main.cpp:259) and its integrator settings */
int rtnw_host_scene_camera(const rtnw_host_scene* s, int32_t nx, int32_t ny, rtnw_camera* cam);
int rtnw_host_scene_view(const rtnw_host_scene* s, rtnw_host_view* view);

/* Texture ingest, replaces `stbi_load("picture.png", &nx, &ny, &nn, 0)` (PSC/main.cpp:93): decode a non-interlaced PNG
 * (grey, grey+alpha, RGB, RGBA, palette; 8-bit, or 16-bit keeping the high byte) into tightly packed RGB8, the layout
 * image_texture::value indexes (PSC/surface_texture.h:19-30).  Alpha is dropped — the reference hands stb's 4-channel
 * buffer to a 3-channel indexer (SURVEY F5).  Free with rtnw_host_free_image.  Scene name "earth@<file.png>" builds
 * earth() (PSC/main.cpp:87-97) with the decoded file as its texture. */
int rtnw_host_load_png(const char* path, unsigned char** rgb, int32_t* nx, int32_t* ny);
void rtnw_host_free_image(unsigned char* rgb);

/* camera(lookfrom, lookat, vup, vfov, aspect, aperture, focus_dist, t0, t1), PSC/camera.h:21-39 */
int rtnw_host_make_camera(const float lookfrom[3], const float lookat[3], const float vup[3], float vfov, float aspect,
                          float aperture, float focus_dist, float t0, float t1, rtnw_camera* cam);

/* PSC/main.cpp:315-325: col = sums/ns; sqrt; int(255.99*c); optional clamp to 255.  rgb_out = nx*ny*3 int32 in the
 * reference's output order (top row first). */
int rtnw_host_quantize(const float* accum_sums, int32_t nx, int32_t ny, int32_t ns, int32_t clamp255, int32_t* rgb_out);
/* PSC/main.cpp:295-334: ASCII P3 writer (binary P6 when binary != 0) */
int rtnw_host_write_ppm(const char* path, const float* accum_sums, int32_t nx, int32_t ny, int32_t ns, int32_t clamp255, int32_t binary);
/* Portable Float Map of an nx x ny image of `channels` floats per pixel (3: "PF" colour, 1: "Pf" greyscale; other counts are
 * RTNW_ERR_INVALID): header "PF\n<nx> <ny>\n-1.0\n" (scale -1: little-endian), then the floats row by row in buffer order.
 * PFM stores the bottom row first, which is row j = 0 of the library's buffers, so an rtnw_render / rtnw_render_aov buffer
 * (after dividing the sums) is written as it is. */
int rtnw_host_write_pfm(const char* path, const float* values, int32_t nx, int32_t ny, int32_t channels);

#ifdef __cplusplus
}
#endif
#endif
