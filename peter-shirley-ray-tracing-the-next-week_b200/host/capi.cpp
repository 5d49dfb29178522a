// extern "C" surface of librtnw_host.so (include/rtnw_host.h).
#include "rtnw_host.h"

#include <cmath>
#include <cstdio>
#include <cstring>
#include <string>
#include <vector>

#include "rtnw/flatten.hpp"
#include "scenes/chapter_scenes.hpp"

struct rtnw_host_scene {
    rtnw::flat_scene flat;
    rtnw_scene_desc desc;
    rtnw_scenes::view view;
};

namespace rtnw { unsigned char* load_png_rgb8(const char* path, int& nx, int& ny, std::string& err); }

namespace {
thread_local std::string g_err;
int fail(int code, const std::string& msg) {
    g_err = msg;
    return code;
}
}  // namespace

extern "C" {

const char* rtnw_host_last_error(void) { return g_err.c_str(); }

int rtnw_host_scene_build(const char* name_c, rtnw_host_scene** out) {
    if (!name_c || !out) return fail(RTNW_ERR_INVALID, "null argument");
    std::string name(name_c);
    // ":chNN" suffix: the camera / integrator settings of that chapter snapshot's main() instead of the live main()'s
    // (SURVEY.md §3.4): ch01 and ch03 use t_min 0.0 (TNW/Chapter01_Motion Blur.cpp:16), ch07 and ch08 t_min 0.01, aperture 0.1,
    // 200x200x100 and neither de_nan nor clamp (TNW/Chapter07_Instance.cpp:25,165-178, TNW/Chapter08_Volume.cpp:26,188-253)
    std::string snapshot;
    const size_t colon = name.find(':');
    if (colon != std::string::npos) { snapshot = name.substr(colon + 1); name.erase(colon); }
    if (!snapshot.empty() && snapshot != "ch01" && snapshot != "ch03" && snapshot != "ch07" && snapshot != "ch08")
        return fail(RTNW_ERR_INVALID, "unknown chapter snapshot view: " + snapshot);
    bool wrap = false;
    const size_t plus = name.find("+bvh");
    if (plus != std::string::npos) {
        wrap = true;
        name.erase(plus);
    }
    // never-seeded drand48 state (glibc: X0 = 0x1234ABCD330E), then the tables the reference draws before main()
    srand48(0x1234ABCD);
    if (name.compare(0, 8, "perlin_v") == 0) perlin::regenerate_readme(); else
    perlin::regenerate();

    using namespace rtnw_scenes;
    hitable* world = nullptr;
    view v;
    if (name == "ch01_random") { world = random_scene_ch01(); v = view_ch01(); }
    else if (name == "two_perlin") { world = two_perlin_spheres(); v = view_two_perlin(); }
    else if (name == "cornell_box") { world = cornell_box(); v = view_cornell(); }
    else if (name == "cornell_smoke") { world = cornell_smoke(); v = view_cornell(); }
    else if (name == "final") { world = final_scene(); v = view_final(); }
    else if (name == "final_northstar") { world = final_northstar(); v = view_final(); }
    else if (name == "simple_light") { world = simple_light(); v = view_two_perlin(); v.sky = false; v.emit = true; }
    else if (name == "two_spheres") { world = two_spheres(); v = view_cornell(); v.sky = true; }
    else if (name == "earth") { world = earth(); v = view_cornell(); }
    else if (name == "earth_bilinear") {  // earth() with the bilinear option of image_texture (not a reference scene)
        int tx = 0, ty = 0;
        unsigned char* tex = synthetic_earth(tx, ty);
        hitable** l = new hitable*[2];
        l[0] = new xz_rect(63, 483, 55, 482, 554, new diffuse_light(new constant_texture(vec3(7, 7, 7))));
        l[1] = new sphere(vec3(360, 250, 150), 100, new lambertian(new image_texture(tex, tx, ty, true)));
        world = new hitable_list(l, 2);
        v = view_cornell();
    }
    else if (name.rfind("earth@", 0) == 0) {  // earth() with its texture decoded from a PNG file, PSC/main.cpp:87-97
        int tx = 0, ty = 0;
        std::string err;
        unsigned char* tex = rtnw::load_png_rgb8(name.c_str() + 6, tx, ty, err);
        if (!tex) return fail(RTNW_ERR_INVALID, err);
        world = earth(tex, tx, ty);
        v = view_cornell();
    }
    else if (name == "random_scene") { world = random_scene(); v = view_ch01(); v.emit = true; }
    else if (name == "test") { world = test_scene(); v = view_two_perlin(); v.sky = false; v.emit = true; }
    else if (name == "stress_shells") { world = stress_shells(); v = view_ch01(); v.aperture = 0.0f; }
    else if (name == "perlin_v1" || name == "perlin_v2" || name == "perlin_v3") {
        // two_perlin_spheres() of the reference's Chapter 4 drafts (README.md:588-596) with the noise function of that stage, and
        // the main() settings of that time (the Ch03 snapshot's: aperture 0.1, t_min 0.0, sky, 200x100x100)
        texture* pertext = new readme_noise_texture(name[8] - '0');
        hitable** l = new hitable*[2];
        l[0] = new sphere(vec3(0, -1000, 0), 1000, new lambertian(pertext));
        l[1] = new sphere(vec3(0, 2, 0), 2, new lambertian(pertext));
        world = new hitable_list(l, 2);
        v = view_ch01();
        v.t_min = 0.0f;
    }
    else if (name == "twin_bvh") { world = twin_bvh(); v = view_ch01(); v.aperture = 0.0f; }
    else return fail(RTNW_ERR_INVALID, "unknown scene name: " + name);
    if (wrap) world = wrap_in_bvh(world, 0, 1);
    if (snapshot == "ch01" || snapshot == "ch03") {
        v.t_min = 0.0f; v.aperture = 0.1f; v.nx = 200; v.ny = 100; v.ns = 100; v.sky = true; v.emit = false; v.de_nan = false;
    } else if (snapshot == "ch07" || snapshot == "ch08") {
        v.t_min = 0.01f; v.aperture = 0.1f; v.nx = 200; v.ny = 200; v.ns = 100; v.lookfrom = vec3(278, 278, -800); v.de_nan = false;
    }

    rtnw_host_scene* s = new rtnw_host_scene();
    const int rc = rtnw::flatten(world, s->flat);
    if (rc != RTNW_OK) {
        const std::string msg = s->flat.error;
        delete s;
        return fail(rc, msg);
    }
    s->desc = s->flat.desc();
    s->view = v;
    *out = s;
    return RTNW_OK;
}

void rtnw_host_scene_free(rtnw_host_scene* s) { delete s; }

const rtnw_scene_desc* rtnw_host_scene_desc(const rtnw_host_scene* s) { return s ? &s->desc : nullptr; }

int32_t rtnw_host_scene_leaf_count(const rtnw_host_scene* s) { return s ? s->flat.n_leaves : 0; }

int rtnw_host_scene_camera(const rtnw_host_scene* s, int32_t nx, int32_t ny, rtnw_camera* cam) {
    if (!s || !cam || nx <= 0 || ny <= 0) return fail(RTNW_ERR_INVALID, "bad camera arguments");
    rtnw::to_c_camera(rtnw_scenes::make_camera(s->view, nx, ny), *cam);
    return RTNW_OK;
}

int rtnw_host_scene_view(const rtnw_host_scene* s, rtnw_host_view* out) {
    if (!s || !out) return fail(RTNW_ERR_INVALID, "null argument");
    out->nx = s->view.nx;
    out->ny = s->view.ny;
    out->ns = s->view.ns;
    out->t_min = s->view.t_min;
    out->background = s->view.sky ? RTNW_BG_SKY : RTNW_BG_BLACK;
    out->flags = (s->view.emit ? RTNW_F_EMIT : 0u) | (s->view.de_nan ? RTNW_F_DE_NAN : 0u);
    return RTNW_OK;
}

int rtnw_host_make_camera(const float lookfrom[3], const float lookat[3], const float vup[3], float vfov, float aspect,
                          float aperture, float focus_dist, float t0, float t1, rtnw_camera* cam) {
    if (!lookfrom || !lookat || !vup || !cam) return fail(RTNW_ERR_INVALID, "null argument");
    camera c(vec3(lookfrom[0], lookfrom[1], lookfrom[2]), vec3(lookat[0], lookat[1], lookat[2]), vec3(vup[0], vup[1], vup[2]),
             vfov, aspect, aperture, focus_dist, t0, t1);
    rtnw::to_c_camera(c, *cam);
    return RTNW_OK;
}

// PSC/main.cpp:315-325
static inline void quantize_pixel(const float* sum, int32_t ns, int clamp255, int32_t out[3]) {
    vec3 col(sum[0], sum[1], sum[2]);
    col /= float(ns);
    col = vec3(std::sqrt(col[0]), std::sqrt(col[1]), std::sqrt(col[2]));
    for (int c = 0; c < 3; ++c) {
        int v = int(255.99 * col[c]);
        if (clamp255 && v > 255) v = 255;
        out[c] = v;
    }
}

int rtnw_host_load_png(const char* path, unsigned char** rgb, int32_t* nx, int32_t* ny) {
    if (!path || !rgb || !nx || !ny) return fail(RTNW_ERR_INVALID, "null argument");
    int tx = 0, ty = 0;
    std::string err;
    unsigned char* px = rtnw::load_png_rgb8(path, tx, ty, err);
    if (!px) return fail(RTNW_ERR_INVALID, err);
    *rgb = px; *nx = tx; *ny = ty;
    return RTNW_OK;
}
void rtnw_host_free_image(unsigned char* rgb) { delete[] rgb; }

int rtnw_host_quantize(const float* sums, int32_t nx, int32_t ny, int32_t ns, int32_t clamp255, int32_t* rgb_out) {
    if (!sums || !rgb_out || nx <= 0 || ny <= 0 || ns <= 0) return fail(RTNW_ERR_INVALID, "bad quantize arguments");
    size_t o = 0;
    for (int j = ny - 1; j >= 0; --j)
        for (int i = 0; i < nx; ++i, o += 3) quantize_pixel(sums + 3 * ((size_t)j * nx + i), ns, clamp255, rgb_out + o);
    return RTNW_OK;
}

int rtnw_host_write_ppm(const char* path, const float* sums, int32_t nx, int32_t ny, int32_t ns, int32_t clamp255, int32_t binary) {
    if (!path || !sums || nx <= 0 || ny <= 0 || ns <= 0) return fail(RTNW_ERR_INVALID, "bad ppm arguments");
    FILE* f = std::fopen(path, binary ? "wb" : "w");
    if (!f) return fail(RTNW_ERR_INVALID, std::string("cannot open ") + path);
    std::fprintf(f, "%s\n%d %d\n255\n", binary ? "P6" : "P3", nx, ny);
    for (int j = ny - 1; j >= 0; --j) {
        for (int i = 0; i < nx; ++i) {
            int32_t q[3];
            quantize_pixel(sums + 3 * ((size_t)j * nx + i), ns, binary ? 1 : clamp255, q);
            if (binary) {
                const unsigned char b[3] = {(unsigned char)q[0], (unsigned char)q[1], (unsigned char)q[2]};
                std::fwrite(b, 1, 3, f);
            } else {
                std::fprintf(f, "%d %d %d\n", q[0], q[1], q[2]);
            }
        }
    }
    std::fclose(f);
    return RTNW_OK;
}

int rtnw_host_write_pfm(const char* path, const float* values, int32_t nx, int32_t ny, int32_t channels) {
    if (!path || !values || nx <= 0 || ny <= 0) return fail(RTNW_ERR_INVALID, "bad pfm arguments");
    if (channels != 1 && channels != 3) return fail(RTNW_ERR_INVALID, "a PFM holds 1 or 3 channels");
    FILE* f = std::fopen(path, "wb");
    if (!f) return fail(RTNW_ERR_INVALID, std::string("cannot open ") + path);
    std::fprintf(f, "%s\n%d %d\n-1.0\n", channels == 3 ? "PF" : "Pf", nx, ny);
    const size_t n = (size_t)nx * ny * channels;
    std::vector<unsigned char> bytes(4 * n);
    for (size_t i = 0; i < n; ++i) {  // little-endian whatever the host's byte order
        uint32_t u;
        std::memcpy(&u, values + i, 4);
        for (int b = 0; b < 4; ++b) bytes[4 * i + b] = (unsigned char)(u >> (8 * b));
    }
    const bool ok = std::fwrite(bytes.data(), 1, bytes.size(), f) == bytes.size();
    if (std::fclose(f) != 0 || !ok) return fail(RTNW_ERR_INVALID, std::string("cannot write ") + path);
    return RTNW_OK;
}

}  // extern "C"
