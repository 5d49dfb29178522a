// rtnw_main — the reference's main() (PSC/main.cpp:244-336) with the triple sample loop replaced by the GPU library.
//
//   rtnw_main [scene] [nx ny ns] [out.ppm] [--binary] [--seed N] [--device D] [--gpus N] [--fast] [--aov PREFIX]
//             [--denoise OUT.ppm]
//   rtnw_main --selftest-bridge          exercises world->hit / scatter / emitted / value through the reference API
//
// Everything before the loop is the reference's host code written against the drop-in scene API (scene builders,
// camera); everything after it is the reference's epilogue (mean, sqrt gamma, quantise, P3 text).
// --aov PREFIX also writes the frame's colour and its first-hit feature buffers (the inputs of a denoiser) as Portable Float
// Maps: PREFIX_color.pfm (radiance sums / ns), PREFIX_albedo.pfm (albedo sums / ns), PREFIX_normal.pfm and PREFIX_depth.pfm
// (sums / hits, 0 where no sample hit).  They cover the same samples as the colour (include/rtnw.h: rtnw_render_aov).
// --denoise OUT.ppm also writes the frame denoised from those buffers (rtnw_denoise with RTNW_DENOISE_DEFAULTS) with the same
// epilogue as the main output; with --aov, PREFIX_denoised.pfm holds the denoised mean colour.  Both need one GPU.
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

#include "rtnw.h"
#include "rtnw_host.h"
#include "rtnw/device_bridge.hpp"
#include "rtnw/flatten.hpp"
#include "scenes/chapter_scenes.hpp"

static int selftest_bridge() {
    if (rtnw::install_cuda_bridge(0, 7) != RTNW_OK) {
        std::fprintf(stderr, "no GPU: %s\n", rtnw_last_error());
        return 2;
    }
    srand48(0x1234ABCD);
    perlin::regenerate();
    hitable* world = rtnw_scenes::cornell_box();
    // the reference's color() written against the API, PSC/main.cpp:25-46 (one sample, a few bounces)
    ray r(vec3(278, 278, -800), vec3(0.1f, -0.2f, 1.0f), 0.5f);
    vec3 throughput(1, 1, 1), radiance(0, 0, 0);
    for (int depth = 0; depth < 8; ++depth) {
        hit_record rec;
        if (!world->hit(r, 0.001f, MAXFLOAT, rec)) break;
        std::printf("hit depth %d t %.9g p %.9g %.9g %.9g n %g %g %g\n", depth, rec.t, rec.p.x(), rec.p.y(), rec.p.z(), rec.normal.x(),
                    rec.normal.y(), rec.normal.z());
        ray scattered;
        vec3 attenuation;
        vec3 emitted = rec.mat_ptr->emitted(rec.u, rec.v, rec.p);
        radiance += throughput * emitted;
        if (!rec.mat_ptr->scatter(r, rec, attenuation, scattered)) break;
        throughput *= attenuation;
        r = scattered;
    }
    camera cam(vec3(278, 278, -800), vec3(278, 278, 0), vec3(0, 1, 0), 40, 1.0f, 0.1f, 10, 0, 1);
    const ray cr = cam.get_ray(0.25f, 0.75f);  // PSC/camera.h:41-47 through the bridge
    std::printf("get_ray o %.9g %.9g %.9g d %.9g %.9g %.9g time %.9g\n", cr.origin().x(), cr.origin().y(), cr.origin().z(), cr.direction().x(),
                cr.direction().y(), cr.direction().z(), cr.time());
    texture* checker = new checker_texture(new constant_texture(vec3(0.2f, 0.3f, 0.1f)), new constant_texture(vec3(0.9f, 0.9f, 0.9f)));
    const vec3 c0 = checker->value(0, 0, vec3(0.1f, 0.1f, 0.1f)), c1 = checker->value(0, 0, vec3(0.4f, 0.1f, 0.1f));
    const vec3 nv = noise_texture(4).value(0, 0, vec3(1, 2, 3));
    std::printf("checker %g %g %g | %g %g %g\nnoise %.9g\nradiance %g %g %g\n", c0.x(), c0.y(), c0.z(), c1.x(), c1.y(), c1.z(), nv.x(),
                radiance.x(), radiance.y(), radiance.z());
    rtnw::bridge_invalidate(world);
    rtnw::bridge_release();
    return 0;
}

int main(int argc, char** argv) {
    std::string scene = "final", out = "Test.ppm", aov, denoise;  // PSC/main.cpp:291,295
    int nx = 0, ny = 0, ns = 0, binary = 0, device = 0, gpus = 1, fast = 0;
    unsigned long long seed = 1;
    std::vector<std::string> pos;
    for (int i = 1; i < argc; ++i) {
        const std::string a = argv[i];
        if (a == "--selftest-bridge") return selftest_bridge();
        if (a == "--binary") binary = 1;
        else if (a == "--seed" && i + 1 < argc) seed = std::strtoull(argv[++i], nullptr, 10);
        else if (a == "--device" && i + 1 < argc) device = std::atoi(argv[++i]);
        else if (a == "--gpus" && i + 1 < argc) gpus = std::atoi(argv[++i]);  // devices device .. device+gpus-1 (rtnw_render_multi)
        else if (a == "--fast") fast = 1;                                       // RTNW_F_FAST_BVH
        else if (a == "--aov" && i + 1 < argc) aov = argv[++i];
        else if (a == "--denoise" && i + 1 < argc) denoise = argv[++i];
        else pos.push_back(a);
    }
    if (pos.size() >= 1) scene = pos[0];
    if (pos.size() >= 4) { nx = std::atoi(pos[1].c_str()); ny = std::atoi(pos[2].c_str()); ns = std::atoi(pos[3].c_str()); }
    if (pos.size() == 2 || pos.size() >= 5) out = pos.back();
    if ((!aov.empty() || !denoise.empty()) && gpus > 1) {
        std::fprintf(stderr, "--aov and --denoise render on one GPU: they cannot be combined with --gpus %d\n", gpus);
        return 1;
    }

    rtnw_host_scene* hs = nullptr;
    if (rtnw_host_scene_build(scene.c_str(), &hs) != RTNW_OK) {
        std::fprintf(stderr, "scene: %s\n", rtnw_host_last_error());
        return 1;
    }
    rtnw_host_view view;
    rtnw_host_scene_view(hs, &view);
    if (nx <= 0) { nx = view.nx; ny = view.ny; ns = view.ns; }
    rtnw_camera cam;
    rtnw_host_scene_camera(hs, nx, ny, &cam);

    rtnw_render_params p;
    std::memset(&p, 0, sizeof p);
    p.nx = nx; p.ny = ny; p.sample_begin = 0; p.sample_count = ns; p.sample_stride = 1; p.max_depth = 50;
    p.t_min = view.t_min; p.t_max = MAXFLOAT; p.background = view.background; p.flags = view.flags | (fast ? RTNW_F_FAST_BVH : 0u); p.seed = seed;
    const size_t npix = (size_t)nx * ny;
    std::vector<float> accum(npix * 3);
    std::vector<float> albedo, normal, depth;
    std::vector<int32_t> hits, prim_id;
    std::vector<float> denoised;  // mean colour
    rtnw_stats st;
    if (gpus > 1) {  // the frame's samples split over `gpus` devices, summed on the first (include/rtnw.h: rtnw_render_multi)
        std::vector<int> ids;
        for (int g = 0; g < gpus; ++g) ids.push_back(device + g);
        rtnw_multi* m = nullptr;
        rtnw_multi_scene* ms = nullptr;
        if (rtnw_ctx_create_multi(ids.data(), gpus, &m) != RTNW_OK || rtnw_scene_upload_multi(m, rtnw_host_scene_desc(hs), &ms) != RTNW_OK) {
            std::fprintf(stderr, "gpu: %s\n", rtnw_last_error());
            return 2;
        }
        if (rtnw_render_multi(m, ms, &cam, &p, accum.data(), &st) != RTNW_OK) {
            std::fprintf(stderr, "render: %s\n", rtnw_last_error());
            return 3;
        }
        rtnw_scene_free_multi(m, ms);
        rtnw_ctx_destroy_multi(m);
    } else {
        rtnw_ctx* ctx = nullptr;
        rtnw_scene* dev = nullptr;
        if (rtnw_ctx_create(device, &ctx) != RTNW_OK || rtnw_scene_upload(ctx, rtnw_host_scene_desc(hs), &dev) != RTNW_OK) {
            std::fprintf(stderr, "gpu: %s\n", rtnw_last_error());
            return 2;
        }
        if (rtnw_render(ctx, dev, &cam, &p, accum.data(), &st) != RTNW_OK) {  // PSC/main.cpp:299-313 for every (i, j, s)
            std::fprintf(stderr, "render: %s\n", rtnw_last_error());
            return 3;
        }
        if (!aov.empty() || !denoise.empty()) {  // the first hits of the same paths
            albedo.resize(npix * 3); normal.resize(npix * 3); depth.resize(npix); hits.resize(npix); prim_id.resize(npix);
            const rtnw_aov bufs = {albedo.data(), normal.data(), depth.data(), hits.data(), prim_id.data()};
            if (rtnw_render_aov(ctx, dev, &cam, &p, &bufs, nullptr) != RTNW_OK) {
                std::fprintf(stderr, "aov: %s\n", rtnw_last_error());
                return 3;
            }
            if (!denoise.empty()) {
                const rtnw_denoise_params dp = RTNW_DENOISE_DEFAULTS;
                denoised.resize(npix * 3);
                if (rtnw_denoise(ctx, accum.data(), &bufs, nx, ny, ns, &dp, denoised.data(), nullptr) != RTNW_OK) {
                    std::fprintf(stderr, "denoise: %s\n", rtnw_last_error());
                    return 3;
                }
            }
        }
        rtnw_scene_free(ctx, dev);
        rtnw_ctx_destroy(ctx);
    }
    if (rtnw_host_write_ppm(out.c_str(), accum.data(), nx, ny, ns, /*clamp255=*/1, binary) != RTNW_OK) {  // :315-334
        std::fprintf(stderr, "ppm: %s\n", rtnw_host_last_error());
        return 4;
    }
    if (!denoise.empty() && rtnw_host_write_ppm(denoise.c_str(), denoised.data(), nx, ny, 1, /*clamp255=*/1, binary) != RTNW_OK) {
        std::fprintf(stderr, "ppm: %s\n", rtnw_host_last_error());
        return 4;
    }
    if (!aov.empty()) {
        std::vector<float> color(npix * 3), alb(npix * 3), nrm(npix * 3), dep(npix);
        for (size_t q = 0; q < npix; ++q) {
            const float h = (float)hits[q];
            for (int c = 0; c < 3; ++c) {
                color[3 * q + c] = accum[3 * q + c] / (float)ns;
                alb[3 * q + c] = albedo[3 * q + c] / (float)ns;
                nrm[3 * q + c] = hits[q] ? normal[3 * q + c] / h : 0.f;
            }
            dep[q] = hits[q] ? depth[q] / h : 0.f;
        }
        const struct { const char* name; const float* v; int channels; } files[] = {
            {"_color.pfm", color.data(), 3}, {"_albedo.pfm", alb.data(), 3}, {"_normal.pfm", nrm.data(), 3}, {"_depth.pfm", dep.data(), 1}};
        for (const auto& f : files) {
            if (rtnw_host_write_pfm((aov + f.name).c_str(), f.v, nx, ny, f.channels) != RTNW_OK) {
                std::fprintf(stderr, "pfm: %s\n", rtnw_host_last_error());
                return 4;
            }
        }
        if (!denoise.empty() && rtnw_host_write_pfm((aov + "_denoised.pfm").c_str(), denoised.data(), nx, ny, 3) != RTNW_OK) {
            std::fprintf(stderr, "pfm: %s\n", rtnw_host_last_error());
            return 4;
        }
    }
    std::printf("%s %dx%d %d spp on %d GPU(s): %llu paths, %llu rays, kernel %.2f ms (%.1f Mpaths/s), with copies %.2f ms -> %s\n", scene.c_str(),
                nx, ny, ns, gpus, (unsigned long long)st.paths, (unsigned long long)st.rays, st.kernel_ms, st.paths / st.kernel_ms / 1e3,
                st.total_ms, out.c_str());
    rtnw_host_scene_free(hs);
    return 0;
}
