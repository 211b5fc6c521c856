// main.cpp — the reference's `main` (main.rs:797-1010) on top of the C ABI.
//
//   rt1w_main [scene] [--width W] [--spp N] [--depth D] [--seed S] [--earth earthmap.ppm] [--device K | --gpus N]
//             [--max-error L [--min-spp M] | --frames F] > image.ppm
//
// `scene` is an arm of `match 5 { .. }` (main.rs:815-937) by number (0..7) or name (random_scene, two_spheres,
// two_perlin_spheres, earth, simple_light, cornel_box, cornel_smoke, final_scene); default 5 like the reference.
// Everything up to the pixel loop is the reference's code path in the C++ mirror (scene function, per-arm
// settings, Camera::new); the pixel loop (main.rs:957-1001) is one rt1w_render_rgb8 call per progress chunk of
// the sample range; the P3 text goes to stdout and the progress line to stderr as in main.rs:953,995-1009.
// `--gpus N`: devices 0..N-1 render every chunk together (rt1w_context_create_multi: sample ranges sharded inside the
// library, one ncclReduce of the radiance sums per chunk); the call sequence below stays the same.
// `--max-error L [--min-spp N]` (N = 16 by default): adaptive sampling instead - ONE rt1w_render_adaptive call renders every
// pixel until its 8-bit value has converged to L levels (include/rt1w.h), `--spp` being the cap; one device only.
// `--frames F`: a turntable of F images instead - frame k looks at look_at from look_from rotated by k * 360 / F degrees
// about the vertical axis through look_at, with seed k (frame 0 is the single image).  ONE rt1w_render_batch call renders
// every frame; the images follow each other on stdout (a netpbm multi-image stream).
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

#include <unistd.h>

#include "../../include/rt1w.h"
#include "scenes.hpp"

namespace {

bool read_ppm(const char *path, rt1w::EarthMap &map) { // binary P6, as tools/prep_earthmap.py writes it
    FILE *f = std::fopen(path, "rb");
    if (!f) return false;
    int w = 0, h = 0, maxv = 0;
    if (std::fscanf(f, "P6 %d %d %d", &w, &h, &maxv) != 3 || w <= 0 || h <= 0 || maxv != 255) {
        std::fclose(f);
        return false;
    }
    std::fgetc(f);
    auto data = std::make_shared<std::vector<uint8_t>>(size_t(w) * size_t(h) * 3);
    const bool ok = std::fread(data->data(), 1, data->size(), f) == data->size();
    std::fclose(f);
    if (!ok) return false;
    map.rgb8 = data, map.width = w, map.height = h;
    return true;
}

int fail(const char *what) {
    std::fprintf(stderr, "rt1w_main: %s: %s\n", what, rt1w_last_error());
    return 1;
}

} // namespace

int main(int argc, char **argv) {
    int which = 5; // `match 5` (main.rs:815)
    int width = 0, spp = 0, depth = 0, device = 0, gpus = 1, min_spp = 16;
    int frames = 0;
    bool adaptive = false;
    double max_error = 0.0;
    uint64_t seed = 1;
    std::string earth_path = "assets/earthmap.ppm";
    for (int i = 1; i < argc; ++i) {
        const std::string a = argv[i];
        auto value = [&]() -> const char * { return i + 1 < argc ? argv[++i] : "0"; };
        if (a == "--width") width = std::atoi(value());
        else if (a == "--spp") spp = std::atoi(value());
        else if (a == "--depth") depth = std::atoi(value());
        else if (a == "--seed") seed = std::strtoull(value(), nullptr, 10);
        else if (a == "--device") device = std::atoi(value());
        else if (a == "--gpus") gpus = std::atoi(value());
        else if (a == "--earth") earth_path = value();
        else if (a == "--max-error") adaptive = true, max_error = std::atof(value());
        else if (a == "--min-spp") min_spp = std::atoi(value());
        else if (a == "--frames") frames = std::atoi(value());
        else if (!a.empty() && (a[0] >= '0' && a[0] <= '9')) which = std::atoi(a.c_str());
        else which = rt1w::scene_id_from_name(a);
    }
    if (which < 0) {
        std::fprintf(stderr, "rt1w_main: unknown scene\n");
        return 2;
    }
    if (frames < 0 || (frames > 0 && adaptive)) {
        std::fprintf(stderr, "rt1w_main: --frames takes a positive count and does not combine with --max-error\n");
        return 2;
    }
    rt1w::EarthMap map;
    if ((which == 3 || which >= 7) && !read_ppm(earth_path.c_str(), map))
        std::fprintf(stderr, "rt1w_main: no earth map at %s (tools/prep_earthmap.py makes one); image textures will fail\n", earth_path.c_str());

    std::unique_ptr<rt1w::SceneSetup> setup;
    try {
        setup = rt1w::select_scene(which, seed, map);
    } catch (const std::exception &e) { // the reference panics here (e.g. `unwrap` on the image, main.rs:348)
        std::fprintf(stderr, "rt1w_main: %s\n", e.what());
        return 1;
    }
    if (width > 0) setup->image_width = width;
    if (spp > 0) setup->samples_per_pixel = spp;
    if (depth > 0) setup->max_depth = depth;
    const int image_width = setup->image_width, image_height = setup->image_height(); // main.rs:939
    const rt1w_scene_desc desc = setup->builder.desc();
    const rt1w::Camera camera = setup->camera();

    rt1w_context *ctx = nullptr;
    if (gpus > 1) {
        // stdout is the image (main.rs:953): NCCL writes its version / debug lines to stdout while the communicator is set
        // up, so file descriptor 1 points at stderr for the duration of that call
        std::vector<int32_t> ids;
        for (int g = 0; g < gpus; ++g) ids.push_back(device + g);
        std::fflush(stdout);
        const int saved_stdout = dup(1);
        dup2(2, 1);
        const rt1w_status st = rt1w_context_create_multi(ids.data(), gpus, &ctx);
        std::fflush(stdout);
        dup2(saved_stdout, 1);
        close(saved_stdout);
        if (st != RT1W_OK) return fail("rt1w_context_create_multi");
    } else if (rt1w_context_create(device, &ctx) != RT1W_OK) {
        return fail("rt1w_context_create");
    }
    rt1w_scene *scene = nullptr;
    if (rt1w_scene_create(ctx, &desc, &scene) != RT1W_OK) return fail("rt1w_scene_create");

    rt1w_render_params p;
    std::memset(&p, 0, sizeof(p));
    p.width = image_width, p.height = image_height, p.max_depth = setup->max_depth, p.seed = 0;
    p.background[0] = setup->background.v.x, p.background[1] = setup->background.v.y, p.background[2] = setup->background.v.z;
    const int total = setup->samples_per_pixel;
    if (adaptive) { // one call; the image is resolved on the device with each pixel's own sample count
        p.sample_begin = 0, p.sample_end = total;
        std::vector<uint8_t> rgb8(size_t(image_width) * image_height * 3);
        if (rt1w_render_adaptive(scene, &camera.pod, &p, min_spp, max_error, nullptr, nullptr, rgb8.data(), nullptr, nullptr) != RT1W_OK)
            return fail("rt1w_render_adaptive");
        std::printf("P3\n%d %d\n255\n", image_width, image_height); // main.rs:953
        std::fprintf(stderr, "\rScanlines remaining: 0 ");
        for (size_t px = 0; px < rgb8.size(); px += 3) std::printf("%d %d %d\n", rgb8[px], rgb8[px + 1], rgb8[px + 2]); // main.rs:1003-1007
        std::fprintf(stderr, "\nDone\n");
        rt1w_scene_destroy(scene);
        rt1w_context_destroy(ctx);
        return 0;
    }

    if (frames > 0) { // one batch call: every frame in one wavefront, resolved on the device
        const double pi = 3.14159265358979323846;
        const rt1w::Vec3 home = setup->look_from, arm = home - setup->look_at;
        std::vector<rt1w_camera> cams;
        std::vector<uint64_t> seeds;
        for (int k = 0; k < frames; ++k) { // (frame 0: exactly the single image's camera)
            const double angle = 2.0 * pi * double(k) / double(frames), c = std::cos(angle), s = std::sin(angle);
            setup->look_from = k == 0 ? home : setup->look_at + rt1w::vec3(c * arm.x + s * arm.z, arm.y, -s * arm.x + c * arm.z);
            cams.push_back(setup->camera().pod), seeds.push_back(uint64_t(k));
        }
        setup->look_from = home;
        p.sample_begin = 0, p.sample_end = total;
        std::vector<uint8_t> rgb8(size_t(frames) * image_width * image_height * 3);
        if (rt1w_render_batch(scene, cams.data(), frames, seeds.data(), &p, nullptr, rgb8.data(), nullptr) != RT1W_OK) return fail("rt1w_render_batch");
        std::fprintf(stderr, "\rScanlines remaining: 0 ");
        const size_t frame_bytes = size_t(image_width) * image_height * 3;
        for (int k = 0; k < frames; ++k) {
            std::printf("P3\n%d %d\n255\n", image_width, image_height); // main.rs:953
            for (size_t px = k * frame_bytes; px < (k + 1) * frame_bytes; px += 3) std::printf("%d %d %d\n", rgb8[px], rgb8[px + 1], rgb8[px + 2]);
        }
        std::fprintf(stderr, "\nDone\n");
        rt1w_scene_destroy(scene);
        rt1w_context_destroy(ctx);
        return 0;
    }

    std::printf("P3\n%d %d\n255\n", image_width, image_height); // main.rs:953

    // The reference counts scanlines down while rayon works through them (main.rs:995-998); here the image is
    // rendered as a whole, one sample range at a time, and the same line counts the rows' worth of work left.
    const int chunk = total >= 16 ? (total + 7) / 8 : total;
    std::vector<float> sum(size_t(image_width) * image_height * 3, 0.0f), part(sum.size());
    for (int s0 = 0; s0 < total; s0 += chunk) {
        p.sample_begin = s0, p.sample_end = s0 + chunk < total ? s0 + chunk : total;
        if (rt1w_render(scene, &camera.pod, &p, part.data(), nullptr, nullptr) != RT1W_OK) return fail("rt1w_render");
        for (size_t i = 0; i < sum.size(); ++i) sum[i] += part[i]; // a NaN sample keeps the pixel NaN -> black (color.rs:16-18)
        std::fprintf(stderr, "\rScanlines remaining: %d ", int((long long)image_height * (total - p.sample_end) / total));
    }
    std::vector<uint8_t> rgb8(sum.size());
    rt1w_resolve_rgb8(sum.data(), image_width, image_height, total, rgb8.data()); // main.rs:992
    for (size_t px = 0; px < rgb8.size(); px += 3) std::printf("%d %d %d\n", rgb8[px], rgb8[px + 1], rgb8[px + 2]); // main.rs:1003-1007
    std::fprintf(stderr, "\nDone\n");

    rt1w_scene_destroy(scene);
    rt1w_context_destroy(ctx);
    return 0;
}
