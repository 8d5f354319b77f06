// vanrijn_main.cpp -- the reference's harness (src/main.rs:104-247) over the C++ host mirror, without the SDL window:
//   * same command line: --size W H (required), --out FILE.png, --time SECONDS          (main.rs:34-73)
//   * same scene: plane + three Lambertian spheres + the bunny BVH, camera (-2, 1, -5)    (main.rs:120-189)
//   * same loop: TileIterator(width, height, 2048) cycled; every tile goes through partial_render_scene and is merged
//     into the frame's AccumulationBuffer with merge_tile; the frame is tone-mapped with ClampingToneMapper and written
//     as PNG                                                                              (main.rs:192-232)
// In the reference `.cycle()` never ends, so --out is never written and --time is never read (SURVEY 8f N4); here the
// loop ends after --time seconds (or --passes passes, default 1 when --time is 0) and then writes --out.
// Additions: --obj FILE (default $VANRIJN_BUNNY_OBJ; the reference hard-codes test_data/stanford_bunny.obj),
// --spp N samples per partial_render_scene call (the reference: 1), --passes N, --depth N (RECURSION_LIMIT, 128),
// --builder host|device|upload, --seed N, --preview-every N (rewrite --out every N passes: the progressive view),
// --cache FILE: the flattened scene on disk (load_scene_cache if FILE exists, else build the scene and save_scene_cache),
// --resident: keep the frame's AccumulationBuffer on the GPU (DeviceAccumulationBuffer) instead of downloading a
// buffer per tile and merging on the host; previews then move 3 bytes per pixel.
// --rel-error E (with --resident): sample adaptively instead (DeviceProgressiveBuffer, vrj_render_progressive), one pass
// of --spp samples per loop iteration: every pixel first takes --min-spp (default 4), then pixels whose mean Y is not yet
// within E take --spp more, up to --max-spp (default 64); the loop also ends when no pixel is active.
// --denoise (with --rel-error): previews and --out are the denoised frame (vrj_render_aux once, vrj_denoise per preview).
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <memory>
#include <string>

#include "vanrijn.hpp"

using namespace vanrijn;

namespace {
struct CommandLineParameters {
    size_t width = 0, height = 0;
    std::string output_file, obj, cache;
    double time = 0.0;
    uint32_t spp = 1, passes = 0, depth = 128, preview_every = 0;
    uint64_t seed = 1;
    bool resident = false, denoise = false;
    double rel_error = 0.0; // > 0: adaptive progressive passes (--rel-error)
    uint32_t min_spp = 4, max_spp = 64;
    BoundingVolumeHierarchy::Builder builder = BoundingVolumeHierarchy::Builder::AtUpload;
};

[[noreturn]] void usage(const char *why) {
    std::fprintf(stderr, "error: %s\nUSAGE: vanrijn --size <WIDTH> <HEIGHT> [--out <FILENAME>] [--time <SECONDS>] [--obj <FILE>] [--spp N] "
                         "[--passes N] [--depth N] [--builder host|device|upload] [--seed N] [--preview-every N] [--resident] [--cache FILE]\n"
                         "       [--rel-error E [--min-spp N] [--max-spp N] [--denoise]]\n", why);
    std::exit(2);
}

CommandLineParameters parse_args(int argc, char **argv) {
    CommandLineParameters p;
    if (const char *env = std::getenv("VANRIJN_BUNNY_OBJ")) p.obj = env;
    for (int i = 1; i < argc; i++) {
        const std::string a = argv[i];
        auto value = [&](int extra = 0) -> const char * {
            if (i + 1 + extra >= argc) usage(("missing value for " + a).c_str());
            return argv[i + 1 + extra];
        };
        if (a == "--size") p.width = std::strtoull(value(), nullptr, 10), p.height = std::strtoull(value(1), nullptr, 10), i += 2;
        else if (a == "--out") p.output_file = value(), i++;
        else if (a == "--time") p.time = std::strtod(value(), nullptr), i++;
        else if (a == "--obj") p.obj = value(), i++;
        else if (a == "--cache") p.cache = value(), i++;
        else if (a == "--spp") p.spp = (uint32_t)std::strtoul(value(), nullptr, 10), i++;
        else if (a == "--passes") p.passes = (uint32_t)std::strtoul(value(), nullptr, 10), i++;
        else if (a == "--depth") p.depth = (uint32_t)std::strtoul(value(), nullptr, 10), i++;
        else if (a == "--seed") p.seed = std::strtoull(value(), nullptr, 10), i++;
        else if (a == "--preview-every") p.preview_every = (uint32_t)std::strtoul(value(), nullptr, 10), i++;
        else if (a == "--resident") p.resident = true;
        else if (a == "--rel-error") p.rel_error = std::strtod(value(), nullptr), i++;
        else if (a == "--min-spp") p.min_spp = (uint32_t)std::strtoul(value(), nullptr, 10), i++;
        else if (a == "--max-spp") p.max_spp = (uint32_t)std::strtoul(value(), nullptr, 10), i++;
        else if (a == "--denoise") p.denoise = true;
        else if (a == "--builder") {
            const std::string b = value();
            i++;
            if (b == "host") p.builder = BoundingVolumeHierarchy::Builder::Host;
            else if (b == "device") p.builder = BoundingVolumeHierarchy::Builder::Device;
            else if (b == "upload") p.builder = BoundingVolumeHierarchy::Builder::AtUpload;
            else usage("--builder takes host, device or upload");
        } else usage(("unknown argument " + a).c_str());
    }
    if (p.width == 0 || p.height == 0) usage("--size <WIDTH> <HEIGHT> is required");
    if (p.spp == 0) usage("--spp must be positive");
    if (p.rel_error > 0.0 && !p.resident) usage("--rel-error needs --resident");
    if (p.rel_error < 0.0 || p.min_spp < 2 || p.max_spp < p.min_spp) usage("--rel-error must be > 0, --min-spp >= 2, --max-spp >= --min-spp");
    if (p.denoise && p.rel_error <= 0.0) usage("--denoise needs --rel-error");
    return p;
}

std::shared_ptr<Material> lambertian(ColourRgbF c, double diffuse) {
    return std::make_shared<LambertianMaterial>(Spectrum::reflection_from_linear_rgb(c), diffuse);
}
double seconds_since(std::chrono::steady_clock::time_point t0) {
    return std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
}
} // namespace

int main(int argc, char **argv) {
    const CommandLineParameters parameters = parse_args(argc, argv);
    const size_t image_width = parameters.width, image_height = parameters.height;
    try {
        AccumulationBuffer rendered_image(image_width, image_height);
        Scene scene;
        bool from_cache = false;
        if (!parameters.cache.empty()) {
            if (FILE *probe = std::fopen(parameters.cache.c_str(), "rb")) {
                std::fclose(probe);
                const auto t_cache = std::chrono::steady_clock::now();
                scene = load_scene_cache(parameters.cache);
                from_cache = true;
                std::printf("Loaded the flattened scene from %s (%.3f s)\n", parameters.cache.c_str(), seconds_since(t_cache));
            }
        }
        auto t_load = std::chrono::steady_clock::now();
        if (!from_cache) {
        scene.camera_location = Vec3(-2.0, 1.0, -5.0);
        auto list = std::unique_ptr<PrimitiveList>(new PrimitiveList());
        list->primitives.push_back(std::make_shared<Plane>(Vec3(0.0, 1.0, 0.0), -2.0, lambertian(ColourRgbF(0.55, 0.27, 0.04), 0.1)));
        list->primitives.push_back(std::make_shared<Sphere>(Vec3(-6.25, -0.5, 1.0), 1.0, lambertian(ColourRgbF::from_named(NamedColour::Green), 0.1)));
        list->primitives.push_back(std::make_shared<Sphere>(Vec3(-4.25, -0.5, 2.0), 1.0, lambertian(ColourRgbF::from_named(NamedColour::Blue), 0.1)));
        list->primitives.push_back(std::make_shared<Sphere>(Vec3(-5.0, 1.5, 1.0), 1.0, lambertian(ColourRgbF::from_named(NamedColour::Red), 0.05)));
        scene.objects.push_back(std::move(list));
        if (!parameters.obj.empty()) {
            std::printf("Loading object...\n");
            const TriangleMesh mesh = load_obj_mesh(parameters.obj);
            std::printf("Building BVH... (%zu triangles)\n", mesh.triangle_count());
            scene.objects.push_back(BoundingVolumeHierarchy::build(mesh, lambertian(ColourRgbF::from_named(NamedColour::Yellow), 0.05), parameters.builder));
        } else {
            std::printf("No --obj and no $VANRIJN_BUNNY_OBJ: rendering the scene without the model.\n");
        }
        if (!parameters.cache.empty()) {
            save_scene_cache(scene, parameters.cache);
            std::printf("Saved the flattened scene to %s\n", parameters.cache.c_str());
        }
        } // !from_cache
        std::printf("Constructing Scene...\n");
        device_scene(scene, 0); // flatten + upload (+ BVH build on the device with --builder upload)
        std::printf("Done. (%.3f s)\n", seconds_since(t_load));

        const uint32_t passes_wanted = parameters.passes ? parameters.passes : (parameters.time > 0.0 ? 0xffffffffu : 1u);
        uint64_t rays = 0;
        double device_ms = 0.0, call_s = 0.0, merge_s = 0.0;
        uint32_t pass = 0;
        const auto t0 = std::chrono::steady_clock::now();
        std::unique_ptr<DeviceAccumulationBuffer> resident;
        std::unique_ptr<DeviceProgressiveBuffer> progressive;
        if (parameters.resident && parameters.rel_error > 0.0) progressive.reset(new DeviceProgressiveBuffer(image_width, image_height));
        else if (parameters.resident) resident.reset(new DeviceAccumulationBuffer(image_width, image_height));
        RenderOptions progressive_options;
        progressive_options.spp = parameters.spp, progressive_options.max_depth = parameters.depth, progressive_options.seed = parameters.seed;
        auto progressive_image = [&] {
            return parameters.denoise ? progressive->denoised_image_rgb_u8(scene, progressive_options) : progressive->to_image_rgb_u8();
        };
        for (; pass < passes_wanted; pass++) {
            if (parameters.time > 0.0 && pass > 0 && seconds_since(t0) >= parameters.time) break;
            if (progressive) {
                ProgressiveOptions pp;
                VrjProgressiveStats pstats{};
                VrjStats stats{};
                pp.min_samples = parameters.min_spp, pp.max_samples = parameters.max_spp, pp.pass_samples = parameters.spp;
                pp.rel_error = parameters.rel_error, pp.stats = &pstats;
                progressive_options.stats = &stats;
                const auto t_call = std::chrono::steady_clock::now();
                progressive->render(scene, progressive_options, pp);
                call_s += seconds_since(t_call);
                rays += stats.primary_rays + stats.bounce_rays + stats.shadow_rays;
                device_ms += stats.device_ms;
                std::printf("pass %u: %llu samples, %llu pixels active, %llu converged, %llu at --max-spp\n", pass + 1,
                            (unsigned long long)pstats.samples, (unsigned long long)pstats.pixels_active,
                            (unsigned long long)pstats.pixels_converged, (unsigned long long)pstats.pixels_at_max);
                if (parameters.preview_every && !parameters.output_file.empty() && (pass + 1) % parameters.preview_every == 0)
                    progressive_image().write_png(parameters.output_file);
                if (pstats.pixels_active == 0) {
                    pass++;
                    break;
                }
                continue;
            }
            if (resident) {
                RenderOptions o;
                VrjStats stats{};
                o.spp = parameters.spp, o.max_depth = parameters.depth, o.seed = parameters.seed, o.stats = &stats;
                const auto t_call = std::chrono::steady_clock::now();
                resident->render(scene, o);
                call_s += seconds_since(t_call);
                rays += stats.primary_rays + stats.bounce_rays + stats.shadow_rays;
                device_ms += stats.device_ms;
                if (parameters.preview_every && !parameters.output_file.empty() && (pass + 1) % parameters.preview_every == 0)
                    resident->to_image_rgb_u8().write_png(parameters.output_file);
                continue;
            }
            TileIterator tiles(image_width, image_height, 2048); // main.rs:199
            Tile tile;
            while (tiles.next(tile)) {
                RenderOptions o;
                VrjStats stats{};
                o.spp = parameters.spp, o.max_depth = parameters.depth, o.seed = parameters.seed;
                o.sample_offset = (uint64_t)pass * parameters.spp;
                o.stats = &stats;
                o.kahan_state = false; // merge_tile reads colour and weight only (main.rs:216): 66 MB back per 1080p pass, not 182 MB
                const auto t_call = std::chrono::steady_clock::now();
                AccumulationBuffer rendered_tile = partial_render_scene(scene, tile, image_height, image_width, o);
                call_s += seconds_since(t_call);
                const auto t_merge = std::chrono::steady_clock::now();
                rendered_image.merge_tile(tile, rendered_tile); // main.rs:216
                merge_s += seconds_since(t_merge);
                rays += stats.primary_rays + stats.bounce_rays + stats.shadow_rays;
                device_ms += stats.device_ms;
            }
            if (parameters.preview_every && !parameters.output_file.empty() && (pass + 1) % parameters.preview_every == 0)
                rendered_image.to_image_rgb_u8().write_png(parameters.output_file);
        }
        const double wall = seconds_since(t0);
        std::printf("%u passes x %u spp at %zux%zu in %.3f s: %.1f Mrays/s wall, %.1f Mrays/s on the device, %.2f spp/s\n", pass,
                    parameters.spp, image_width, image_height, wall, rays / wall / 1e6, device_ms > 0 ? rays / device_ms / 1e3 : 0.0,
                    pass * (double)parameters.spp / wall);
        std::printf("host time: partial_render_scene %.3f s (device %.3f s), merge_tile %.3f s\n", call_s, device_ms / 1e3, merge_s);
        if (!parameters.output_file.empty()) {
            if (progressive) progressive_image().write_png(parameters.output_file);
            else if (resident) resident->to_image_rgb_u8().write_png(parameters.output_file);
            else rendered_image.to_image_rgb_u8().write_png(parameters.output_file); // main.rs:222-225
            std::printf("wrote %s\n", parameters.output_file.c_str());
        }
    } catch (const std::exception &e) {
        std::fprintf(stderr, "vanrijn: %s\n", e.what());
        return 1;
    }
    return 0;
}
