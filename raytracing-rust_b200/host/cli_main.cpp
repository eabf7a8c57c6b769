// ptb200-cli — the reference frontend's command line (src/parameters.rs:20-43, src/main.rs:144-231) for the CUDA backend.
// Same flags, same defaults, same log lines; `--backend cuda` is the only backend this binary contains.
//
//   ptb200-cli -f scenes/rtweekend1.ssml -s 64 -x 800 -y 450 -r mis -o out.png [--backend cuda] [--device 0]
//              [--gpus 1] [--seed 0] [--max-depth 50] [-b sah|middle|equal-counts (accepted, ignored: the device builds its own tree)]
// --gpus N renders on GPUs device .. device+N-1 through ptb_render_multi (samples split N ways, or bands of image rows
// when there are fewer samples than GPUs; one ncclReduce of the accumulators) — the rayon fan-out of random_sampler.rs:40-80.
// --denoise renders the first-hit feature buffers of the same camera samples (ptb_render_aov, on GPU `device` after the
// reduce) and writes the image ptb_denoise makes of them instead of the noisy one; use .pfm or .exr to keep it linear f32.
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <ctime>
#include <string>
#include <thread>
#include <vector>

#include "../../include/ptb200.h"

namespace {

struct Cli {
  bool gui = false;
  unsigned long long samples = 128;   // parameters.rs:25-26
  unsigned long long width = 1920;    // :27-28
  unsigned long long height = 1080;   // :29-30
  std::string filepath;               // :31-32 (required)
  std::string bvh_type = "sah";       // :33-34
  std::string render_method = "mis";  // :35-36
  std::string output;                 // :37-38
  float gamma = 2.2f;                 // :39-40
  std::string backend = "cuda";
  int device = 0;
  int gpus = 1;
  unsigned long long seed = 0;
  unsigned max_depth = 50;
  bool denoise = false;
};

void log_line(const char* level, const char* target, const std::string& msg) {
  // output/src/lib.rs:16-24: "{HH:MM:SS} {LEVEL} [{target}] {message}" on stderr
  char ts[16];
  std::time_t t = std::time(nullptr);
  std::strftime(ts, sizeof ts, "%H:%M:%S", std::localtime(&t));
  std::fprintf(stderr, "%s %s [%s] %s\n", ts, level, target, msg.c_str());
}

// output/src/lib.rs:33-62
std::string readable_duration(double secs_f) {
  unsigned long long secs = (unsigned long long)secs_f;
  unsigned long long days = secs / 86400, hours = (secs - days * 86400) / 3600,
                     minutes = (secs - days * 86400 - hours * 3600) / 60, seconds = secs % 60;
  std::string s;
  auto part = [&](unsigned long long v, const char* one, const char* many) {
    if (v == 0) return;
    s += std::to_string(v) + (v == 1 ? one : many);
  };
  part(days, " day, ", " days, ");
  part(hours, " hour, ", " hours, ");
  part(minutes, " minute, ", " minutes, ");
  if (seconds == 0) s += "~0 seconds";
  else s += std::to_string(seconds) + (seconds == 1 ? " second" : " seconds");
  return s;
}

int usage(const char* argv0, const char* err) {
  if (err) std::fprintf(stderr, "error: %s\n\n", err);
  std::fprintf(stderr,
               "An experimental pathtracer written in Rust — CUDA (B200) backend\n\n"
               "Usage: %s [OPTIONS] --filepath <FILEPATH>\n\n"
               "Options:\n"
               "  -g, --gui\n"
               "  -s, --samples <SAMPLES>              [default: 128]\n"
               "  -x, --width <WIDTH>                  [default: 1920]\n"
               "  -y, --height <HEIGHT>                [default: 1080]\n"
               "  -f, --filepath <FILEPATH>\n"
               "  -b, --bvh-type <BVH_TYPE>            [default: sah] [possible values: sah, middle, equal-counts]\n"
               "  -r, --render-method <RENDER_METHOD>  [default: mis] [possible values: naive, mis]\n"
               "  -o, --output <OUTPUT>\n"
               "      --gamma <GAMMA>                  [default: 2.2]\n"
               "      --backend <BACKEND>              [default: cuda] [possible values: cuda]\n"
               "      --device <INDEX>                 [default: 0]\n"
               "      --gpus <N>                       [default: 1] GPUs device .. device+N-1 of this box\n"
               "      --seed <SEED>                    [default: 0]\n"
               "      --max-depth <DEPTH>              [default: 50]\n"
               "      --denoise                        write the denoised image (spatial SVGF guided by first-hit albedo,\n"
               "                                       normal and depth of the same samples)\n",
               argv0);
  return 2;
}

struct Progress {
  unsigned long long total;
  unsigned long long last = ~0ull;
};
int32_t on_progress(void* user, uint64_t samples, uint64_t /*rays*/) {
  Progress* p = static_cast<Progress*>(user);
  if (samples != p->last) {  // indicatif-style bar of src/main.rs:167-190, reduced to one carriage-returned line
    p->last = samples;
    std::fprintf(stderr, "\r[%7llu/%-7llu]", (unsigned long long)samples, p->total);
    if (samples == p->total) std::fprintf(stderr, "\r%40s\r", "");
  }
  return 0;
}

}  // namespace

int main(int argc, char** argv) {
  Cli cli;
  for (int i = 1; i < argc; ++i) {
    std::string a = argv[i];
    auto value = [&](const char* name) -> const char* {
      if (i + 1 >= argc) { usage(argv[0], (std::string("missing value for ") + name).c_str()); std::exit(2); }
      return argv[++i];
    };
    if (a == "-g" || a == "--gui") cli.gui = true;
    else if (a == "-s" || a == "--samples") cli.samples = std::strtoull(value("--samples"), nullptr, 10);
    else if (a == "-x" || a == "--width") cli.width = std::strtoull(value("--width"), nullptr, 10);
    else if (a == "-y" || a == "--height") cli.height = std::strtoull(value("--height"), nullptr, 10);
    else if (a == "-f" || a == "--filepath") cli.filepath = value("--filepath");
    else if (a == "-b" || a == "--bvh-type") cli.bvh_type = value("--bvh-type");
    else if (a == "-r" || a == "--render-method") cli.render_method = value("--render-method");
    else if (a == "-o" || a == "--output") cli.output = value("--output");
    else if (a == "--gamma") cli.gamma = std::strtof(value("--gamma"), nullptr);
    else if (a == "--backend") cli.backend = value("--backend");
    else if (a == "--device") cli.device = std::atoi(value("--device"));
    else if (a == "--gpus") cli.gpus = std::atoi(value("--gpus"));
    else if (a == "--seed") cli.seed = std::strtoull(value("--seed"), nullptr, 10);
    else if (a == "--max-depth") cli.max_depth = (unsigned)std::atoi(value("--max-depth"));
    else if (a == "--denoise") cli.denoise = true;
    else if (a == "-h" || a == "--help") return usage(argv[0], nullptr), 0;
    else return usage(argv[0], ("unexpected argument '" + a + "'").c_str());
  }
  if (cli.filepath.empty()) return usage(argv[0], "the following required arguments were not provided: --filepath <FILEPATH>");
  if (cli.bvh_type != "sah" && cli.bvh_type != "middle" && cli.bvh_type != "equal-counts")
    return usage(argv[0], "invalid value for --bvh-type");
  if (cli.render_method != "naive" && cli.render_method != "mis") return usage(argv[0], "invalid value for --render-method");
  if (cli.backend != "cuda") return usage(argv[0], "this binary only contains the cuda backend (no CPU fallback)");
  if (cli.gpus < 1 || cli.gpus > 64) return usage(argv[0], "invalid value for --gpus");
  if (cli.gui) {  // src/main.rs:226-229
    std::printf("feature: gui not enabled\n");
    return 0;
  }

  // parameters.rs:48-58: load_file_full, panic on error
  log_line("INFO", "loader", "Loading textures...");
  ptb_host_scene* scene = nullptr;
  int32_t rc = ptb_ssml_load_file(cli.filepath.c_str(), &scene);
  if (rc != PTB_OK) {
    log_line("ERROR", "frontend", std::string("failed to load scene: ") + ptb_host_last_error());
    return 101;  // the reference panics here
  }
  // one context per GPU, the scene replicated on each (uploads and builds run concurrently, one host thread per GPU)
  std::vector<ptb_ctx*> ctxs((size_t)cli.gpus, nullptr);
  auto destroy_all = [&]() {
    for (ptb_ctx* c : ctxs) ptb_destroy(c);
    ptb_host_scene_free(scene);
  };
  for (int g = 0; g < cli.gpus; ++g)
    if ((rc = ptb_create(cli.device + g, &ctxs[(size_t)g])) != PTB_OK) {
      log_line("ERROR", "frontend", std::string("cuda backend unavailable: ") + ptb_last_error(nullptr));
      destroy_all();
      return 1;
    }
  ptb_ctx* ctx = ctxs[0];
  auto fail = [&](const char* what, ptb_ctx* which = nullptr) {
    log_line("ERROR", "frontend", std::string(what) + ": " + ptb_last_error(which ? which : ctx));
    destroy_all();
    return 1;
  };
  // --bvh-type (parameters.rs:35-36, split.rs SplitType): `sah` = the device's SAH builder (or what PTB_BVH says); `middle`
  // = the Karras LBVH, whose nodes split at the spatial middle of their Morton cell; `equal-counts` has no device builder
  // and gets the LBVH too. Every tree returns the same hits, so the image does not depend on the choice.
  const uint32_t build_flags = cli.bvh_type == "sah" ? (uint32_t)PTB_BUILD_DEFAULT : (uint32_t)PTB_BUILD_BINARY;
  {
    std::vector<int32_t> rcs((size_t)cli.gpus, PTB_OK);
    std::vector<std::thread> th;
    for (int g = 0; g < cli.gpus; ++g)
      th.emplace_back([&, g]() {
        int32_t r = ptb_scene_upload(ctxs[(size_t)g], scene);
        if (r == PTB_OK) r = ptb_scene_commit(ctxs[(size_t)g], build_flags);  // Bvh::new(primitives, sky, cli.bvh_type) (parameters.rs:61)
        rcs[(size_t)g] = r;
      });
    for (auto& t : th) t.join();
    for (int g = 0; g < cli.gpus; ++g)
      if (rcs[(size_t)g] != PTB_OK) return fail("scene upload / bvh build", ctxs[(size_t)g]);
  }
  if (cli.bvh_type == "equal-counts")
    log_line("WARN", "frontend", "--bvh-type equal-counts: the cuda backend has no equal-counts builder, using its spatial-middle tree (same image)");

  // output/src/lib.rs:126-136
  {
    char buf[256];
    std::snprintf(buf, sizeof buf, "Render started:\n\tWidth:\t\t%llu\n\tHeight:\t\t%llu\n\tGamma:\t\t%.3f\n\tSamples:\t%llu",
                  cli.width, cli.height, (double)cli.gamma, cli.samples);
    log_line("INFO", "output", buf);
  }
  const auto start = std::chrono::steady_clock::now();
  ptb_render_opts o{};
  o.width = (uint32_t)cli.width;
  o.height = (uint32_t)cli.height;
  o.samples_per_pixel = (uint32_t)cli.samples;
  o.sample_offset = 0;
  o.method = cli.render_method == "naive" ? PTB_METHOD_NAIVE : PTB_METHOD_MIS;
  o.max_depth = cli.max_depth;
  o.rr_threshold = PTB_RR_DEFAULT;
  o.seed = cli.seed;
  Progress prog{cli.samples};
  if (cli.gpus == 1) {
    if (ptb_render(ctx, &o, on_progress, &prog) != PTB_OK) return fail("render");
  } else {
    if (ptb_render_multi(ctxs.data(), cli.gpus, &o) != PTB_OK) return fail("multi-GPU render");
  }
  std::vector<float> image((size_t)cli.width * cli.height * 3);
  if (cli.denoise) {  // the feature buffers of the same samples, then the filter with its defaults
    ptb_denoise_opts d{};
    if (ptb_render_aov(ctx, &o) != PTB_OK) return fail("feature buffers");
    if (ptb_denoise(ctx, &d, image.data(), image.size()) != PTB_OK) return fail("denoise");
  } else if (ptb_accum_read(ctx, image.data(), image.size(), 1) != PTB_OK) {
    return fail("accumulator read-back");
  }
  const double secs = std::chrono::duration<double>(std::chrono::steady_clock::now() - start).count();
  ptb_stats st{};
  ptb_stats_get(ctx, &st);
  for (int g = 1; g < cli.gpus; ++g) {  // counters add up over the GPUs; times are the slowest GPU's
    ptb_stats s2{};
    ptb_stats_get(ctxs[(size_t)g], &s2);
    st.rays_camera += s2.rays_camera; st.rays_bounce += s2.rays_bounce; st.rays_shadow_light += s2.rays_shadow_light;
    st.rays_shadow_sky += s2.rays_shadow_sky; st.rays_reference += s2.rays_reference; st.kernel_launches += s2.kernel_launches;
    if (s2.render_ms > st.render_ms) st.render_ms = s2.render_ms;
    if (s2.build_ms > st.build_ms) st.build_ms = s2.build_ms;
  }

  // output/src/lib.rs:115-124 — the reference's own counter (Q7), then this backend's per-class counts
  {
    char buf[512];
    std::snprintf(buf, sizeof buf, "Finished rendering:\n\tSamples:\t%llu\n\tTime taken:\t%s\n\tRays shot:\t%llu @ %.2f Mray/s",
                  cli.samples, readable_duration(secs).c_str(), (unsigned long long)st.rays_reference,
                  (double)st.rays_reference / secs / 1e6);
    log_line("INFO", "output", buf);
    const unsigned long long all = st.rays_camera + st.rays_bounce + st.rays_shadow_light + st.rays_shadow_sky;
    std::snprintf(buf, sizeof buf,
                  "cuda backend: %llu traversals (camera %llu, bounce %llu, light-shadow %llu, sky-shadow %llu) @ %.2f Mray/s; "
                  "device render %.1f ms, bvh build %.2f ms, %llu kernel launches, %d GPU(s)",
                  all, (unsigned long long)st.rays_camera, (unsigned long long)st.rays_bounce,
                  (unsigned long long)st.rays_shadow_light, (unsigned long long)st.rays_shadow_sky, (double)all / secs / 1e6,
                  st.render_ms, st.build_ms, (unsigned long long)st.kernel_launches, cli.gpus);
    log_line("INFO", "output", buf);
  }
  int exit_code = 0;
  if (!cli.output.empty()) {  // src/main.rs:199-207
    rc = ptb_image_save(cli.output.c_str(), (uint32_t)cli.width, (uint32_t)cli.height, image.data(), cli.gamma);
    if (rc == PTB_OK) log_line("INFO", "output", "Image " + cli.output + " saved");
    else if (rc == PTB_ERR_INVALID) { std::printf("Invalid filename: %s\n", cli.output.c_str()); }
    else { log_line("ERROR", "output", "Unable to save file: " + cli.output); exit_code = 1; }
  }
  destroy_all();
  return exit_code;
}
