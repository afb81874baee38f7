// cli_main.cpp — `lumilly <scene.toml>`: the reference's command line (src/main.rs:43-145) on top of the C ABI.
// Prints the same progress lines (start / loading / resolution / spp / threads / integrator / polygons /
// bvh construction / saving... / end / elapse) plus GPU throughput, and writes
// images/image_<YYYYmmddHHMMSS>_<spp>.<png|hdr> (main.rs:147-169).  Errors that the reference turns into
// panics become a message on stderr and a non-zero exit status.
//
// Extra, optional arguments (not in the reference):  --spp N  --resolution WxH  --seed S  --device D
//   --gpus N (render on devices D..D+N-1 of this box from this one process: lr_render_multi, samples sharded by index;
//   with --progress the film is sharded by pixel tile, and its checkpoints resume under any other --gpus)
//   --assets DIR (root that mesh/IBL paths are resolved against; default: the current directory, like the reference)
//   --progress N (render N samples per pixel at a time through an LrMultiFilm and print the progress line main.rs:81-91 left
//   commented out)  --checkpoint FILE (with --progress: the film is saved after every chunk, and an existing FILE is
//   resumed — bit for bit the image of an uninterrupted run)  --aov normal|depth (Scene::normal / Scene::depth,
//   scene.rs:48-62, instead of the radiance; depth is written normalised to its maximum)
#include <sys/stat.h>

#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <ctime>
#include <string>
#include <vector>

#include "lumilly.h"

static int die(const char* what) {
  std::fprintf(stderr, "error: %s: %s\n", what, lr_last_error());
  return 1;
}

static std::string stamp(const char* fmt) {
  char buf[64];
  std::time_t t = std::time(nullptr);
  std::tm tm_buf;
  localtime_r(&t, &tm_buf);
  std::strftime(buf, sizeof(buf), fmt, &tm_buf);
  return buf;
}

int main(int argc, char** argv) {
  const auto t_start = std::chrono::steady_clock::now();
  std::printf("start: %s\n", stamp("%Y-%m-%dT%H:%M:%S%z").c_str());
  const char* scene_path = nullptr;
  const char* assets = nullptr;
  const char* checkpoint = nullptr;
  const char* aov = nullptr;
  int spp = -1, ow = 0, oh = 0, device = 0, gpus = 1, progress = 0;
  unsigned long long seed = 0;
  for (int i = 1; i < argc; i++) {
    const std::string a = argv[i];
    auto need = [&](const char* flag) -> const char* {
      if (i + 1 >= argc) { std::fprintf(stderr, "error: %s needs a value\n", flag); std::exit(2); }
      return argv[++i];
    };
    if (a == "--spp") spp = std::atoi(need("--spp"));
    else if (a == "--resolution") { if (std::sscanf(need("--resolution"), "%dx%d", &ow, &oh) != 2) { std::fprintf(stderr, "error: --resolution WxH\n"); return 2; } }
    else if (a == "--seed") seed = std::strtoull(need("--seed"), nullptr, 10);
    else if (a == "--device") device = std::atoi(need("--device"));
    else if (a == "--gpus") gpus = std::atoi(need("--gpus"));
    else if (a == "--assets") assets = need("--assets");
    else if (a == "--progress") progress = std::atoi(need("--progress"));
    else if (a == "--checkpoint") checkpoint = need("--checkpoint");
    else if (a == "--aov") aov = need("--aov");
    else if (!scene_path) scene_path = argv[i];
    else { std::fprintf(stderr, "error: unexpected argument `%s`\n", argv[i]); return 2; }
  }
  if (!scene_path) { std::fprintf(stderr, "Path for .toml must be specified.\n"); return 2; }   // main.rs:47-49
  if (aov && std::strcmp(aov, "normal") != 0 && std::strcmp(aov, "depth") != 0) { std::fprintf(stderr, "error: --aov normal|depth\n"); return 2; }
  if (checkpoint && progress <= 0) { std::fprintf(stderr, "error: --checkpoint needs --progress N\n"); return 2; }
  if (gpus > 8) { std::fprintf(stderr, "error: --gpus takes 1..8\n"); return 2; }
  if (aov && gpus > 1) { std::fprintf(stderr, "error: --aov renders on one GPU\n"); return 2; }
  std::printf("loading: %s\n", scene_path);

  LrHostScene* hs = nullptr;
  if (lr_host_scene_load(scene_path, assets, ow, oh, &hs) != LR_OK) return die("loading scene");
  LrSceneConfig cfg;
  lr_host_scene_config(hs, &cfg);
  if (spp > 0) cfg.samples = spp;
  std::printf("resolution: %dx%d\n", cfg.width, cfg.height);
  std::printf("spp: %d\n", cfg.samples);
  if (lr_init(device) != LR_OK) return die("initialising the GPU");
  int sms = 0;
  char name[128] = "";
  lr_device_info(&sms, nullptr, nullptr, name, sizeof(name));
  std::printf("threads: %d SMs (%s)\n", sms, name);
  std::printf("integrator: %s\n", cfg.integrator == LR_INTEGRATOR_PT ? "pt" : "pt-direct");
  std::printf("polygons: %d\n", cfg.n_prims);                                   // description.rs:66
  std::printf("bvh construction: %gs\n", cfg.bvh_build_seconds);                 // description.rs:70-73

  const bool film = progress > 0 && !aov;
  LrScene* scene = nullptr;
  if (gpus <= 1 && !film && lr_scene_create(lr_host_scene_desc(hs), &scene) != LR_OK) return die("uploading scene");
  LrRenderParams p;
  std::memset(&p, 0, sizeof(p));
  p.integrator = cfg.integrator; p.spp_begin = 0; p.spp_count = cfg.samples;
  p.depth = cfg.depth; p.depth_limit = cfg.depth_limit; p.no_direct_emitter = cfg.no_direct_emitter; p.seed = seed;
  std::vector<float> img((size_t)cfg.width * cfg.height * 3);
  LrStats st;
  int32_t devices[8];
  for (int i = 0; i < 8; i++) devices[i] = device + i;
  if (gpus > 1 && progress <= 0) {
    std::printf("gpus: %d (devices %d..%d, samples sharded by index, one peer-reading reduce)\n", gpus, device, device + gpus - 1);
    if (lr_render_multi(lr_host_scene_desc(hs), &p, gpus, devices, img.data(), nullptr, &st) != LR_OK) return die("rendering");
  } else if (aov) {
    std::memset(&st, 0, sizeof(st));
    const bool normal = std::strcmp(aov, "normal") == 0;
    std::vector<float> buf((size_t)cfg.width * cfg.height * (normal ? 3 : 1));
    if (lr_render_aov(scene, &p, normal ? LR_AOV_NORMAL : LR_AOV_DEPTH, buf.data()) != LR_OK) return die("rendering the AOV");
    if (normal) img = buf;
    else {
      float mx = 0.0f;
      for (float v : buf) mx = v > mx ? v : mx;
      for (size_t i = 0; i < buf.size(); i++) img[3 * i] = img[3 * i + 1] = img[3 * i + 2] = mx > 0.0f ? buf[i] / mx : 0.0f;
    }
    std::printf("aov: %s\n", aov);
  } else if (film) {
    // the progress hook of main.rs:81-91 (chunks of samples instead of pixels), resumable through a checkpoint file; the
    // film is sharded by pixel over the devices, so its image and its checkpoints do not depend on --gpus
    p.splits = 1;                                             // samples are added in order: any cut of the range gives the same bits
    LrMultiScene* ms = nullptr;
    LrMultiFilm* mfilm = nullptr;
    if (gpus > 1) std::printf("gpus: %d (devices %d..%d, pixels sharded by tile)\n", gpus, device, device + gpus - 1);
    if (lr_multi_scene_create(lr_host_scene_desc(hs), gpus > 1 ? gpus : 1, devices, &ms) != LR_OK) return die("uploading scene");
    struct stat sb;
    if (checkpoint && stat(checkpoint, &sb) == 0) {
      if (lr_multi_film_load(ms, checkpoint, &mfilm) != LR_OK) return die("resuming the checkpoint");
    } else if (lr_multi_film_create(ms, &p, 0, &mfilm) != LR_OK) return die("creating the film");
    int32_t done = 0;
    lr_multi_film_info(mfilm, &done, nullptr, nullptr, nullptr);
    if (done > 0) std::printf("resuming: %d of %d spp are in %s\n", done, cfg.samples, checkpoint);
    std::memset(&st, 0, sizeof(st));
    while (done < cfg.samples) {
      const int n = cfg.samples - done < progress ? cfg.samples - done : progress;
      LrStats part;
      if (lr_multi_film_render(mfilm, n, &part) != LR_OK) return die("rendering");
      done += n;
      st.kernel_ms += part.kernel_ms; st.samples += part.samples; st.rays += part.rays; st.nonfinite_samples += part.nonfinite_samples;
      if (checkpoint && lr_multi_film_save(mfilm, checkpoint) != LR_OK) return die("writing the checkpoint");
      std::printf("\rprocessing... (%d/%d : %.0f%%) ", done, cfg.samples, 100.0 * done / cfg.samples);
      std::fflush(stdout);
    }
    std::printf("\n");
    if (lr_multi_film_read(mfilm, img.data(), nullptr) != LR_OK) return die("reading the film");
    lr_multi_film_destroy(mfilm);
    lr_multi_scene_destroy(ms);
  } else if (lr_render(scene, &p, img.data(), nullptr, &st) != LR_OK) return die("rendering");
  if (!aov) std::printf("render: %.3f ms on the GPU, %.1f Msamples/s, %.1f Mrays/s, %llu non-finite samples\n", st.kernel_ms,
              st.samples / (st.kernel_ms * 1e3), st.rays / (st.kernel_ms * 1e3), (unsigned long long)st.nonfinite_samples);

  std::printf("\nsaving...\n");
  mkdir("images", 0755);
  const std::string out = "images/image_" + stamp("%Y%m%d%H%M%S") + "_" + std::to_string(cfg.samples) + (cfg.output == 0 ? ".png" : ".hdr");
  const int rc = cfg.output == 0 ? lr_save_png(out.c_str(), img.data(), cfg.width, cfg.height, cfg.gamma)
                                 : lr_save_hdr(out.c_str(), img.data(), cfg.width, cfg.height);
  if (rc != LR_OK) return die("saving image");
  std::printf("wrote: %s\n", out.c_str());
  lr_scene_destroy(scene);
  lr_host_scene_free(hs);
  lr_shutdown();
  std::printf("end: %s\n", stamp("%Y-%m-%dT%H:%M:%S%z").c_str());
  std::printf("elapse: %gs\n", std::chrono::duration<float>(std::chrono::steady_clock::now() - t_start).count());
  return 0;
}
