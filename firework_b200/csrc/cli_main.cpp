// firework — native command-line driver, the counterpart of the reference's src/main.rs:1-62 on top of the C ABI
// (SURVEY.md §8f row 1).  Same options (--scene-file, -n/--name, -s/--samples, -o/--output), the same hard-coded camera
// (0,30,50) -> (0,0,0), fov 40 and the same 960 x 540 BVH render (main.rs:28-38), the same two progress lines
// (main.rs:45, 54); the image is written as PNG (window.rs `save_image`).  Without --output the reference opens a
// window (out of scope here): the image goes to "<name>.png" instead.
//
// Extras (not in the reference): --width / --height / --seed, --gpus N (fw_render_multi: sample range split over N GPUs of
// the box), a .gz scene file is inflated on the fly, and --checkpoint FILE [--chunk N]: the samples are rendered N at a time,
// the fp32 sums and the number of samples done are saved after every chunk, and a later run with the same arguments continues
// where the file stops (SURVEY.md §8f row 2; the reference's 3.36 h render had no way to resume).  --target-error E
// [--min-samples N]: adaptive sampling (fw_render_adaptive), each pixel renders until its relative standard error is <= E,
// with -s as the cap per pixel; it owns its sample schedule, so it is refused together with --checkpoint, --chunk or --gpus > 1.
// --denoise: a denoised render (fw_render_denoised, default filter settings), refused with the same flags and --target-error.  The file format is shared
// with `python -m firework_b200 --checkpoint x.fwck` (firework_b200/progressive.py), so either driver finishes what the other began.
// Links libfirework_b200.a: nothing here goes through Python.
#include <zlib.h>

#include <algorithm>
#include <chrono>
#include <cmath>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

#include "../../include/firework_b200.h"

namespace {

void usage(FILE* f) {
    fprintf(f,
            "firework (B200)\n\nUSAGE:\n    firework [OPTIONS] --samples <samples> --scene-file <scene-file>\n\nOPTIONS:\n"
            "    -n, --name <name>\n    -o, --output <output>\n    -s, --samples <samples>\n        --scene-file <scene-file>\n"
            "        --width <px>       (default 960)\n        --height <px>      (default 540)\n        --seed <u64>       (default 0)\n"
            "        --gpus <n>         render on n GPUs of this box (default 1)\n"
            "        --checkpoint <f>   resume from / save to this file after every chunk\n        --chunk <n>        samples per chunk (default: all)\n"
            "        --target-error <e> adaptive sampling: render each pixel until its relative standard error <= e (-s is the cap)\n"
            "        --min-samples <n>  adaptive sampling: samples of the first round (default 16)\n"
            "        --denoise          filter the render with first-hit albedo / normal / depth as guides (-s >= 2)\n    -h, --help\n");
}
[[noreturn]] void die(const std::string& msg) {
    fprintf(stderr, "error: %s\n", msg.c_str());
    exit(1);
}
void check(int rc, const char* what) {
    if (rc != FW_OK) die(std::string(what) + ": " + fw_last_error());
}
bool ends_with(const std::string& s, const char* suffix) {
    size_t n = strlen(suffix);
    return s.size() >= n && s.compare(s.size() - n, n, suffix) == 0;
}
std::string dirname_of(const std::string& p) {
    size_t k = p.find_last_of('/');
    return k == std::string::npos ? std::string(".") : (k == 0 ? std::string("/") : p.substr(0, k));
}
std::string basename_of(const std::string& p) {
    size_t k = p.find_last_of('/');
    return k == std::string::npos ? p : p.substr(k + 1);
}
bool exists(const std::string& p) {
    FILE* f = fopen(p.c_str(), "rb");
    if (f) fclose(f);
    return f != nullptr;
}
// gzopen reads plain files transparently, so one path serves .yml and .yml.gz
std::string read_text(const std::string& path) {
    gzFile f = gzopen(path.c_str(), "rb");
    if (!f) die("cannot open scene file `" + path + "`");
    std::string text;
    char buf[1 << 16];
    int n;
    while ((n = gzread(f, buf, sizeof buf)) > 0) text.append(buf, (size_t)n);
    if (n < 0) { gzclose(f); die("cannot read scene file `" + path + "`"); }
    gzclose(f);
    return text;
}
// ImageTexture / HdrEnvironment paths are relative to the working directory in the reference (texture.rs:288); the
// committed scenes name bare files that live next to the scene or in its assets/ directory.
std::string resolve_asset(const std::string& scene_dir, const std::string& path) {
    const std::string cands[] = {path, scene_dir + "/" + path, scene_dir + "/" + basename_of(path), scene_dir + "/assets/" + basename_of(path)};
    for (const std::string& c : cands)
        if (exists(c)) return c;
    die("asset `" + path + "` not found (looked in ., " + scene_dir + " and " + scene_dir + "/assets)");
}

// ---- checkpoint file (shared with firework_b200/progressive.py) -----------------------------------------------------------
// "FWCKPT01" | u32 width | u32 height | u64 samples done | u64 seed | u64 fingerprint | f32 sums[height * width * 3]   (little endian)
// fingerprint = crc32 << 32 | adler32 (zlib) over the scene text followed by the packed render parameters: WHAT is being
// rendered, not how far.
uint64_t fingerprint(const std::string& yaml, const fw_params& p) {
    unsigned char packed[3 * 4 + 10 * 4 + 8];
    const uint32_t ints[3] = {p.width, p.height, p.use_bvh};
    const float flts[10] = {p.gamma, p.cam_pos[0], p.cam_pos[1], p.cam_pos[2], p.look_at[0], p.look_at[1], p.look_at[2], p.vfov, p.aperture, p.focus_dist};
    memcpy(packed, ints, 12); memcpy(packed + 12, flts, 40); memcpy(packed + 52, &p.seed, 8);
    uLong c = crc32(0L, reinterpret_cast<const Bytef*>(yaml.data()), (uInt)yaml.size());
    c = crc32(c, packed, sizeof packed);
    uLong a = adler32(1L, reinterpret_cast<const Bytef*>(yaml.data()), (uInt)yaml.size());
    a = adler32(a, packed, sizeof packed);
    return ((uint64_t)(c & 0xffffffffu) << 32) | (uint64_t)(a & 0xffffffffu);
}
struct CkHeader {
    char magic[8];
    uint32_t width, height;
    uint64_t done, seed, fp;
};
bool load_checkpoint(const std::string& path, const fw_params& p, uint64_t fp, std::vector<float>& sums, uint64_t& done) {
    FILE* f = fopen(path.c_str(), "rb");
    if (!f) return false;   // nothing to resume
    CkHeader h;
    const bool ok = fread(&h, sizeof h, 1, f) == 1 && !memcmp(h.magic, "FWCKPT01", 8);
    if (!ok) { fclose(f); die("`" + path + "` is not a firework checkpoint"); }
    if (h.width != p.width || h.height != p.height || h.seed != p.seed || h.fp != fp) {
        fclose(f);
        die("checkpoint does not match this render (scene, camera, renderer parameters or size differ)");
    }
    if (h.done > p.samples) { fclose(f); die("checkpoint holds " + std::to_string(h.done) + " samples but this render has " + std::to_string(p.samples)); }
    if (fread(sums.data(), sizeof(float), sums.size(), f) != sums.size()) { fclose(f); die("checkpoint `" + path + "` is truncated"); }
    fclose(f);
    done = h.done;
    return true;
}
void save_checkpoint(const std::string& path, const fw_params& p, uint64_t fp, const std::vector<float>& sums, uint64_t done) {
    const std::string tmp = path + ".tmp";
    FILE* f = fopen(tmp.c_str(), "wb");
    if (!f) die("cannot write `" + tmp + "`");
    CkHeader h;
    memcpy(h.magic, "FWCKPT01", 8);
    h.width = p.width; h.height = p.height; h.done = done; h.seed = p.seed; h.fp = fp;
    const bool ok = fwrite(&h, sizeof h, 1, f) == 1 && fwrite(sums.data(), sizeof(float), sums.size(), f) == sums.size();
    if (fclose(f) != 0 || !ok) die("short write to `" + tmp + "`");
    if (rename(tmp.c_str(), path.c_str()) != 0) die("cannot replace `" + path + "`");   // atomic: a killed run leaves the old file
}

}  // namespace

int main(int argc, char** argv) {
    std::string scene_file, name, output, checkpoint;
    long samples = -1, width = 960, height = 540, gpus = 1, chunk = 0, min_samples = 16;
    double target_error = -1.0;   // < 0: uniform render
    bool adaptive = false, denoise = false;
    unsigned long long seed = 0;
    for (int i = 1; i < argc; ++i) {
        std::string a = argv[i];
        auto value = [&](const char* opt) -> std::string {
            size_t eq = a.find('=');
            if (a.rfind("--", 0) == 0 && eq != std::string::npos) return a.substr(eq + 1);
            if (i + 1 >= argc) die(std::string("The argument '") + opt + "' requires a value");
            return argv[++i];
        };
        auto is = [&](const char* lng, const char* sht) {
            return a == lng || (sht && a == sht) || a.rfind(std::string(lng) + "=", 0) == 0;
        };
        if (is("--help", "-h")) { usage(stdout); return 0; }
        else if (is("--scene-file", nullptr)) scene_file = value("--scene-file <scene-file>");
        else if (is("--name", "-n")) name = value("--name <name>");
        else if (is("--samples", "-s")) samples = atol(value("--samples <samples>").c_str());
        else if (is("--output", "-o")) output = value("--output <output>");
        else if (is("--width", nullptr)) width = atol(value("--width").c_str());
        else if (is("--height", nullptr)) height = atol(value("--height").c_str());
        else if (is("--gpus", nullptr)) gpus = atol(value("--gpus").c_str());
        else if (is("--seed", nullptr)) seed = strtoull(value("--seed").c_str(), nullptr, 10);
        else if (is("--checkpoint", nullptr)) checkpoint = value("--checkpoint");
        else if (is("--chunk", nullptr)) chunk = atol(value("--chunk").c_str());
        else if (is("--target-error", nullptr)) { target_error = atof(value("--target-error <e>").c_str()); adaptive = true; }
        else if (is("--min-samples", nullptr)) min_samples = atol(value("--min-samples <n>").c_str());
        else if (a == "--denoise") denoise = true;
        else { usage(stderr); die("Found argument '" + a + "' which wasn't expected"); }
    }
    if (scene_file.empty() || samples < 0) {
        usage(stderr);
        die("The following required arguments were not provided: " + std::string(scene_file.empty() ? "--scene-file <scene-file> " : "") +
            (samples < 0 ? "--samples <samples>" : ""));
    }
    if (width <= 0 || height <= 0 || width > 65535 || height > 65535 || gpus < 1) die("bad --width / --height / --gpus");
    if (adaptive) {   // an adaptive render owns its sample schedule: no chunks, no checkpoint, one GPU
        if (!checkpoint.empty() || chunk > 0) die("--target-error can not be combined with --checkpoint or --chunk");
        if (gpus > 1) die("--target-error renders on one GPU: it can not be combined with --gpus > 1");
        if (!(target_error >= 0.0) || !std::isfinite(target_error) || min_samples < 1) die("--target-error must be finite and >= 0, --min-samples >= 1");
    }
    if (denoise) {    // a denoised render owns its sample range and needs the moments of one device
        if (!checkpoint.empty() || chunk > 0) die("--denoise can not be combined with --checkpoint or --chunk");
        if (gpus > 1) die("--denoise renders on one GPU: it can not be combined with --gpus > 1");
        if (adaptive) die("--denoise can not be combined with --target-error");
        if (samples < 2) die("--denoise needs --samples >= 2");
    }

    // main.rs:25-26
    const std::string text = read_text(scene_file);
    fw_scene* scene = nullptr;
    check(fw_scene_from_yaml(text.data(), text.size(), &scene), "scene");
    const std::string scene_dir = dirname_of(scene_file);
    for (int i = 0; i < fw_scene_num_assets(scene); ++i) {
        const std::string path = fw_scene_asset_path(scene, i);
        uint32_t w = 0, h = 0;
        if (fw_scene_asset_kind(scene, i) == 0) {                  // texture.rs:285-292
            uint8_t* rgba = nullptr;
            check(fw_image_load(resolve_asset(scene_dir, path).c_str(), &w, &h, &rgba), "image texture");
            check(fw_scene_set_image(scene, i, w, h, rgba), "image texture");
            fw_image_free(rgba);
        } else {                                                   // examples/hdri_test.rs:45-67
            float* rgb = nullptr;
            check(fw_hdr_load(resolve_asset(scene_dir, path).c_str(), &w, &h, &rgb), "environment map");
            check(fw_scene_set_hdr(scene, i, w, h, rgb), "environment map");
            fw_hdr_free(rgb);
        }
    }
    if (fw_device_count() < 1) die("no CUDA device (there is no CPU fallback)");
    check(fw_scene_commit(scene, 0), "commit");

    // main.rs:28-38
    fw_params p;
    memset(&p, 0, sizeof p);
    p.width = (uint32_t)width; p.height = (uint32_t)height;
    p.samples = (uint32_t)samples; p.sample_begin = 0; p.sample_count = (uint32_t)samples;
    p.use_bvh = 1;
    p.gamma = 2.2f;                                               // Renderer::default(), render.rs:57-70
    p.cam_pos[0] = 0.0f; p.cam_pos[1] = 30.0f; p.cam_pos[2] = 50.0f;
    p.look_at[0] = p.look_at[1] = p.look_at[2] = 0.0f;
    p.vfov = 40.0f; p.aperture = 0.0f; p.focus_dist = 10.0f;      // CameraSettings::default(), camera.rs:26-36
    p.seed = seed;

    std::vector<uint8_t> rgb((size_t)width * height * 3);
    fw_stats st;
    memset(&st, 0, sizeof st);
    const auto start = std::chrono::steady_clock::now();
    auto render_range = [&](const fw_params& q, uint8_t* rgb_out, float* sum_out) {
        if (gpus > 1) check(fw_render_multi(scene, &q, (int)gpus, nullptr, FW_REDUCE_NCCL, rgb_out, sum_out, &st, nullptr), "render");
        else check(fw_render(scene, &q, rgb_out, sum_out, &st), "render");
    };
    fw_adaptive_result ares;
    memset(&ares, 0, sizeof ares);
    if (denoise) {
        const fw_denoise dn{5, 4, 4.0f, 0.1f, 0.1f};   // engine.DENOISE_DEFAULTS
        check(fw_render_denoised(scene, &p, &dn, rgb.data(), nullptr, nullptr, nullptr, nullptr, &st), "render");
    } else if (adaptive) {
        fw_adaptive ad;
        ad.min_samples = (uint32_t)min_samples; ad.threshold = (float)target_error; ad.floor = 0.01f;   // engine.ADAPTIVE_FLOOR
        check(fw_render_adaptive(scene, &p, &ad, rgb.data(), nullptr, nullptr, nullptr, &st, &ares), "render");
    } else if (checkpoint.empty() && chunk <= 0) {
        render_range(p, rgb.data(), nullptr);
    } else {
        // sample-range chunks: RNG streams are keyed by the global sample index, so [0, k) now and [k, n) later are the
        // samples of one render of [0, n); the per-pixel sums are added in chunk order
        const size_t nval = (size_t)width * height * 3;
        std::vector<float> sums(nval, 0.0f), part(nval);
        const uint64_t fp = fingerprint(text, p);
        uint64_t done = 0;
        if (!checkpoint.empty() && load_checkpoint(checkpoint, p, fp, sums, done)) printf("Resuming at sample %llu of %ld\n", (unsigned long long)done, samples);
        const uint64_t step = chunk > 0 ? (uint64_t)chunk : (uint64_t)std::max(samples, 1l);
        while (done < (uint64_t)samples) {
            fw_params q = p;
            q.sample_begin = (uint32_t)done;
            q.sample_count = (uint32_t)std::min<uint64_t>(step, (uint64_t)samples - done);
            render_range(q, nullptr, part.data());
            for (size_t i = 0; i < nval; ++i) sums[i] += part[i];
            done += q.sample_count;
            if (!checkpoint.empty()) save_checkpoint(checkpoint, p, fp, sums, done);
        }
        check(fw_resolve_host(0, sums.data(), (uint32_t)((size_t)width * height), (uint32_t)std::max<uint64_t>(done, 1), p.gamma, rgb.data()), "resolve");
    }
    const auto end = std::chrono::steady_clock::now();
    printf("Finished Rendering in %lld s\n", (long long)std::chrono::duration_cast<std::chrono::seconds>(end - start).count());
    if (adaptive)
        printf("Adaptive: %llu samples in %u rounds, %.2f spp mean (cap %ld)\n", (unsigned long long)ares.samples, ares.rounds,
               (double)ares.samples / ((double)width * height), samples);
    fw_scene_destroy(scene);

    if (name.empty()) name = "Firework Render";
    if (output.empty()) {
        output = name + ".png";
        for (char& c : output)
            if (c == ' ') c = '_';
    }
    printf("Saving image to \"%s\"\n", output.c_str());
    check(fw_png_write(output.c_str(), (uint32_t)width, (uint32_t)height, rgb.data()), "save");
    return 0;
}
