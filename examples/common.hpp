// Shared main() of the restated examples: `--yaml` prints serde_yaml::to_string(&scene) and exits (no GPU needed); otherwise the
// scene is rendered like the crate's example does and — instead of opening a window (window.rs, out of scope) — saved as PNG.
#pragma once
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>

#include "../include/firework.hpp"

inline int run_example(int argc, char** argv, const char* title, const firework::Scene& scene, firework::Renderer renderer) {
    std::string out = std::string(title) + ".png";
    for (char& c : out)
        if (c == ' ') c = '_';
    float target_error = -1.0f;
    uint32_t min_samples = 16;
    bool denoise = false;
    for (int i = 1; i < argc; ++i) {
        const std::string a = argv[i];
        auto next = [&]() -> const char* { if (i + 1 >= argc) { fprintf(stderr, "error: %s needs a value\n", a.c_str()); exit(1); } return argv[++i]; };
        if (a == "--yaml") { fputs(scene.to_yaml().c_str(), stdout); return 0; }
        else if (a == "--samples" || a == "-s") renderer = renderer.samples((size_t)atol(next()));
        else if (a == "--width") renderer = renderer.width((size_t)atol(next()));
        else if (a == "--height") renderer = renderer.height((size_t)atol(next()));
        else if (a == "--seed") renderer = renderer.seed(strtoull(next(), nullptr, 10));
        else if (a == "--gpus") renderer = renderer.gpus(atoi(next()));
        else if (a == "--target-error") target_error = (float)atof(next());
        else if (a == "--min-samples") min_samples = (uint32_t)atol(next());
        else if (a == "--denoise") denoise = true;
        else if (a == "--asset-dir") renderer = renderer.asset_dir(next());
        else if (a == "--output" || a == "-o") out = next();
        else { fprintf(stderr, "usage: %s [--yaml] [-s samples] [--width w] [--height h] [--seed n] [--gpus n] [--target-error e] [--min-samples n] [--denoise] [--asset-dir d] [-o out.png]\n", argv[0]); return 1; }
    }
    if (target_error >= 0.0f) renderer = renderer.adaptive(target_error, min_samples);
    if (denoise) renderer = renderer.denoise();
    try {
        const auto start = std::chrono::steady_clock::now();
        const std::vector<firework::Color> render = renderer.render(scene);
        const auto end = std::chrono::steady_clock::now();
        printf("Finished Rendering in %lld s\n", (long long)std::chrono::duration_cast<std::chrono::seconds>(end - start).count());
        firework::save_image(render, out, renderer.width_, renderer.height_);
        printf("Saved %s\n", out.c_str());
    } catch (const firework::Error& e) {
        fprintf(stderr, "error: %s\n", e.what());
        return 1;
    }
    return 0;
}
