// Renderer::trace_rays of the C++ mirror (include/firework.hpp) for tests/test_gpu_trace.py:
//   trace_rays_mirror <scene.yml> <asset dir> <samples> <seed> <use_bvh> <n> <rays.f32> <means.f32>
// rays.f32 holds the origins then the directions (3 n or samples * 3 n floats each); means.f32 receives 3 n floats.
#include <cstdio>
#include <cstdlib>
#include <fstream>
#include <sstream>

#include "../include/firework.hpp"

int main(int argc, char** argv) {
    if (argc != 9) { fprintf(stderr, "usage: %s scene.yml asset_dir samples seed use_bvh n rays.f32 means.f32\n", argv[0]); return 2; }
    std::ifstream yf(argv[1]);
    std::stringstream yaml;
    yaml << yf.rdbuf();
    const size_t samples = (size_t)atol(argv[3]), n = (size_t)atol(argv[6]);
    std::ifstream rf(argv[7], std::ios::binary | std::ios::ate);
    const size_t floats = (size_t)rf.tellg() / sizeof(float);
    rf.seekg(0);
    std::vector<float> origins(floats / 2), dirs(floats / 2);
    rf.read(reinterpret_cast<char*>(origins.data()), origins.size() * sizeof(float));
    rf.read(reinterpret_cast<char*>(dirs.data()), dirs.size() * sizeof(float));
    try {
        const firework::Renderer r = firework::Renderer::default_().samples(samples).seed(strtoull(argv[4], nullptr, 10)).use_bvh(atoi(argv[5]) != 0).asset_dir(argv[2]);
        const std::vector<float> means = r.trace_rays_yaml(yaml.str(), n, origins, dirs);
        std::ofstream out(argv[8], std::ios::binary);
        out.write(reinterpret_cast<const char*>(means.data()), means.size() * sizeof(float));
    } catch (const firework::Error& e) {
        fprintf(stderr, "error: %s\n", e.what());
        return 1;
    }
    return 0;
}
