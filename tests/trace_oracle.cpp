// orc_trace_rays: the CPU oracle's counterpart of fw_trace_rays (DESIGN.md §13).  Test infrastructure only: compiled by
// tests/test_gpu_trace.py together with the unchanged oracle source, so the paths are the oracle's own color() (render.rs:12-33).
// Ray i of sample s starts one path keyed exactly as orc_render keys a camera ray: (pixel = keys ? keys[i] : i, sample s); its
// radiances are added in sample order into sum_out[3i .. 3i+2].  per_sample: the ray of (i, s) is entry (s - sample_begin) * n + i.
#include "../oracle/firework_oracle.cpp"

extern "C" int orc_trace_rays(void* sp, uint32_t n, const float* origins, const float* dirs, const uint32_t* keys, int per_sample,
                              uint32_t sample_begin, uint32_t sample_count, uint64_t seed, int use_bvh, float* sum_out) {
    Scene* s = (Scene*)sp;
    if (use_bvh && !s->bvh) return -2;
#pragma omp parallel for schedule(dynamic, 16)
    for (int64_t i = 0; i < (int64_t)n; ++i) {
        Rng rng;
        rng.seed(seed);
        Vec3 total = v3(0, 0, 0);
        for (uint32_t si = 0; si < sample_count; ++si) {
            const size_t k = per_sample ? (size_t)si * n + (size_t)i : (size_t)i;
            rng.begin(keys ? keys[i] : (uint32_t)i, sample_begin + si);
            Ray ray{v3(origins[3 * k], origins[3 * k + 1], origins[3 * k + 2]), v3(dirs[3 * k], dirs[3 * k + 1], dirs[3 * k + 2])};
            total = total + color(ray, *s, use_bvh != 0, 0, rng);
        }
        sum_out[3 * i] = total.x; sum_out[3 * i + 1] = total.y; sum_out[3 * i + 2] = total.z;
    }
    return 0;
}
