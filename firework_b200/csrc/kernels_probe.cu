// Probe kernels (the parity gates of BASELINE.json) and the roofline-denominator microbenchmarks.
#include "launch.h"
#include "wavefront.cuh"

namespace fw {

__global__ void primary_rays_probe(CameraRec cam, uint32_t width, uint32_t height, uint32_t sample, uint2 seed,
                                   uint32_t pix_begin, uint32_t n, float* origins, float* dirs) {
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        float3 o, d;
        primary_ray(cam, width, height, pix_begin + i, sample, seed, o, d);
        origins[3 * i] = o.x; origins[3 * i + 1] = o.y; origins[3 * i + 2] = o.z;
        dirs[3 * i] = d.x; dirs[3 * i + 1] = d.y; dirs[3 * i + 2] = d.z;
    }
}
template <bool USE_BVH>
__global__ void first_hit_probe(DeviceScene S, uint2 seed, uint32_t n, const float* origins, const float* dirs,
                                const uint32_t* pixel, const uint32_t* sample, const uint32_t* bounce,
                                FirstHitOut out) {
    Counters cnt{0, 0};
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        float3 o = f3(origins[3 * i], origins[3 * i + 1], origins[3 * i + 2]);
        float3 d = f3(dirs[3 * i], dirs[3 * i + 1], dirs[3 * i + 2]);
        RngKey key{seed, pixel ? pixel[i] : i, sample ? sample[i] : 0u, bounce ? bounce[i] : 0u};
        HitRecord rec;
        if (scene_closest_hit<USE_BVH, true>(S, o, d, key, rec, &cnt)) {
            out.obj[i] = rec.obj; out.prim[i] = rec.prim; out.material[i] = rec.material; out.t[i] = rec.t;
            out.point[3 * i] = rec.point.x; out.point[3 * i + 1] = rec.point.y; out.point[3 * i + 2] = rec.point.z;
            out.normal[3 * i] = rec.normal.x; out.normal[3 * i + 1] = rec.normal.y; out.normal[3 * i + 2] = rec.normal.z;
            out.uv[2 * i] = rec.uv.x; out.uv[2 * i + 1] = rec.uv.y;
        } else {
            out.obj[i] = -1; out.prim[i] = 0; out.material[i] = -1; out.t[i] = 0.0f;
            out.point[3 * i] = out.point[3 * i + 1] = out.point[3 * i + 2] = 0.0f;
            out.normal[3 * i] = out.normal[3 * i + 1] = out.normal[3 * i + 2] = 0.0f;
            out.uv[2 * i] = out.uv[2 * i + 1] = 0.0f;
        }
    }
    atomicAdd(&out.counters[0], cnt.node_tests);
    atomicAdd(&out.counters[1], cnt.prim_tests);
}

// first-hit probe through the LinProgram path (what linear-scan renders execute)
template <bool GENERIC>
__global__ void first_hit_prog_probe(const __grid_constant__ LinProgram P, DeviceScene S, uint2 seed, uint32_t n, const float* origins,
                                     const float* dirs, const uint32_t* pixel, const uint32_t* sample, const uint32_t* bounce,
                                     FirstHitOut out) {
    Counters cnt{0, 0};
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        float3 o = f3(origins[3 * i], origins[3 * i + 1], origins[3 * i + 2]);
        float3 d = f3(dirs[3 * i], dirs[3 * i + 1], dirs[3 * i + 2]);
        RngKey key{seed, pixel ? pixel[i] : i, sample ? sample[i] : 0u, bounce ? bounce[i] : 0u};
        Winner w;
        trace_linear_prog<true, GENERIC, true, false, !GENERIC>(P, S, o, d, key, w, &cnt);
        if (w.found) {
            HitRecord rec;
            finalize_hit(S, w, o, d, rec);
            out.obj[i] = rec.obj; out.prim[i] = rec.prim; out.material[i] = rec.material; out.t[i] = rec.t;
            out.point[3 * i] = rec.point.x; out.point[3 * i + 1] = rec.point.y; out.point[3 * i + 2] = rec.point.z;
            out.normal[3 * i] = rec.normal.x; out.normal[3 * i + 1] = rec.normal.y; out.normal[3 * i + 2] = rec.normal.z;
            out.uv[2 * i] = rec.uv.x; out.uv[2 * i + 1] = rec.uv.y;
        } else {
            out.obj[i] = -1; out.prim[i] = 0; out.material[i] = -1; out.t[i] = 0.0f;
            out.point[3 * i] = out.point[3 * i + 1] = out.point[3 * i + 2] = 0.0f;
            out.normal[3 * i] = out.normal[3 * i + 1] = out.normal[3 * i + 2] = 0.0f;
            out.uv[2 * i] = out.uv[2 * i + 1] = 0.0f;
        }
    }
    atomicAdd(&out.counters[0], cnt.node_tests);
    atomicAdd(&out.counters[1], cnt.prim_tests);
}
// One emit + scatter step per item.  Stream = ArrayStream: explicit uniforms; Stream = PhiloxStream: the keyed stream
// scatter_segment draws from, so the production sampler (random_in_unit_sphere_fresh) runs.
template <class Stream>
FW_DEV Stream scatter_probe_stream(const ScatterProbeIO& io, uint32_t i);
template <>
FW_DEV ArrayStream scatter_probe_stream<ArrayStream>(const ScatterProbeIO& io, uint32_t i) {
    return ArrayStream(io.uniforms + (size_t)i * io.nu, (int)io.nu);
}
template <>
FW_DEV PhiloxStream scatter_probe_stream<PhiloxStream>(const ScatterProbeIO& io, uint32_t i) {
    return PhiloxStream(RngKey{io.seed, io.pixel[i], io.sample[i], io.bounce[i]}, STREAM_SCATTER);
}
FW_DEV int scatter_probe_consumed(const ArrayStream& rng) { return rng.overrun ? -1 : rng.i; }
FW_DEV int scatter_probe_consumed(const PhiloxStream& rng) { return (int)rng.idx; }

template <class Stream>
__global__ void scatter_step_probe(DeviceScene S, uint32_t n, ScatterProbeIO io) {
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        int mat = io.material[i];
        const float4* mq = reinterpret_cast<const float4*>(&S.mats[mat]);
        float4 m0 = __ldg(mq), m1 = __ldg(mq + 1);
        int kind = __float_as_int(m0.x), tex = __float_as_int(m0.y);
        float3 in_d = f3(io.ray_d[3 * i], io.ray_d[3 * i + 1], io.ray_d[3 * i + 2]);
        float3 point = f3(io.hit_point[3 * i], io.hit_point[3 * i + 1], io.hit_point[3 * i + 2]);
        float3 normal = f3(io.hit_normal[3 * i], io.hit_normal[3 * i + 1], io.hit_normal[3 * i + 2]);
        float2 uv = make_float2(io.hit_uv[2 * i], io.hit_uv[2 * i + 1]);
        Stream rng = scatter_probe_stream<Stream>(io, i);
        ScatterOut out;
        out.scattered = false;
        out.attenuation = out.origin = out.dir = f3(0.0f, 0.0f, 0.0f);
        float3 emit = f3(0.0f, 0.0f, 0.0f);
        switch (kind) {
            case MAT_LAMBERTIAN: scatter_lambertian(S, tex, point, normal, uv, rng, out); break;
            case MAT_METAL: scatter_metal(f3(m1), m0.z, in_d, point, normal, rng, out); break;
            case MAT_DIELECTRIC: scatter_dielectric(m0.z, in_d, point, normal, rng, out); break;
            case MAT_EMISSIVE: emit = texture_sample(S, tex, uv, point); break;
            case MAT_ISOTROPIC: scatter_isotropic(S, tex, point, uv, rng, out); break;
        }
        if (!out.scattered) out.attenuation = out.origin = out.dir = f3(0.0f, 0.0f, 0.0f);
        io.emit[3 * i] = emit.x; io.emit[3 * i + 1] = emit.y; io.emit[3 * i + 2] = emit.z;
        io.scattered[i] = out.scattered ? 1 : 0;
        io.atten[3 * i] = out.attenuation.x; io.atten[3 * i + 1] = out.attenuation.y; io.atten[3 * i + 2] = out.attenuation.z;
        io.out_o[3 * i] = out.origin.x; io.out_o[3 * i + 1] = out.origin.y; io.out_o[3 * i + 2] = out.origin.z;
        io.out_d[3 * i] = out.dir.x; io.out_d[3 * i + 1] = out.dir.y; io.out_d[3 * i + 2] = out.dir.z;
        io.consumed[i] = scatter_probe_consumed(rng);
    }
}

// Self-test of intersect.cuh div_by / shared_div against the hardware's IEEE `/`: pseudo-random and adversarial
// operands around and inside the fast domain.  violations[0] counts results that differ in any bit where the helper
// promises the exact quotient (|n| >= 2^-60 or outside the fast domain), violations[1] counts tiny-numerator cases
// where either value reaches the only threshold it is ever compared with (t_min = 0.001).
__global__ void shared_division_probe(uint64_t n_pairs, uint2 seed, unsigned long long* violations) {
    unsigned long long bad = 0, bad_tiny = 0;
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n_pairs; i += (uint64_t)gridDim.x * blockDim.x) {
        uint4 r = philox4x32_10(make_uint4((uint32_t)i, (uint32_t)(i >> 32), 0x5d1fu, 7u), seed);
        // mantissas: random, or one of the adversarial patterns
        const uint32_t pat[8] = {0x000000u, 0x7fffffu, 0x000001u, 0x7ffffeu, 0x400000u, 0x3fffffu, 0x555555u, 0x2aaaaau};
        uint32_t mn = (r.z & 8u) ? pat[r.z & 7u] : (r.x & 0x7fffffu);
        uint32_t md = (r.z & 128u) ? pat[(r.z >> 4) & 7u] : (r.y & 0x7fffffu);
        int en = -70 + (int)((r.w & 0xffffu) % 133u);        // 2^-70 .. 2^62
        int ed = -42 + (int)((r.w >> 16) % 85u);              // 2^-42 .. 2^42
        uint32_t sn = (r.x >> 31) << 31, sd = (r.y >> 31) << 31;
        float n = __uint_as_float(sn | ((uint32_t)(en + 127) << 23) | mn);
        float d = __uint_as_float(sd | ((uint32_t)(ed + 127) << 23) | md);
        if ((r.z & 0xff00u) == 0x1100u) n = __uint_as_float(sn);   // exact zero numerators
        float want = n / d;
        float got = div_by<true>(n, d, shared_div(d));
        bool in_domain = fabsf(d) >= 9.094947017729282e-13f && fabsf(d) <= 1.099511627776e12f && fabsf(n) <= 1.152921504606846976e18f;
        bool tiny = in_domain && fabsf(n) < 8.673617379884035e-19f;   // 2^-60
        if (tiny) {
            if (!(fabsf(want) < 0.001f) || !(fabsf(got) < 0.001f)) ++bad_tiny;
        } else if (__float_as_uint(want) != __float_as_uint(got)) {
            ++bad;
        }
    }
    if (bad) atomicAdd(&violations[0], bad);
    if (bad_tiny) atomicAdd(&violations[1], bad_tiny);
}

__global__ void env_sample_probe(DeviceScene S, uint32_t n, const float* dirs, float* out) {
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        float3 c = environment_sample(S.env, f3(dirs[3 * i], dirs[3 * i + 1], dirs[3 * i + 2]));
        out[3 * i] = c.x; out[3 * i + 1] = c.y; out[3 * i + 2] = c.z;
    }
}
__global__ void texture_sample_probe(DeviceScene S, int tex, uint32_t n, const float* uv, const float* point, float* out) {
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        float3 c = texture_sample(S, tex, make_float2(uv[2 * i], uv[2 * i + 1]),
                                  f3(point[3 * i], point[3 * i + 1], point[3 * i + 2]));
        out[3 * i] = c.x; out[3 * i + 1] = c.y; out[3 * i + 2] = c.z;
    }
}

// ---- first-hit probe through the PRODUCTION extend kernels (fw_first_hit_wavefront) -----------------------------
// probe_fill_kernel plays raygen's role with caller-supplied rays (ray i = path i, dealt to the segments tile by tile);
// the scene's own extend kernels then run exactly as in a render; probe_collect_kernel reads every shade / miss queue
// back and rebuilds the full hit record with finalize_hit, the routine the shade kernels use.
__global__ void __launch_bounds__(FW_BLOCK) probe_fill_kernel(PathState ps, uint32_t n, const float* __restrict__ origins,
                                                              const float* __restrict__ dirs, uint32_t bounce) {
    const uint32_t seg = blockIdx.x;
    const size_t base = (size_t)seg * ps.seg_cap;
    uint32_t count = 0;
    for (uint32_t e = threadIdx.x; e < ps.seg_cap; e += FW_BLOCK) {
        uint32_t p = ((e / FW_TILE) * ps.nseg + seg) * FW_TILE + (e % FW_TILE);
        if (p >= n) break;
        ps.xo[bounce & 1][base + e] = make_float4(origins[3 * p], origins[3 * p + 1], origins[3 * p + 2], __uint_as_float(p));
        ps.xd[bounce & 1][base + e] = make_float4(dirs[3 * p], dirs[3 * p + 1], dirs[3 * p + 2], 0.0f);
        count = e + 1;
    }
    __shared__ uint32_t s_count;
    if (threadIdx.x == 0) s_count = 0;
    __syncthreads();
    if (count) atomicMax(&s_count, count);
    __syncthreads();
    if (threadIdx.x == 0) counter_row(ps, bounce, FW_Q_EXTEND)[seg] = s_count;
}
template <int K>
FW_DEV void probe_collect_queue(const DeviceScene& S, const PathState& ps, uint32_t bounce, const FirstHitOut& out) {
    const uint32_t total = counter_row(ps, bounce, K)[blockIdx.x];
    const uint32_t base = blockIdx.x * ps.seg_cap;
    for (uint32_t e = threadIdx.x; e < total; e += FW_BLOCK) {
        if (K == MAT_MISS) {
            const uint32_t i = __float_as_uint(ps.hq[K].d[base + e].w);
            out.obj[i] = -1; out.prim[i] = 0; out.material[i] = -1; out.t[i] = 0.0f;
            out.point[3 * i] = out.point[3 * i + 1] = out.point[3 * i + 2] = 0.0f;
            out.normal[3 * i] = out.normal[3 * i + 1] = out.normal[3 * i + 2] = 0.0f;
            out.uv[2 * i] = out.uv[2 * i + 1] = 0.0f;
            continue;
        }
        const HitIn h = get_hit<K>(ps, base + e);
        HitRecord rec;
        finalize_hit(S, h.w, h.o, h.d, rec);
        const uint32_t i = h.path;
        out.obj[i] = rec.obj; out.prim[i] = rec.prim; out.material[i] = rec.material; out.t[i] = rec.t;
        out.point[3 * i] = rec.point.x; out.point[3 * i + 1] = rec.point.y; out.point[3 * i + 2] = rec.point.z;
        out.normal[3 * i] = rec.normal.x; out.normal[3 * i + 1] = rec.normal.y; out.normal[3 * i + 2] = rec.normal.z;
        out.uv[2 * i] = rec.uv.x; out.uv[2 * i + 1] = rec.uv.y;
    }
}
__global__ void __launch_bounds__(FW_BLOCK) probe_collect_kernel(DeviceScene S, PathState ps, uint32_t bounce, FirstHitOut out) {
    probe_collect_queue<0>(S, ps, bounce, out); probe_collect_queue<1>(S, ps, bounce, out); probe_collect_queue<2>(S, ps, bounce, out);
    probe_collect_queue<3>(S, ps, bounce, out); probe_collect_queue<4>(S, ps, bounce, out); probe_collect_queue<5>(S, ps, bounce, out);
}
void launch_probe_fill(const PathState& ps, uint32_t n, const float* origins, const float* dirs, uint32_t bounce, cudaStream_t st) {
    probe_fill_kernel<<<ps.nseg, FW_BLOCK, 0, st>>>(ps, n, origins, dirs, bounce);
}
void launch_probe_collect(const DeviceScene& S, const PathState& ps, uint32_t bounce, const FirstHitOut& out, cudaStream_t st) {
    probe_collect_kernel<<<ps.nseg, FW_BLOCK, 0, st>>>(S, ps, bounce, out);
}

// ---- roofline denominators (fw_measure_peaks) --------------------------------------------------------------
__global__ void fp32_peak_kernel(float* out, int iters) {
    float a0 = threadIdx.x * 1e-3f, a1 = a0 + 1.f, a2 = a0 + 2.f, a3 = a0 + 3.f, a4 = a0 + 4.f, a5 = a0 + 5.f, a6 = a0 + 6.f, a7 = a0 + 7.f;
    const float m = 1.000001f, c = 1e-7f;
    for (int i = 0; i < iters; ++i) {
        a0 = __fmaf_rn(a0, m, c); a1 = __fmaf_rn(a1, m, c); a2 = __fmaf_rn(a2, m, c); a3 = __fmaf_rn(a3, m, c);
        a4 = __fmaf_rn(a4, m, c); a5 = __fmaf_rn(a5, m, c); a6 = __fmaf_rn(a6, m, c); a7 = __fmaf_rn(a7, m, c);
    }
    if (a0 + a1 + a2 + a3 + a4 + a5 + a6 + a7 == 123.456f) out[0] = a0;
}
__global__ void l2_read_kernel(const float4* __restrict__ buf, size_t n_vec, int reps, float* out) {
    float acc = 0.f;
    size_t stride = (size_t)gridDim.x * blockDim.x;
    for (int r = 0; r < reps; ++r)
        for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n_vec; i += stride) {
            float4 v = __ldcg(&buf[i]);  // cache-global: served by L2, bypasses L1
            acc += v.x + v.y + v.z + v.w;
        }
    if (acc == 123.456f) out[0] = acc;
}

// ---- launchers -------------------------------------------------------------------------------------------
void launch_primary_rays_probe(const CameraRec& cam, uint32_t width, uint32_t height, uint32_t sample, uint2 seed,
                               uint32_t pix_begin, uint32_t n, float* origins, float* dirs, unsigned blocks, cudaStream_t st) {
    primary_rays_probe<<<blocks, 256, 0, st>>>(cam, width, height, sample, seed, pix_begin, n, origins, dirs);
}
void launch_first_hit_probe(int mode, const LinProgram& prog, const DeviceScene& S, uint2 seed, uint32_t n, const float* origins,
                            const float* dirs, const uint32_t* pixel, const uint32_t* sample, const uint32_t* bounce,
                            const FirstHitOut& out, unsigned blocks, cudaStream_t st) {
    switch (mode) {
        case 1: first_hit_probe<true><<<blocks, 128, 0, st>>>(S, seed, n, origins, dirs, pixel, sample, bounce, out); break;
        case 2: first_hit_prog_probe<true><<<blocks, 128, 0, st>>>(prog, S, seed, n, origins, dirs, pixel, sample, bounce, out); break;
        case 3: first_hit_prog_probe<false><<<blocks, 128, 0, st>>>(prog, S, seed, n, origins, dirs, pixel, sample, bounce, out); break;
        default: first_hit_probe<false><<<blocks, 128, 0, st>>>(S, seed, n, origins, dirs, pixel, sample, bounce, out); break;
    }
}
void launch_scatter_step_probe(const DeviceScene& S, uint32_t n, const ScatterProbeIO& io, unsigned blocks, cudaStream_t st) {
    if (io.uniforms) scatter_step_probe<ArrayStream><<<blocks, 128, 0, st>>>(S, n, io);
    else scatter_step_probe<PhiloxStream><<<blocks, 128, 0, st>>>(S, n, io);
}
void launch_env_sample_probe(const DeviceScene& S, uint32_t n, const float* dirs, float* out, unsigned blocks, cudaStream_t st) {
    env_sample_probe<<<blocks, 256, 0, st>>>(S, n, dirs, out);
}
void launch_texture_sample_probe(const DeviceScene& S, int tex, uint32_t n, const float* uv, const float* point, float* out,
                                 unsigned blocks, cudaStream_t st) {
    texture_sample_probe<<<blocks, 256, 0, st>>>(S, tex, n, uv, point, out);
}
void launch_shared_division_probe(uint64_t n_pairs, uint2 seed, unsigned long long* violations) {
    shared_division_probe<<<148 * 8, 256>>>(n_pairs, seed, violations);
}
void launch_fp32_peak(float* out, int iters, int blocks, int threads) { fp32_peak_kernel<<<blocks, threads>>>(out, iters); }
void launch_l2_read(const float4* buf, size_t n_vec, int reps, float* out, int blocks, int threads) {
    l2_read_kernel<<<blocks, threads>>>(buf, n_vec, reps, out);
}

}  // namespace fw
