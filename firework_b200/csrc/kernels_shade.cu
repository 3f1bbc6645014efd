// Ray generation, shading, miss, accumulation and resolve kernels (and fw_render_multi's fused peer reduce + resolve).
#include "launch.h"
#include "wavefront.cuh"

namespace fw {

// One block per segment.  Tile t (FW_TILE consecutive paths) belongs to segment t % nseg, so every segment gets an
// even mix of the image; entry e of segment `seg` is path ((e / TILE) * nseg + seg) * TILE + e % TILE.  The rays
// go straight into the segment's bounce-0 extend queue.
template <bool LIST>
__global__ void __launch_bounds__(FW_BLOCK) raygen_kernel(CameraRec cam, Batch b, uint2 seed, PathState ps) {
    const uint32_t total = b.npix * b.ns;
    const uint32_t seg = blockIdx.x;
    const size_t base = (size_t)seg * ps.seg_cap;
    uint32_t count = 0;
    for (uint32_t e = threadIdx.x; e < ps.seg_cap; e += FW_BLOCK) {
        uint32_t p = ((e / FW_TILE) * ps.nseg + seg) * FW_TILE + (e % FW_TILE);
        if (p >= total) break;   // p grows with e: the valid entries are a prefix
        uint32_t pixel, sample;
        batch_path<LIST>(b, p, pixel, sample);
        float3 o, d;
        uint32_t row, px;
        div_magic(pixel, b.width, b.width_magic, row, px);
        primary_ray_at(cam, b.width, b.height, px, row, pixel, sample, seed, o, d);
        st_stream(&ps.xo[0][base + e], make_float4(o.x, o.y, o.z, __uint_as_float(p)));
        st_stream(&ps.xd[0][base + e], make_float4(d.x, d.y, d.z, 0.0f));
        st_stream(&ps.radiance[p], make_float4(0.0f, 0.0f, 0.0f, 0.0f));
        count = e + 1;
    }
    // the segment's entry count = 1 + the largest valid e over the block
    __shared__ uint32_t s_count;
    if (threadIdx.x == 0) s_count = 0;
    __syncthreads();
    if (count) atomicMax(&s_count, count);
    __syncthreads();
    if (threadIdx.x == 0) counter_row(ps, 0, FW_Q_EXTEND)[seg] = s_count;
}

// render.rs:23 evaluated without recursion: colour = a0 * (a1 * (... (a_{k-1} * terminal))) with the same
// right-nested association as `emit + attenuation * color(...)`; emit is zero at every scattering vertex
// (material.rs:13-15), so the chain of attenuations is all that is needed.
FW_DEV float3 fold_radiance(const PathState& ps, uint32_t path, uint32_t bounce, float3 terminal) {
    // all loads first (independent, one HBM round trip), then the multiplications in the reference's order
    float4 a[FW_MAX_DEPTH];
#pragma unroll
    for (int k = 0; k < FW_MAX_DEPTH; ++k)
        if (k < (int)bounce) a[k] = ld_stream(&ps.atten[(size_t)k * ps.cap + path]);
    float3 x = terminal;
#pragma unroll
    for (int k = FW_MAX_DEPTH - 1; k >= 0; --k)
        if (k < (int)bounce) x = f3(a[k].x, a[k].y, a[k].z) * x;
    return x;
}

// render.rs:31 — environment lookup for rays that left the scene
// BLACK_ENV: the environment is a black ColorEnv, so an escaping path returns chain * 0 = exactly 0 — which the radiance
// buffer already holds — unless some attenuation of the batch was NaN / inf / huge (NaN * 0 = NaN must survive, e.g. noise
// textures evaluated at a non-finite hit point).  The shade kernels raise ps.poison for such a value; without it the
// whole kernel is a no-op and returns at once (no attenuation chain is read at all).
template <bool BLACK_ENV>
FW_DEV void miss_segment(const DeviceScene& S, const PathState& ps, uint32_t bounce, uint32_t seg) {
    if (BLACK_ENV && *reinterpret_cast<volatile uint32_t*>(ps.poison) == 0u) return;
    const uint32_t total = counter_row(ps, bounce, MAT_MISS)[seg];
    const float4* qd = ps.hq[MAT_MISS].d + (size_t)seg * ps.seg_cap;
    for (uint32_t i = threadIdx.x; i < total; i += FW_BLOCK) {
        float4 rec = ld_stream(&qd[i]);
        uint32_t path = __float_as_uint(rec.w);
        float3 env = environment_sample(S.env, f3(rec));
        float3 c = fold_radiance(ps, path, bounce, env);
        st_stream(&ps.radiance[path], make_float4(c.x, c.y, c.z, 0.0f));
    }
}
template <bool BLACK_ENV>
__global__ void __launch_bounds__(FW_BLOCK) miss_kernel(DeviceScene S, PathState ps, uint32_t bounce) {
    miss_segment<BLACK_ENV>(S, ps, bounce, blockIdx.x);
}

// render.rs:20,25-28 with material.rs:174-180 — emissive surfaces end the path with their texture value
FW_DEV void emissive_segment(const DeviceScene& S, const PathState& ps, uint32_t bounce, uint32_t seg) {
    const uint32_t total = counter_row(ps, bounce, MAT_EMISSIVE)[seg];
    const uint32_t base = seg * ps.seg_cap;
    for (uint32_t i = threadIdx.x; i < total; i += FW_BLOCK) {
        HitIn h = get_hit<MAT_EMISSIVE>(ps, base + i);
        HitRecord rec;
        finalize_hit(S, h.w, h.o, h.d, rec, true);
        int tex = __ldg(&S.mats[h.material].tex);
        float3 emit = texture_sample(S, tex, rec.uv, rec.point);
        float3 c = fold_radiance(ps, h.path, bounce, emit);
        st_stream(&ps.radiance[h.path], make_float4(c.x, c.y, c.z, 0.0f));
    }
}
__global__ void __launch_bounds__(FW_BLOCK) shade_emissive_kernel(DeviceScene S, PathState ps, uint32_t bounce) {
    emissive_segment(S, ps, bounce, blockIdx.x);
}

// Scattering materials: the next ray goes into the next extend queue, this vertex's attenuation into the chain.
// Not launched for bounce == FW_MAX_DEPTH (render.rs:21: no scatter at depth 10; emit is zero).
// The material kernels of one bounce run back to back and append to the same regions of the next extend queue.
// The entries of material MAT's queue of one segment; s_fill[0] is the segment's open fill count of the next extend queue.
template <int MAT, bool LIST>
FW_DEV void scatter_segment(const DeviceScene& S, const PathState& ps, const Batch& b, uint2 seed, uint32_t bounce, uint32_t seg, uint32_t total,
                            uint32_t* s_fill) {
    const uint32_t base = seg * ps.seg_cap;
    float4* __restrict__ xo = ps.xo[(bounce + 1) & 1];
    float4* __restrict__ xd = ps.xd[(bounce + 1) & 1];
    for (uint32_t e0 = 0; e0 < total; e0 += FW_BLOCK) {
        uint32_t i = e0 + threadIdx.x;
        int mine = -1;
        uint32_t path = 0;
        ScatterOut out;
        out.scattered = false;
        out.origin = out.dir = out.attenuation = f3(0.0f, 0.0f, 0.0f);
        if (i + FW_BLOCK < total) {
            prefetch_l2(&ps.hq[MAT].o[base + i + FW_BLOCK]); prefetch_l2(&ps.hq[MAT].d[base + i + FW_BLOCK]);
            prefetch_l2(&ps.hq[MAT].w[base + i + FW_BLOCK]);
        }
        if (i < total) {
            HitIn h = get_hit<MAT>(ps, base + i);
            path = h.path;
            const float4* mq = reinterpret_cast<const float4*>(&S.mats[h.material]);
            float4 m0 = __ldg(mq), m1 = __ldg(mq + 1);  // (kind, tex, param, needs_uv), (albedo, -)
            HitRecord rec;
            finalize_hit(S, h.w, h.o, h.d, rec, __float_as_int(m0.w) != 0);
            float3 point = rec.point, normal = rec.normal;
            uint32_t pixel, sample;
            batch_path<LIST>(b, path, pixel, sample);
            RngKey key{seed, pixel, sample, bounce};
            PhiloxStream rng(key, STREAM_SCATTER);
            if (MAT == MAT_LAMBERTIAN) {
                scatter_lambertian(S, __float_as_int(m0.y), point, normal, rec.uv, rng, out);
            } else if (MAT == MAT_METAL) {
                scatter_metal(f3(m1), m0.z, h.d, point, normal, rng, out);
            } else if (MAT == MAT_DIELECTRIC) {
                scatter_dielectric(m0.z, h.d, point, normal, rng, out);
            } else {
                scatter_isotropic(S, __float_as_int(m0.y), point, rec.uv, rng, out);
            }
            if (out.scattered) {
                st_stream(&ps.atten[(size_t)bounce * ps.cap + path],
                          make_float4(out.attenuation.x, out.attenuation.y, out.attenuation.z, 0.0f));
                mine = 0;
                // ten factors of magnitude <= 1e3 can not overflow; anything else (NaN included) poisons the batch
                if (!(fabsf(out.attenuation.x) <= 1e3f && fabsf(out.attenuation.y) <= 1e3f && fabsf(out.attenuation.z) <= 1e3f)) *ps.poison = 1u;
            }
            // absorbed (metal below the surface): radiance stays 0 (render.rs:25)
        }
        uint32_t slot = seg_reserve<1>(s_fill, base, mine);
        if (mine == 0) {
            st_stream(&xo[slot], make_float4(out.origin.x, out.origin.y, out.origin.z, __uint_as_float(path)));
            st_stream(&xd[slot], make_float4(out.dir.x, out.dir.y, out.dir.z, 0.0f));
        }
    }
}
template <int MAT, bool LIST>
__global__ void __launch_bounds__(FW_BLOCK, FW_SHADE_MIN_BLOCKS) shade_scatter_kernel(DeviceScene S, PathState ps, Batch b, uint2 seed, uint32_t bounce) {
    __shared__ uint32_t s_fill[1];
    const uint32_t seg = blockIdx.x;
    const uint32_t total = counter_row(ps, bounce, MAT)[seg];
    if (total == 0) return;  // block-uniform
    uint32_t* row_out = counter_row(ps, bounce + 1, FW_Q_EXTEND);
    seg_open<1>(s_fill, ps, row_out, seg);
    scatter_segment<MAT, LIST>(S, ps, b, seed, bounce, seg, total, s_fill);
    seg_close<1>(s_fill, ps, row_out, seg);
}

// Ray statistics without a host round trip per batch: rays traced = every entry of every bounce's extend queue.
__global__ void __launch_bounds__(256) tally_kernel(PathState ps, unsigned long long* total_rays) {
    __shared__ unsigned long long s_part[256];
    unsigned long long r = 0;
    for (int bn = 0; bn <= FW_MAX_DEPTH; ++bn) {   // row b = rays traced at bounce b (row 0 = the primary rays)
        const uint32_t* row = counter_row(ps, bn, FW_Q_EXTEND);
        for (uint32_t i = threadIdx.x; i < ps.nseg; i += 256) r += row[i];
    }
    s_part[threadIdx.x] = r;
    __syncthreads();
    for (int w = 128; w > 0; w >>= 1) {
        if ((int)threadIdx.x < w) s_part[threadIdx.x] += s_part[threadIdx.x + w];
        __syncthreads();
    }
    if (threadIdx.x == 0) *total_rays += s_part[0];
}

// render.rs:177-182 `total_color += color(...)`: samples of a pixel are added in sample order, so the fp32
// sum is independent of queue order and identical for any batch split along the sample axis.
__global__ void __launch_bounds__(256) accumulate_kernel(float* __restrict__ sum, PathState ps, Batch b) {
    for (uint32_t pl = blockIdx.x * blockDim.x + threadIdx.x; pl < b.npix; pl += gridDim.x * blockDim.x) {
        size_t pix = (size_t)b.pix0 + pl;
        float r = sum[3 * pix], g = sum[3 * pix + 1], bl = sum[3 * pix + 2];
        for (uint32_t s = 0; s < b.ns; ++s) {
            float4 c = ld_stream(&ps.radiance[(size_t)s * b.npix + pl]);
            r += c.x; g += c.y; bl += c.z;
        }
        sum[3 * pix] = r; sum[3 * pix + 1] = g; sum[3 * pix + 2] = bl;
    }
}

// quantise (wavefront.cuh): render.rs:184-189 + util.rs:14-23
__global__ void __launch_bounds__(256) resolve_kernel(const float* __restrict__ sum, uint32_t npix, float samples,
                                                      float gamma, unsigned char* __restrict__ rgb) {
    float inv_gamma = 1.0f / gamma;
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < npix; i += gridDim.x * blockDim.x) {
        rgb[3 * i] = quantise(sum[3 * i] / samples, inv_gamma);
        rgb[3 * i + 1] = quantise(sum[3 * i + 1] / samples, inv_gamma);
        rgb[3 * i + 2] = quantise(sum[3 * i + 2] / samples, inv_gamma);
    }
}

// resolve_kernel over the sum of src.n per-device buffers, read in place through peer mappings (rank order).
__global__ void __launch_bounds__(256) peer_reduce_resolve_kernel(PeerSums src, float* __restrict__ total, uint32_t n_values,
                                                                   float samples, float gamma, unsigned char* __restrict__ rgb) {
    const float inv_gamma = 1.0f / gamma;
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n_values; i += gridDim.x * blockDim.x) {
        float s = src.p[0][i];
        for (int k = 1; k < src.n; ++k) s += __ldcs(&src.p[k][i]);   // peer memory: read once, streaming
        total[i] = s;
        if (rgb) rgb[i] = quantise(s / samples, inv_gamma);
    }
}

// ---- launchers -------------------------------------------------------------------------------------------
void launch_raygen(const CameraRec& cam, const Batch& b, uint2 seed, const PathState& ps, cudaStream_t st) {
    if (b.pixels) raygen_kernel<true><<<ps.nseg, FW_BLOCK, 0, st>>>(cam, b, seed, ps);   // a pixel list (adaptive rounds)
    else raygen_kernel<false><<<ps.nseg, FW_BLOCK, 0, st>>>(cam, b, seed, ps);
}
void launch_miss(const DeviceScene& S, const PathState& ps, uint32_t bounce, bool black_env, cudaStream_t st) {
    if (black_env) miss_kernel<true><<<ps.nseg, FW_BLOCK, 0, st>>>(S, ps, bounce);
    else miss_kernel<false><<<ps.nseg, FW_BLOCK, 0, st>>>(S, ps, bounce);
}
void launch_shade_emissive(const DeviceScene& S, const PathState& ps, uint32_t bounce, cudaStream_t st) {
    shade_emissive_kernel<<<ps.nseg, FW_BLOCK, 0, st>>>(S, ps, bounce);
}
template <bool LIST>
static void launch_shade_scatter_t(int mat, const DeviceScene& S, const PathState& ps, const Batch& b, uint2 seed, uint32_t bounce,
                                   cudaStream_t st) {
    const unsigned G = ps.nseg;
    switch (mat) {
        case MAT_LAMBERTIAN: shade_scatter_kernel<MAT_LAMBERTIAN, LIST><<<G, FW_BLOCK, 0, st>>>(S, ps, b, seed, bounce); break;
        case MAT_METAL: shade_scatter_kernel<MAT_METAL, LIST><<<G, FW_BLOCK, 0, st>>>(S, ps, b, seed, bounce); break;
        case MAT_DIELECTRIC: shade_scatter_kernel<MAT_DIELECTRIC, LIST><<<G, FW_BLOCK, 0, st>>>(S, ps, b, seed, bounce); break;
        case MAT_ISOTROPIC: shade_scatter_kernel<MAT_ISOTROPIC, LIST><<<G, FW_BLOCK, 0, st>>>(S, ps, b, seed, bounce); break;
        default: break;
    }
}
void launch_shade_scatter(int mat, const DeviceScene& S, const PathState& ps, const Batch& b, uint2 seed, uint32_t bounce,
                          cudaStream_t st) {
    if (b.pixels) launch_shade_scatter_t<true>(mat, S, ps, b, seed, bounce, st);
    else launch_shade_scatter_t<false>(mat, S, ps, b, seed, bounce, st);
}
void launch_accumulate(float* d_sum, const PathState& ps, const Batch& b, unsigned blocks, cudaStream_t st) {
    accumulate_kernel<<<blocks, 256, 0, st>>>(d_sum, ps, b);
}
void launch_tally(const PathState& ps, unsigned long long* d_rays, cudaStream_t st) {
    tally_kernel<<<1, 256, 0, st>>>(ps, d_rays);
}
void launch_resolve(const float* d_sum, uint32_t npix, float samples, float gamma, unsigned char* d_rgb, unsigned blocks,
                    cudaStream_t st) {
    resolve_kernel<<<blocks, 256, 0, st>>>(d_sum, npix, samples, gamma, d_rgb);
}
void launch_peer_reduce_resolve(const PeerSums& src, float* total, uint32_t n_values, float samples, float gamma, unsigned char* rgb,
                                unsigned blocks, cudaStream_t st) {
    peer_reduce_resolve_kernel<<<blocks, 256, 0, st>>>(src, total, n_values, samples, gamma, rgb);
}

}  // namespace fw
