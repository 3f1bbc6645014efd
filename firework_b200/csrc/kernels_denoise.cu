// Denoised renders (fw_render_aov, fw_denoise_host, fw_render_denoised; DESIGN.md §12): first-hit feature buffers and the
// spatial filter of SVGF (Schied et al. 2017), an edge-avoiding a-trous wavelet filter.
//
// The AOV pass is raygen + the scene's own bounce-0 extend.  aov_collect_kernel reads the bounce-0 shade and miss queues back
// like probe_collect_kernel and rebuilds each hit with finalize_hit; the record of path p goes to atten rows 0 and 1 (the pass
// runs no shade kernel, so the attenuation chain is free), and aov_accumulate_kernel adds a pixel's samples in sample order.
// The RNG is keyed by (pixel, sample, bounce), so a pixel's record for sample s describes the first vertex of fw_render's path
// for that sample: the same ray, the same ConstantMedium draw, the attenuation its shade kernel applies.
//
// The filter is plain fp32 SIMT in this --fmad=false unit with a fixed tap and operation order, so tests replay it in numpy;
// only expf differs from numpy's exp (<= 2 ulp).
#include "launch.h"
#include "wavefront.cuh"

namespace fw {

// ---- AOV pass ---------------------------------------------------------------------------------------------
template <int K>
FW_DEV void aov_collect_queue(const DeviceScene& S, const PathState& ps) {
    const uint32_t total = counter_row(ps, 0, K)[blockIdx.x];
    const uint32_t base = blockIdx.x * ps.seg_cap;
    for (uint32_t e = threadIdx.x; e < total; e += FW_BLOCK) {
        uint32_t path;
        float4 albedo = make_float4(1.0f, 1.0f, 1.0f, __int_as_float(-1)), nz = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
        if (K == MAT_MISS) {
            path = __float_as_uint(ps.hq[K].d[base + e].w);
        } else {
            const HitIn h = get_hit<K>(ps, base + e);
            path = h.path;
            HitRecord rec;
            finalize_hit(S, h.w, h.o, h.d, rec);
            // the bounce-0 attenuation of the shade kernels (shade.cuh scatter_*); emissive vertices end the path: 1
            float3 a = f3(1.0f, 1.0f, 1.0f);
            if (K == MAT_LAMBERTIAN || K == MAT_ISOTROPIC) {
                a = texture_sample(S, __ldg(&S.mats[h.material].tex), rec.uv, rec.point);
            } else if (K == MAT_METAL) {
                const float4* mq = reinterpret_cast<const float4*>(&S.mats[h.material]);
                a = f3(__ldg(mq + 1));
            }
            const float3 n = normalized3(rec.normal);
            albedo = make_float4(a.x, a.y, a.z, __int_as_float(rec.obj));
            nz = make_float4(n.x, n.y, n.z, rec.t * mag3(h.d));
        }
        ps.atten[path] = albedo;
        ps.atten[(size_t)ps.cap + path] = nz;
    }
}
__global__ void __launch_bounds__(FW_BLOCK) aov_collect_kernel(DeviceScene S, PathState ps) {
    aov_collect_queue<0>(S, ps); aov_collect_queue<1>(S, ps); aov_collect_queue<2>(S, ps);
    aov_collect_queue<3>(S, ps); aov_collect_queue<4>(S, ps); aov_collect_queue<5>(S, ps);
}

// Pixels [pix0, pix0 + npix) of the image: the batch's samples in sample order into the fp32 sums (accumulate_kernel's order).
__global__ void __launch_bounds__(256) aov_accumulate_kernel(AovState a, PathState ps, Batch b, bool first) {
    for (uint32_t pl = blockIdx.x * blockDim.x + threadIdx.x; pl < b.npix; pl += gridDim.x * blockDim.x) {
        const size_t pix = (size_t)b.pix0 + pl;
        float4 sa = a.alb[pix], sn = a.nz[pix];
        for (uint32_t s = 0; s < b.ns; ++s) {
            const size_t p = (size_t)s * b.npix + pl;
            const float4 ra = ps.atten[p], rn = ps.atten[(size_t)ps.cap + p];
            sa.x += ra.x; sa.y += ra.y; sa.z += ra.z;
            sn.x += rn.x; sn.y += rn.y; sn.z += rn.z; sn.w += rn.w;
            if (first && s == 0) a.obj[pix] = __float_as_int(ra.w);
        }
        a.alb[pix] = sa;
        a.nz[pix] = sn;
    }
}

__global__ void __launch_bounds__(256) aov_finalize_kernel(AovState a, uint32_t npix, float samples, float* __restrict__ planar) {
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < npix; i += gridDim.x * blockDim.x) {
        float4 sa = a.alb[i], sn = a.nz[i];
        sa = make_float4(sa.x / samples, sa.y / samples, sa.z / samples, 0.0f);
        sn = make_float4(sn.x / samples, sn.y / samples, sn.z / samples, sn.w / samples);
        a.alb[i] = sa;
        a.nz[i] = sn;
        if (planar) {
            float* albedo = planar;
            float* normal = planar + 3 * (size_t)npix;
            float* depth = planar + 6 * (size_t)npix;
            albedo[3 * (size_t)i] = sa.x; albedo[3 * (size_t)i + 1] = sa.y; albedo[3 * (size_t)i + 2] = sa.z;
            normal[3 * (size_t)i] = sn.x; normal[3 * (size_t)i + 1] = sn.y; normal[3 * (size_t)i + 2] = sn.z;
            depth[i] = sn.w;
        }
    }
}

// ---- filter inputs -------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) denoise_pack_kernel(const float* __restrict__ color, const float* __restrict__ variance,
                                                           const float* __restrict__ albedo, const float* __restrict__ normal,
                                                           const float* __restrict__ depth, uint32_t npix, float4* __restrict__ cv,
                                                           float4* __restrict__ nz, float4* __restrict__ alb) {
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < npix; i += gridDim.x * blockDim.x) {
        const size_t k = 3 * (size_t)i;
        cv[i] = make_float4(color[k], color[k + 1], color[k + 2], variance[i]);
        nz[i] = make_float4(normal[k], normal[k + 1], normal[k + 2], depth[i]);
        alb[i] = make_float4(albedo[k], albedo[k + 1], albedo[k + 2], 0.0f);
    }
}

// mean = sum / (float)n (the resolve's division); v = max(0, (B - A (A / n)) / (n - 1)) / n in fp64 from the luminance moments,
// the maximum propagating NaN.
__global__ void __launch_bounds__(256) denoise_input_kernel(const float* __restrict__ sum, AdaptiveState a, uint32_t npix, uint32_t n,
                                                            float4* __restrict__ cv, float* __restrict__ variance) {
    const float fn = (float)n;
    const double dn = (double)n;
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < npix; i += gridDim.x * blockDim.x) {
        const double A = a.m1[i], B = a.m2[i];
        double var = (B - A * (A / dn)) / (dn - 1.0);
        var = var < 0.0 ? 0.0 : var;
        const float v = (float)(var / dn);
        cv[i] = make_float4(sum[3 * (size_t)i] / fn, sum[3 * (size_t)i + 1] / fn, sum[3 * (size_t)i + 2] / fn, v);
        variance[i] = v;
    }
}

__global__ void __launch_bounds__(256) denoise_unpack_kernel(const float4* __restrict__ cv, uint32_t npix, float* __restrict__ color,
                                                             float* __restrict__ variance) {
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < npix; i += gridDim.x * blockDim.x) {
        const float4 c = cv[i];
        color[3 * (size_t)i] = c.x; color[3 * (size_t)i + 1] = c.y; color[3 * (size_t)i + 2] = c.z;
        if (variance) variance[i] = c.w;
    }
}

// ---- the a-trous iteration -------------------------------------------------------------------------------------
constexpr int FW_ATROUS_BX = 16, FW_ATROUS_BY = 16;

FW_DEV bool finite4(float4 c) { return isfinite(c.x) && isfinite(c.y) && isfinite(c.z) && isfinite(c.w); }
FW_DEV float luminance_f(float4 c) { return (0.2126f * c.x + 0.7152f * c.y) + 0.0722f * c.z; }

// Tap order (dy outer, dx inner), weights and sums as DESIGN.md §12 states them; taps outside the image are dropped.
__global__ void __launch_bounds__(FW_ATROUS_BX * FW_ATROUS_BY) atrous_kernel(const float4* __restrict__ cv_in, const float4* __restrict__ nz,
                                                                             const float4* __restrict__ alb, uint32_t width, uint32_t height,
                                                                             int step, DenoiseSigmas sg, float4* __restrict__ cv_out) {
    const int x = blockIdx.x * FW_ATROUS_BX + threadIdx.x, y = blockIdx.y * FW_ATROUS_BY + threadIdx.y;
    if (x >= (int)width || y >= (int)height) return;
    const int W = (int)width, H = (int)height;
    const size_t i = (size_t)y * width + x;
    const float4 c = __ldg(&cv_in[i]);
    if (!finite4(c)) {   // a non-finite centre passes through unchanged
        cv_out[i] = c;
        return;
    }
    const float g1[3] = {0.25f, 0.5f, 0.25f};
    float gs = 0.0f, gw = 0.0f;
    for (int dy = -1; dy <= 1; ++dy)
        for (int dx = -1; dx <= 1; ++dx) {
            const int qx = x + dx, qy = y + dy;
            if (qx < 0 || qx >= W || qy < 0 || qy >= H) continue;
            const float4 q = __ldg(&cv_in[(size_t)qy * width + qx]);
            if (!finite4(q)) continue;
            const float w = g1[dx + 1] * g1[dy + 1];
            gs += w * q.w;
            gw += w;
        }
    const float den_l = sg.luminance * sqrtf(gs / gw) + 1e-6f;
    const float sa2 = sg.albedo * sg.albedo;
    const float lp = luminance_f(c);
    const float4 np = __ldg(&nz[i]), ap = __ldg(&alb[i]);
    const bool np_zero = np.x == 0.0f && np.y == 0.0f && np.z == 0.0f;
    const float k1[5] = {0.0625f, 0.25f, 0.375f, 0.25f, 0.0625f};
    float sw = 0.0f, sr = 0.0f, sgr = 0.0f, sb = 0.0f, sv = 0.0f;
    for (int dy = -2; dy <= 2; ++dy)
        for (int dx = -2; dx <= 2; ++dx) {
            const int qx = x + step * dx, qy = y + step * dy;
            if (qx < 0 || qx >= W || qy < 0 || qy >= H) continue;
            const size_t j = (size_t)qy * width + qx;
            const float4 q = __ldg(&cv_in[j]);
            if (!finite4(q)) continue;
            float w = 0.140625f;   // 9/64: the centre tap
            if (dx != 0 || dy != 0) {
                const float4 nq = __ldg(&nz[j]), aq = __ldg(&alb[j]);
                const float wl = expf(-fabsf(lp - luminance_f(q)) / den_l);
                float wn = 1.0f;
                if (!(np_zero && nq.x == 0.0f && nq.y == 0.0f && nq.z == 0.0f)) {
                    wn = fmaxf((np.x * nq.x + np.y * nq.y) + np.z * nq.z, 0.0f);
#pragma unroll
                    for (int k = 0; k < 7; ++k) wn = wn * wn;
                }
                const float wz = expf(-fabsf(np.w - nq.w) / (sg.depth * fmaxf(np.w, nq.w) + 1e-6f));
                const float ax = ap.x - aq.x, ay = ap.y - aq.y, az = ap.z - aq.z;
                const float wa = expf(-((ax * ax + ay * ay) + az * az) / sa2);
                w = k1[dx + 2] * k1[dy + 2];
                w = w * wl;
                w = w * wn;
                w = w * wz;
                w = w * wa;
            }
            sw += w;
            sr += w * q.x; sgr += w * q.y; sb += w * q.z;
            sv += (w * w) * q.w;
        }
    cv_out[i] = make_float4(sr / sw, sgr / sw, sb / sw, sv / (sw * sw));
}

// ---- launchers -------------------------------------------------------------------------------------------
void launch_aov_collect(const DeviceScene& S, const PathState& ps, cudaStream_t st) {
    aov_collect_kernel<<<ps.nseg, FW_BLOCK, 0, st>>>(S, ps);
}
void launch_aov_accumulate(const AovState& a, const PathState& ps, const Batch& b, bool first, unsigned blocks, cudaStream_t st) {
    aov_accumulate_kernel<<<blocks, 256, 0, st>>>(a, ps, b, first);
}
void launch_aov_finalize(const AovState& a, uint32_t npix, float samples, float* planar, unsigned blocks, cudaStream_t st) {
    aov_finalize_kernel<<<blocks, 256, 0, st>>>(a, npix, samples, planar);
}
void launch_denoise_pack(const float* color, const float* variance, const float* albedo, const float* normal, const float* depth,
                         uint32_t npix, float4* cv, float4* nz, float4* alb, unsigned blocks, cudaStream_t st) {
    denoise_pack_kernel<<<blocks, 256, 0, st>>>(color, variance, albedo, normal, depth, npix, cv, nz, alb);
}
void launch_denoise_input(const float* d_sum, const AdaptiveState& a, uint32_t npix, uint32_t n, float4* cv, float* variance,
                          unsigned blocks, cudaStream_t st) {
    denoise_input_kernel<<<blocks, 256, 0, st>>>(d_sum, a, npix, n, cv, variance);
}
void launch_atrous(const float4* cv_in, const float4* nz, const float4* alb, uint32_t width, uint32_t height, uint32_t iteration,
                   const DenoiseSigmas& sg, float4* cv_out, cudaStream_t st) {
    const dim3 block(FW_ATROUS_BX, FW_ATROUS_BY);
    const dim3 grid((width + FW_ATROUS_BX - 1) / FW_ATROUS_BX, (height + FW_ATROUS_BY - 1) / FW_ATROUS_BY);
    atrous_kernel<<<grid, block, 0, st>>>(cv_in, nz, alb, width, height, 1 << iteration, sg, cv_out);
}
void launch_denoise_unpack(const float4* cv, uint32_t npix, float* color, float* variance, unsigned blocks, cudaStream_t st) {
    denoise_unpack_kernel<<<blocks, 256, 0, st>>>(cv, npix, color, variance);
}

}  // namespace fw
