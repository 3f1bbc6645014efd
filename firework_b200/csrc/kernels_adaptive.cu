// Adaptive sampling (fw_render_adaptive, DESIGN.md §11): per-pixel moments, the stop rule, the stable compaction of the active
// pixel list and the per-pixel-count resolve.
//
// A round renders one sample range [n_r, n_{r+1}) for every pixel of the active list, through the ordinary wavefront with
// Batch::pixels pointing at the list.  Its accumulate adds the samples of a pixel in sample order into the same fp32 sum that
// accumulate_kernel would build, so a pixel that ends with k samples holds the sum of fw_render at samples = k, bit for bit.
// The stop rule runs in fp64 in a fixed operation order (the translation unit is --fmad=false; fp64 `/` and sqrt are IEEE),
// so a host replay in numpy decides identically.  The compaction is per-block counts -> one exclusive scan -> scatter: the
// survivors keep their ascending pixel order and no atomic decides any position.
#include "launch.h"
#include "wavefront.cuh"

namespace fw {

constexpr int FW_ADAPT_THREADS = 256;
constexpr uint32_t FW_ADAPT_CHUNK = 2048;   // list entries per compaction block

uint32_t adaptive_blocks(uint32_t n) { return n == 0 ? 1u : (n + FW_ADAPT_CHUNK - 1) / FW_ADAPT_CHUNK; }

// Y = (0.2126 r + 0.7152 g) + 0.0722 b of one fp32 sample, in fp64
FW_DEV double luminance(float4 c) { return (0.2126 * (double)c.x + 0.7152 * (double)c.y) + 0.0722 * (double)c.z; }

// Relative standard error of the mean after n samples with A = ΣY, B = ΣY².  Both maxima propagate NaN (numpy.maximum), so
// NaN radiance gives a NaN error, which never satisfies err <= threshold; n = 1 gives 0 / 0 = NaN as well.
FW_DEV double relative_error(double A, double B, uint32_t n, double floor) {
    const double dn = (double)n;
    const double mean = A / dn;
    double var = (B - A * mean) / (dn - 1.0);
    var = var < 0.0 ? 0.0 : var;
    const double am = fabs(mean);
    const double den = am < floor ? floor : am;
    return sqrt(var / dn) / den;
}

// accumulate_kernel for a round's batch over list entries [pix0, pix0 + npix) (LIST), or over pixels [pix0, pix0 + npix) of the
// image (the render stage of fw_render_denoised): the samples of a pixel in sample order into its fp32 sum, and their luminance
// into its fp64 moments.
template <bool LIST>
__global__ void __launch_bounds__(256) accumulate_adaptive_kernel(float* __restrict__ sum, AdaptiveState a, PathState ps, Batch b) {
    for (uint32_t pl = blockIdx.x * blockDim.x + threadIdx.x; pl < b.npix; pl += gridDim.x * blockDim.x) {
        const size_t pix = LIST ? (size_t)b.pixels[b.pix0 + pl] : (size_t)b.pix0 + pl;
        float r = sum[3 * pix], g = sum[3 * pix + 1], bl = sum[3 * pix + 2];
        double m1 = a.m1[pix], m2 = a.m2[pix];
        for (uint32_t s = 0; s < b.ns; ++s) {
            float4 c = ld_stream(&ps.radiance[(size_t)s * b.npix + pl]);
            r += c.x; g += c.y; bl += c.z;
            const double y = luminance(c);
            m1 += y;
            m2 += y * y;
        }
        sum[3 * pix] = r; sum[3 * pix + 1] = g; sum[3 * pix + 2] = bl;
        a.m1[pix] = m1; a.m2[pix] = m2;
        a.count[pix] += b.ns;
    }
}

__global__ void __launch_bounds__(256) adaptive_init_kernel(uint32_t* __restrict__ list, uint32_t n) {
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) list[i] = i;
}

// Pass 1: the stop rule for list entries [blockIdx.x * CHUNK, +CHUNK); keep[i] = 1 for a pixel that goes on, one count per block.
__global__ void __launch_bounds__(FW_ADAPT_THREADS) converge_count_kernel(AdaptiveState a, const uint32_t* __restrict__ list, uint32_t n,
                                                                          double threshold, double floor, uint32_t* __restrict__ block_count) {
    const uint32_t begin = blockIdx.x * FW_ADAPT_CHUNK, end = min(n, begin + FW_ADAPT_CHUNK);
    uint32_t kept = 0;
    for (uint32_t i = begin + threadIdx.x; i < end; i += FW_ADAPT_THREADS) {
        const uint32_t pix = list[i];
        const uint32_t cnt = a.count[pix];
        const bool stop = cnt >= 2 && relative_error(a.m1[pix], a.m2[pix], cnt, floor) <= threshold;
        a.keep[i] = stop ? 0 : 1;
        kept += stop ? 0u : 1u;
    }
    __shared__ uint32_t s_part[FW_ADAPT_THREADS / 32];
    for (int o = 16; o > 0; o >>= 1) kept += __shfl_xor_sync(0xffffffffu, kept, o);
    if ((threadIdx.x & 31u) == 0) s_part[threadIdx.x >> 5] = kept;
    __syncthreads();
    if (threadIdx.x == 0) {
        uint32_t t = 0;
        for (int w = 0; w < FW_ADAPT_THREADS / 32; ++w) t += s_part[w];
        block_count[blockIdx.x] = t;
    }
}

// Pass 2 (one block): exclusive scan of the block counts in place; base[nb] = the survivors in total.
__global__ void __launch_bounds__(1024) compact_scan_kernel(uint32_t* __restrict__ base, uint32_t nb) {
    __shared__ uint32_t s_tot[1024];
    const uint32_t per = (nb + 1023) / 1024;
    const uint32_t i0 = min(nb, threadIdx.x * per), i1 = min(nb, i0 + per);
    uint32_t t = 0;
    for (uint32_t i = i0; i < i1; ++i) t += base[i];
    s_tot[threadIdx.x] = t;
    __syncthreads();
    for (uint32_t o = 1; o < 1024; o <<= 1) {   // inclusive Hillis-Steele scan of the thread totals
        const uint32_t v = threadIdx.x >= o ? s_tot[threadIdx.x - o] : 0u;
        __syncthreads();
        s_tot[threadIdx.x] += v;
        __syncthreads();
    }
    uint32_t run = s_tot[threadIdx.x] - t;
    for (uint32_t i = i0; i < i1; ++i) {
        const uint32_t c = base[i];
        base[i] = run;
        run += c;
    }
    if (threadIdx.x == 1023) base[nb] = s_tot[1023];
}

// Pass 3: the kept entries of each block, in list order, from the block's base on.
__global__ void __launch_bounds__(FW_ADAPT_THREADS) compact_scatter_kernel(const uint8_t* __restrict__ keep, const uint32_t* __restrict__ list, uint32_t n,
                                                                           const uint32_t* __restrict__ base, uint32_t* __restrict__ out) {
    __shared__ uint32_t s_warp[FW_ADAPT_THREADS / 32];
    const uint32_t begin = blockIdx.x * FW_ADAPT_CHUNK, end = min(n, begin + FW_ADAPT_CHUNK);
    const unsigned lane = threadIdx.x & 31u, warp = threadIdx.x >> 5;
    uint32_t at = base[blockIdx.x];
    for (uint32_t i0 = begin; i0 < end; i0 += FW_ADAPT_THREADS) {   // block-uniform loop
        const uint32_t i = i0 + threadIdx.x;
        const bool k = i < end && keep[i] != 0;
        const unsigned m = __ballot_sync(0xffffffffu, k);
        if (lane == 0) s_warp[warp] = __popc(m);
        __syncthreads();
        uint32_t off = 0, tot = 0;
#pragma unroll
        for (int w = 0; w < FW_ADAPT_THREADS / 32; ++w) {
            const uint32_t c = s_warp[w];
            off += (unsigned)w < warp ? c : 0u;
            tot += c;
        }
        if (k) out[at + off + __popc(m & ((1u << lane) - 1u))] = list[i];
        at += tot;
        __syncthreads();
    }
}

// resolve_kernel with samples = the pixel's own count, and the pixel's final relative error
__global__ void __launch_bounds__(256) resolve_adaptive_kernel(const float* __restrict__ sum, AdaptiveState a, uint32_t npix, float gamma,
                                                               double floor, unsigned char* __restrict__ rgb) {
    float inv_gamma = 1.0f / gamma;
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < npix; i += gridDim.x * blockDim.x) {
        const uint32_t cnt = a.count[i];
        const float samples = (float)cnt;
        rgb[3 * i] = quantise(sum[3 * i] / samples, inv_gamma);
        rgb[3 * i + 1] = quantise(sum[3 * i + 1] / samples, inv_gamma);
        rgb[3 * i + 2] = quantise(sum[3 * i + 2] / samples, inv_gamma);
        a.err[i] = (float)relative_error(a.m1[i], a.m2[i], cnt, floor);
    }
}

// ---- launchers -------------------------------------------------------------------------------------------
void launch_accumulate_adaptive(float* d_sum, const AdaptiveState& a, const PathState& ps, const Batch& b, unsigned blocks, cudaStream_t st) {
    if (b.pixels) accumulate_adaptive_kernel<true><<<blocks, 256, 0, st>>>(d_sum, a, ps, b);
    else accumulate_adaptive_kernel<false><<<blocks, 256, 0, st>>>(d_sum, a, ps, b);
}
void launch_adaptive_init(uint32_t* list, uint32_t n, unsigned blocks, cudaStream_t st) {
    adaptive_init_kernel<<<blocks, 256, 0, st>>>(list, n);
}
int launch_converge_compact(const AdaptiveState& a, const uint32_t* list_in, uint32_t n, double threshold, double floor, uint32_t* list_out,
                            cudaStream_t st) {
    const uint32_t nb = adaptive_blocks(n);
    converge_count_kernel<<<nb, FW_ADAPT_THREADS, 0, st>>>(a, list_in, n, threshold, floor, a.block_base);
    compact_scan_kernel<<<1, 1024, 0, st>>>(a.block_base, nb);
    compact_scatter_kernel<<<nb, FW_ADAPT_THREADS, 0, st>>>(a.keep, list_in, n, a.block_base, list_out);
    return 3;
}
void launch_resolve_adaptive(const float* d_sum, const AdaptiveState& a, uint32_t npix, float gamma, double floor, unsigned char* d_rgb,
                             unsigned blocks, cudaStream_t st) {
    resolve_adaptive_kernel<<<blocks, 256, 0, st>>>(d_sum, a, npix, gamma, floor, d_rgb);
}

}  // namespace fw
