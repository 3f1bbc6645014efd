// Host-callable launchers of the kernels in kernels_extend.cu / kernels_shade.cu / kernels_probe.cu.
// api.cu orchestrates the wavefront through these; each translation unit compiles on its own (parallel build).
#pragma once
#include <cuda_runtime.h>

#include <cstdint>

#include "fw_types.h"
#include "wavefront_types.h"

namespace fw {

// Which extend kernel serves a scene (decided once at commit from the flattened scene).
struct ExtendPlan {
    bool has_mesh = false;          // some object is (or wraps) a TriangleMesh
    bool has_top_mesh = false;      // some render object IS a TriangleMesh
    bool has_medium_mesh = false;   // some ConstantMedium wraps a TriangleMesh
    bool lin_prog_ok = false;       // the linear-scan program fits kernel-parameter space
    bool lin_generic = false;       // ... and contains LIN_GENERIC items
    int lin_rect_tests = 0;         // AARect::hit calls per ray in the program
    bool small_top = false;         // the top-level tree has so few leaves that pass 1 scans them in order instead of walking
    bool walk = false;              // BVH scenes: collect / test walk kernels (walk.cuh) instead of the lock-step ones
};

// Device buffers of the walk kernels (allocated with the path state).
struct WalkAuxHost {
    unsigned long long* tkey = nullptr;   // [queue capacity] per-ray keys (scenes with top-level meshes)
    void* entries = nullptr;              // uint4 [nseg_max * ent_cap] (ray slot, mesh rank, mesh root node, first triangle slot)
    uint32_t ent_cap = 0;                 // entries per segment
    int prim_bits = 0;
};

void launch_raygen(const CameraRec& cam, const Batch& b, uint2 seed, const PathState& ps, cudaStream_t st);
// raygen from the caller's rays (fw_trace_rays): entry e of the bounce-0 queue gets the ray of its path, as launch_raygen lays it out.
void launch_raygen_rays(const RaySource& rs, const Batch& b, const PathState& ps, cudaStream_t st);
// The lock-step and linear-scan extend kernels.  Returns the number of kernels launched (2 for the two-pass mesh extend).
int launch_extend(const ExtendPlan& plan, bool use_bvh, const LinProgram& prog, const DeviceScene& S, const PathState& ps,
                  const Batch& b, uint2 seed, uint32_t bounce, cudaStream_t st);
// The same query through the collect / test walk kernels (kernels_walk.cu), one of its three kernels per call:
// 0 = pass 1 with entries, 1 = mesh walk, 2 = classification.
void launch_extend_walk_part(int part, const ExtendPlan& plan, const DeviceScene& S, const PathState& ps, const Batch& b, uint2 seed,
                             uint32_t bounce, const WalkAuxHost& aux, cudaStream_t st);
void launch_extend_pass1_entries(bool small_top, bool nested, const DeviceScene& S, const PathState& ps, const Batch& b, uint2 seed, uint32_t bounce,
                                 const WalkAuxHost& aux, cudaStream_t st);
void launch_miss(const DeviceScene& S, const PathState& ps, uint32_t bounce, bool black_env, cudaStream_t st);
void launch_shade_emissive(const DeviceScene& S, const PathState& ps, uint32_t bounce, cudaStream_t st);
void launch_shade_scatter(int mat, const DeviceScene& S, const PathState& ps, const Batch& b, uint2 seed, uint32_t bounce,
                          cudaStream_t st);
void launch_accumulate(float* d_sum, const PathState& ps, const Batch& b, unsigned blocks, cudaStream_t st);
void launch_tally(const PathState& ps, unsigned long long* d_rays, cudaStream_t st);
void launch_resolve(const float* d_sum, uint32_t npix, float samples, float gamma, unsigned char* d_rgb, unsigned blocks,
                    cudaStream_t st);
// fw_render_multi's peer reduce: the per-device sum buffers of up to kMaxPeers devices, read in place through peer mappings.
constexpr int kMaxPeers = 16;
struct PeerSums {
    const float* p[kMaxPeers];
    int n;
};
// total = the sum of the n_values floats of src.p[0 .. n) in rank order; rgb (nullable) = its resolve, as launch_resolve does.
void launch_peer_reduce_resolve(const PeerSums& src, float* total, uint32_t n_values, float samples, float gamma, unsigned char* rgb,
                                unsigned blocks, cudaStream_t st);

// Per-pixel state of an adaptive or denoised render (kernels_adaptive.cu), in the render context next to d_sum.
struct AdaptiveState {
    double* m1 = nullptr;           // [npix] sum of the samples' luminance
    double* m2 = nullptr;           // [npix] sum of its squares
    uint32_t* count = nullptr;      // [npix] samples rendered
    float* err = nullptr;           // [npix] final relative error (written by the resolve)
    uint32_t* list[2] = {nullptr, nullptr};   // active pixel lists, ascending (ping-pong between rounds)
    uint8_t* keep = nullptr;        // [npix] by list position: the pixel goes on to the next round
    uint32_t* block_base = nullptr; // [adaptive_blocks(npix) + 1] compaction block counts -> bases; [nb] = survivors
};
uint32_t adaptive_blocks(uint32_t n);   // compaction blocks of a list of n entries
void launch_accumulate_adaptive(float* d_sum, const AdaptiveState& a, const PathState& ps, const Batch& b, unsigned blocks, cudaStream_t st);
void launch_adaptive_init(uint32_t* list, uint32_t n, unsigned blocks, cudaStream_t st);   // list = 0, 1, ..., n - 1
// Stop rule over list_in[0, n), survivors to list_out in the same order, their number to a.block_base[adaptive_blocks(n)].
// Returns the number of kernels launched.
int launch_converge_compact(const AdaptiveState& a, const uint32_t* list_in, uint32_t n, double threshold, double floor, uint32_t* list_out,
                            cudaStream_t st);
void launch_resolve_adaptive(const float* d_sum, const AdaptiveState& a, uint32_t npix, float gamma, double floor, unsigned char* d_rgb,
                             unsigned blocks, cudaStream_t st);

// First-hit feature buffers and the edge-aware filter (kernels_denoise.cu, DESIGN.md §12).
struct AovState {
    float4* nz = nullptr;     // [npix] sum, then mean, of (normal.xyz, depth)
    float4* alb = nullptr;    // [npix] sum, then mean, of (albedo.rgb, 0)
    int* obj = nullptr;       // [npix] first-hit object of the range's first sample, -1 on a miss
};
// Bounce-0 shade and miss queues -> (albedo, asfloat(object)) into atten row 0 and (normal, depth) into atten row 1, by path.
void launch_aov_collect(const DeviceScene& S, const PathState& ps, cudaStream_t st);
// Adds the batch's records into a.nz / a.alb in sample order; `first`: the batch starts at the range's first sample (object ids).
void launch_aov_accumulate(const AovState& a, const PathState& ps, const Batch& b, bool first, unsigned blocks, cudaStream_t st);
// Sums -> means (divided by `samples`); `planar` (nullable): albedo [3 npix], normal [3 npix], depth [npix], one after the other.
void launch_aov_finalize(const AovState& a, uint32_t npix, float samples, float* planar, unsigned blocks, cudaStream_t st);
struct DenoiseSigmas {
    float luminance, depth, albedo;
};
// Planar colour / variance / guides -> (colour, variance) and the two guide float4 streams.
void launch_denoise_pack(const float* color, const float* variance, const float* albedo, const float* normal, const float* depth,
                         uint32_t npix, float4* cv, float4* nz, float4* alb, unsigned blocks, cudaStream_t st);
// (sum / (float)n, variance of the mean luminance from the moments) per pixel into cv, and the variance to `variance` [npix].
void launch_denoise_input(const float* d_sum, const AdaptiveState& a, uint32_t npix, uint32_t n, float4* cv, float* variance,
                          unsigned blocks, cudaStream_t st);
// One a-trous iteration at step 2^iteration.
void launch_atrous(const float4* cv_in, const float4* nz, const float4* alb, uint32_t width, uint32_t height, uint32_t iteration,
                   const DenoiseSigmas& sg, float4* cv_out, cudaStream_t st);
void launch_denoise_unpack(const float4* cv, uint32_t npix, float* color, float* variance, unsigned blocks, cudaStream_t st);

// probes (tests/ parity gates)
void launch_primary_rays_probe(const CameraRec& cam, uint32_t width, uint32_t height, uint32_t sample, uint2 seed,
                               uint32_t pix_begin, uint32_t n, float* origins, float* dirs, unsigned blocks, cudaStream_t st);
// mode: 0 = object-loop linear scan, 1 = BVH, 2 = LinProgram (generic items), 3 = LinProgram (no generic items)
void launch_first_hit_probe(int mode, const LinProgram& prog, const DeviceScene& S, uint2 seed, uint32_t n, const float* origins,
                            const float* dirs, const uint32_t* pixel, const uint32_t* sample, const uint32_t* bounce,
                            const FirstHitOut& out, unsigned blocks, cudaStream_t st);
void launch_probe_fill(const PathState& ps, uint32_t n, const float* origins, const float* dirs, uint32_t bounce, cudaStream_t st);
void launch_probe_collect(const DeviceScene& S, const PathState& ps, uint32_t bounce, const FirstHitOut& out, cudaStream_t st);
void launch_scatter_step_probe(const DeviceScene& S, uint32_t n, const ScatterProbeIO& io, unsigned blocks, cudaStream_t st);
void launch_env_sample_probe(const DeviceScene& S, uint32_t n, const float* dirs, float* out, unsigned blocks, cudaStream_t st);
void launch_texture_sample_probe(const DeviceScene& S, int tex, uint32_t n, const float* uv, const float* point, float* out,
                                 unsigned blocks, cudaStream_t st);
void launch_shared_division_probe(uint64_t n_pairs, uint2 seed, unsigned long long* violations);
void launch_fp32_peak(float* out, int iters, int blocks, int threads);
void launch_l2_read(const float4* buf, size_t n_vec, int reps, float* out, int blocks, int threads);

}  // namespace fw
