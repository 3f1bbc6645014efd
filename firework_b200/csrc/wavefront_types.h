// Host-visible types of the wavefront state (shared by the launchers in api.cu and the kernel translation units).
#pragma once
#include <cstdint>
#include "fw_types.h"

namespace fw {

#ifndef FW_SHADE_MIN_BLOCKS
#define FW_SHADE_MIN_BLOCKS 8    // shade kernels wait on dependent loads: cap registers at 64 (10 blocks = 51 regs spills: measured slower)
#endif
#ifndef FW_EXTEND_MIN_BLOCKS
#define FW_EXTEND_MIN_BLOCKS 8   // __launch_bounds__ min blocks / SM of the BVH extend kernels (register cap knob)
#endif
constexpr int FW_MAX_DEPTH = 10;          // render.rs:21  `depth < 10`
constexpr int FW_NUM_QUEUES = 9;          // [0..5] material queues (MatKind), [6] next extend queue, [7] mesh queue (rays that enter
                                          // a TriangleMesh), [8] (ray, mesh) entries of the mesh walk (counter only)
constexpr int FW_Q_EXTEND = 6, FW_Q_MESH = 7, FW_Q_ENTRY = 8;
constexpr int FW_TILE = 128;              // paths per tile: bounce 0 deals tiles round-robin to the segments
#ifndef FW_BLOCK_THREADS
#define FW_BLOCK_THREADS 128
#endif
constexpr int FW_BLOCK = FW_BLOCK_THREADS;             // threads per block of every queue-driven kernel

struct HitQueue {      // one shade queue: records of the paths whose ray hit a surface of that material
    float4* o;         // [nseg][seg_cap] ray origin.xyz, asfloat(path)
    float4* d;         // ray direction.xyz (never normalised: ray.rs), winning t        (miss queue: d.xyz, asfloat(path))
    float4* w;         // asfloat(object), asfloat(primitive), asfloat(material), asfloat(rank)   (rank: two-pass extend only)
};
struct PathState {
    float4* xo[2];     // ping-pong extend queues: ray origin.xyz, asfloat(path)
    float4* xd[2];     //                          ray direction.xyz
    HitQueue hq[8];    // [0..5] per-material shade queues (MatKind; MAT_MISS uses .d only), [7] mesh queue
    float4* atten;     // [FW_MAX_DEPTH][cap] attenuation chain, by path (see fold_radiance)
    float4* radiance;  // [cap] finished path radiance, by path
    uint32_t* counters;                // [FW_MAX_DEPTH + 2][FW_NUM_QUEUES][nseg] fill counts
    uint32_t* poison;                  // [1] set by a shade kernel that wrote an attenuation which is not small and finite (per batch)
    uint32_t cap;
    uint32_t nseg, seg_cap;
};
struct Batch {
    uint32_t pix0, npix, s0, ns;
    uint32_t width, height;
    uint32_t npix_magic;   // ceil(2^32 / npix) (0xffffffff for npix == 1): p / npix without the emulated 32-bit division
    uint32_t width_magic;  // the same for `width` (pixel -> column / row in raygen)
    const uint32_t* pixels;   // null: pixel = pix0 + p % npix.  Else a pixel list (adaptive rounds): pixel = pixels[pix0 + p % npix]
};
// Caller-supplied rays of a trace call (fw_trace_rays, DESIGN.md §13), device pointers to fp32 x3 per ray.  The ray of list
// position i and sample s is entry i (shared layout) or entry (s - sample_begin) * n + i (per-sample layout).
struct RaySource {
    const float* origins;
    const float* dirs;
    uint32_t n;
    uint32_t sample_begin;
    bool per_sample;
};

struct FirstHitOut {
    int *obj, *prim, *material;
    float *t, *point, *normal, *uv;
    unsigned long long* counters;  // [2] node tests, prim tests
};
struct ScatterProbeIO {
    const int* material;
    const float *ray_o, *ray_d, *hit_t, *hit_point, *hit_normal, *hit_uv, *uniforms;
    uint32_t nu;
    float* emit;
    int* scattered;
    float *atten, *out_o, *out_d;
    int* consumed;
};

}  // namespace fw
