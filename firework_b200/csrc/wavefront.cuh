// Wavefront path tracer kernels: raygen -> [extend -> miss / shade_<material>]* -> accumulate -> resolve.
// Iterative form of render.rs:12-33 `color()` (depth cap 10) inside render.rs:163-196 `render_pixel`.
//
// Path p of a batch covers pixel  pix0 + p % npix  and sample  s0 + p / npix  (implicit mapping: no id arrays).
// The queues carry the path's working state with them (ray, winning hit) as SoA float4 streams in queue order,
// compacted with warp ballot / popc, so every kernel reads its input fully coalesced and without a dependent
// "queue entry -> path -> record" hop; only the attenuation chain and the final radiance are indexed by path.
// extend publishes just the winning (t, object, primitive, barycentrics); the shade kernel that consumes a path
// rebuilds point / normal / uv (finalize_hit) in registers.
#pragma once
#include "intersect.cuh"
#include "shade.cuh"
#include "wavefront_types.h"

namespace fw {

// Queues are SEGMENTED: each of the `nseg` segments owns a fixed region of `seg_cap` slots in every queue and is
// processed by exactly one thread block per kernel, which is also the only writer of that segment's regions in
// the kernel's output queues.  A segment's paths therefore stay in the segment for the whole batch (its
// population only shrinks, so `seg_cap` = its bounce-0 share always suffices), fill counts are plain
// shared-memory counters written back once per block, and no global atomic is issued anywhere.  (One global
// counter per queue was the top stall of both extend and shade: ~2.5 same-sector atomics per warp iteration.)
// Path-state streams are touched once per kernel: load / store them with the streaming (evict-first) policy so
// that they do not push the scene tables (nodes, objects, shapes, materials) out of L1.
#ifndef FW_STREAM_HINTS
#define FW_STREAM_HINTS 1
#endif
FW_DEV float4 ld_stream(const float4* p) { return FW_STREAM_HINTS ? __ldcs(p) : *p; }
#ifndef FW_PREFETCH
#define FW_PREFETCH 1
#endif
// The record a shade thread will need in its NEXT iteration is FW_BLOCK slots ahead: ask L2 for it now (no register
// cost).  Measured: +1-2 % on the latency-bound shade kernels, +0.3 ... +0.6 % on the extend kernels (FW_EXTEND_PREFETCH).
FW_DEV void prefetch_l2(const void* p) {
    if (FW_PREFETCH) asm volatile("prefetch.global.L2 [%0];" ::"l"(p));
}
FW_DEV void st_stream(float4* p, float4 v) { if (FW_STREAM_HINTS) __stcs(p, v); else *p = v; }
// Counter rows: material / mesh queues of bounce b live in row b; the extend queue CONSUMED at bounce b lives in
// row b (raygen fills row 0, the shade kernels of bounce b fill row b + 1).
FW_DEV uint32_t* counter_row(const PathState& ps, uint32_t row, int queue) {
    return ps.counters + ((size_t)row * FW_NUM_QUEUES + queue) * ps.nseg;
}
// pixel = pix0 + p % npix, sample = s0 + p / npix.  q = umulhi(p, ceil(2^32 / npix)) is floor(p / npix) or one more
// (one less for npix == 1); one correction step makes it exact for every 32-bit p.
// LIST (adaptive rounds): pix0 / npix index the pixel list b.pixels instead of the image.  A template parameter rather than
// a run-time branch on b.pixels: the branch costs the shade and two-pass extend kernels 4-12 bytes of extra spills.
template <bool LIST>
FW_DEV void batch_path(const Batch& b, uint32_t p, uint32_t& pixel, uint32_t& sample) {
    uint32_t q = __umulhi(p, b.npix_magic);
    int r = (int)(p - q * b.npix);
    if (r < 0) { q -= 1u; r += (int)b.npix; }
    else if (r >= (int)b.npix) { q += 1u; r -= (int)b.npix; }
    pixel = b.pix0 + (uint32_t)r;
    if (LIST) pixel = __ldg(&b.pixels[pixel]);
    sample = b.s0 + q;
}
// render.rs:184-189 + util.rs:14-23: mean, powf(1/gamma), clamp, *255.99 -> saturating u8 (NaN -> 0)
FW_DEV unsigned char quantise(float mean, float inv_gamma) {
    float x = powf(mean, inv_gamma);
    if (x < 0.0f) x = 0.0f;
    if (x > 1.0f) x = 1.0f;
    float y = x * 255.99f;
    if (!(y == y)) return 0;
    return (unsigned char)fminf(fmaxf(truncf(y), 0.0f), 255.0f);
}

// render.rs:173-180 + camera.rs:109-116 + util.rs:31-33
// x / n and x % n for any 32-bit x, n >= 1, magic = ceil(2^32 / n) (0xffffffff for n == 1): umulhi gives the quotient or one
// more (one less for n == 1); one correction step makes it exact — no emulated 32-bit division.
FW_DEV void div_magic(uint32_t x, uint32_t n, uint32_t magic, uint32_t& q, uint32_t& r) {
    q = __umulhi(x, magic);
    int rr = (int)(x - q * n);
    if (rr < 0) { q -= 1u; rr += (int)n; }
    else if (rr >= (int)n) { q += 1u; rr -= (int)n; }
    r = (uint32_t)rr;
}
FW_DEV void primary_ray_at(const CameraRec& cam, uint32_t width, uint32_t height, uint32_t px, uint32_t row, uint32_t pixel, uint32_t sample,
                           uint2 seed, float3& o, float3& d);
FW_DEV void primary_ray(const CameraRec& cam, uint32_t width, uint32_t height, uint32_t pixel, uint32_t sample,
                        uint2 seed, float3& o, float3& d) {
    primary_ray_at(cam, width, height, pixel % width, pixel / width, pixel, sample, seed, o, d);
}
FW_DEV void primary_ray_at(const CameraRec& cam, uint32_t width, uint32_t height, uint32_t px, uint32_t row, uint32_t pixel, uint32_t sample,
                           uint2 seed, float3& o, float3& d) {
    uint32_t py = height - row;  // Coord::from_index: y counts down from `height`
    RngKey key{seed, pixel, sample, 0u};
    PhiloxStream rng(key, STREAM_CAMERA);
    float u = ((float)px + rng.next()) / (float)width;
    float v = ((float)py + rng.next()) / (float)height;
    float3 rd = cam.lens_radius * random_in_unit_disk(rng);
    float3 cu = f3(cam.u[0], cam.u[1], cam.u[2]), cv = f3(cam.v[0], cam.v[1], cam.v[2]);
    float3 pos = f3(cam.position[0], cam.position[1], cam.position[2]);
    float3 ll = f3(cam.lower_left[0], cam.lower_left[1], cam.lower_left[2]);
    float3 hor = f3(cam.horizontal[0], cam.horizontal[1], cam.horizontal[2]);
    float3 ver = f3(cam.vertical[0], cam.vertical[1], cam.vertical[2]);
    float3 offset = cu * rd.x + cv * rd.y;
    o = pos + offset;
    d = ll + u * hor + v * ver - pos - offset;
}
// ---- segment plumbing ------------------------------------------------------------------------------------
// Every queue-driven kernel runs one block per segment (gridDim.x == nseg).  Fill counters of the block's segment
// live in shared memory while the block runs.  `open` continues from the counts already in global memory: earlier
// kernels of the same bounce append to the same regions (the shade kernels share the next extend queue, pass 2
// continues pass 1's material queues); rows nobody wrote yet hold the zeros of the per-batch memset.
template <int NQ>
FW_DEV void seg_open(uint32_t* s_fill, const PathState& ps, const uint32_t* counter_rows /* [NQ][nseg] */, uint32_t seg) {
    if (threadIdx.x < NQ) s_fill[threadIdx.x] = counter_rows[(size_t)threadIdx.x * ps.nseg + seg];
    __syncthreads();
}
template <int NQ>
FW_DEV void seg_close(const uint32_t* s_fill, const PathState& ps, uint32_t* counter_rows, uint32_t seg) {
    __syncthreads();
    if (threadIdx.x < NQ) counter_rows[(size_t)threadIdx.x * ps.nseg + seg] = s_fill[threadIdx.x];
}
// Reserve one slot in queue `mine` of the segment for every lane with 0 <= mine < NQ: one shared-memory atomic per
// warp per non-empty queue (warp ballot / popc compaction).  Returns the slot (global index); all 32 lanes must call.
#ifndef FW_RESERVE_MATCH
#define FW_RESERVE_MATCH 1   // 1 = group the lanes of a warp by queue with one match.any instead of one ballot round per queue
#endif
template <int NQ>
FW_DEV uint32_t seg_reserve(uint32_t* s_fill, uint32_t seg_base, int mine) {
    unsigned lane = threadIdx.x & 31u;
    unsigned lt = (1u << lane) - 1u;
    uint32_t slot = 0;
    if (FW_RESERVE_MATCH && NQ > 2) {
        const unsigned grp = __match_any_sync(0xffffffffu, mine);   // the lanes that go to the same queue (or to none: mine < 0)
        const int leader = __ffs(grp) - 1;
        uint32_t base = 0;
        if (mine >= 0 && (int)lane == leader) base = atomicAdd(&s_fill[mine], (uint32_t)__popc(grp));
        base = __shfl_sync(0xffffffffu, base, leader);
        if (mine >= 0) slot = seg_base + base + __popc(grp & lt);
        return slot;
    }
#pragma unroll
    for (int k = 0; k < NQ; ++k) {
        unsigned mask = __ballot_sync(0xffffffffu, mine == k);
        if (mask == 0u) continue;
        int leader = __ffs(mask) - 1;
        uint32_t base = 0;
        if ((int)lane == leader) base = atomicAdd(&s_fill[k], (uint32_t)__popc(mask));
        base = __shfl_sync(0xffffffffu, base, leader);
        if (mine == k) slot = seg_base + base + __popc(mask & lt);
    }
    return slot;
}

// extend: closest hit for every queued ray; the ray moves on, together with the winning (t, object, primitive,
// barycentrics), into its material's shade queue (or the miss queue).  The full hit record is rebuilt by the
// shade kernel that consumes it (finalize_hit), so it never travels through HBM.

// The shade queue a winner belongs to, and its material (which travels with the record so that the shade kernel can
// fetch its material in parallel with the object records).
FW_DEV int classify_winner(const DeviceScene& S, const Winner& w, int& material) {
    material = -1;
    if (!w.found) return MAT_MISS;
    int4 meta = __ldg(&S.obj_meta[w.obj]);
    material = meta.y;
    if ((meta.x & OBJ_KIND_MASK) == SH_RECT3D) material = winner_material(S, w.obj, w.h.prim);  // faces may carry their own material
    return __ldg(&S.mats[material].kind);
}
// Writes the hit record of one ray into slot `slot` of queue K (K is a compile-time constant at every call site, so
// the queue's pointers are plain kernel parameters).
template <int K>
FW_DEV void put_hit(const PathState& ps, uint32_t slot, float3 o, float3 d, uint32_t path, const Winner& w, int material) {
    if (K == MAT_MISS) {
        st_stream(&ps.hq[K].d[slot], make_float4(d.x, d.y, d.z, __uint_as_float(path)));
        return;
    }
    st_stream(&ps.hq[K].o[slot], make_float4(o.x, o.y, o.z, __uint_as_float(path)));
    st_stream(&ps.hq[K].d[slot], make_float4(d.x, d.y, d.z, w.t));
    st_stream(&ps.hq[K].w[slot], make_float4(__int_as_float(w.obj), __int_as_float(w.h.prim), __int_as_float(material), __int_as_float(w.rank)));
}
#ifndef FW_ENQUEUE_INDEXED
#define FW_ENQUEUE_INDEXED 1   // 1 = pick the queue's stream pointers with a (constant-bank) indexed load: one store sequence for the warp
#endif
template <int NQ>
FW_DEV uint32_t enqueue_hit(const PathState& ps, uint32_t* s_fill, uint32_t seg_base, int mine, float3 o, float3 d, uint32_t path,
                            const Winner& w, int material) {
    uint32_t slot = seg_reserve<NQ>(s_fill, seg_base, mine);
    if (FW_ENQUEUE_INDEXED) {
        if (mine >= 0) {
            const HitQueue q = ps.hq[mine];   // kernel-parameter space, indexed per lane
            if (mine == MAT_MISS) {
                st_stream(&q.d[slot], make_float4(d.x, d.y, d.z, __uint_as_float(path)));
            } else {
                st_stream(&q.o[slot], make_float4(o.x, o.y, o.z, __uint_as_float(path)));
                st_stream(&q.d[slot], make_float4(d.x, d.y, d.z, w.t));
                st_stream(&q.w[slot], make_float4(__int_as_float(w.obj), __int_as_float(w.h.prim), __int_as_float(material), __int_as_float(w.rank)));
            }
        }
        return slot;
    }
    switch (mine) {   // one arm per queue keeps the queue index a compile-time constant
        case 0: put_hit<0>(ps, slot, o, d, path, w, material); break;
        case 1: put_hit<1>(ps, slot, o, d, path, w, material); break;
        case 2: put_hit<2>(ps, slot, o, d, path, w, material); break;
        case 3: put_hit<3>(ps, slot, o, d, path, w, material); break;
        case 4: put_hit<4>(ps, slot, o, d, path, w, material); break;
        case 5: put_hit<5>(ps, slot, o, d, path, w, material); break;
        case FW_Q_MESH: if (NQ > FW_Q_MESH) put_hit<FW_Q_MESH>(ps, slot, o, d, path, w, material); break;
        default: break;
    }
    return slot;   // global slot index (meaningful for lanes with 0 <= mine < NQ)
}
// A hit record read back by the kernel that consumes queue K.
struct HitIn {
    float3 o, d;
    uint32_t path;
    int material;
    Winner w;
};
template <int K>
FW_DEV HitIn get_hit(const PathState& ps, uint32_t slot) {
    float4 A = ld_stream(&ps.hq[K].o[slot]), B = ld_stream(&ps.hq[K].d[slot]), C = ld_stream(&ps.hq[K].w[slot]);
    HitIn h;
    h.o = f3(A); h.d = f3(B);
    h.path = __float_as_uint(A.w);
    h.material = __float_as_int(C.z);
    h.w.found = __float_as_int(C.x) >= 0;
    h.w.t = B.w; h.w.obj = __float_as_int(C.x); h.w.rank = __float_as_int(C.w);
    h.w.h.t = B.w; h.w.h.prim = __float_as_int(C.y);
    h.w.h.b0 = h.w.h.b1 = h.w.h.b2 = 0.0f;   // the winning triangle's barycentrics are recomputed by finalize_hit
    return h;
}

// Common shape of the extend kernels: one block per segment, FW_BLOCK rays per iteration.  The body sets `w`
// for valid lanes; the epilogue sorts the ray into its shade queue.
#ifndef FW_EXTEND_PREFETCH
#define FW_EXTEND_PREFETCH 1   // L2 prefetch of the next iteration's ray records: +0.3 ... +0.6 % (profiles/r02_variants.md)
#endif
#define FW_EXTEND_PROLOGUE(NQ_OUT)                                                                         \
    __shared__ uint32_t s_fill[FW_NUM_QUEUES];                                                               \
    const uint32_t in_count = counter_row(ps, bounce, FW_Q_EXTEND)[blockIdx.x];                              \
    seg_open<NQ_OUT>(s_fill, ps, counter_row(ps, bounce, 0), blockIdx.x);                                    \
    for (uint32_t e0 = 0; e0 < in_count; e0 += FW_BLOCK) {                                                   \
        const bool valid = e0 + threadIdx.x < in_count;                                                      \
        uint32_t path = 0;                                                                                   \
        float3 o = f3(1e30f, 1e30f, 1e30f), d = f3(1.0f, 1.0f, 1.0f);                                        \
        if (valid) {                                                                                         \
            const size_t slot_in = (size_t)blockIdx.x * ps.seg_cap + e0 + threadIdx.x;                       \
            float4 ro = ld_stream(&ps.xo[bounce & 1][slot_in]), rd = ld_stream(&ps.xd[bounce & 1][slot_in]);     \
            o = f3(ro); d = f3(rd); path = __float_as_uint(ro.w);                                            \
            if (FW_EXTEND_PREFETCH && e0 + FW_BLOCK + threadIdx.x < in_count) {                              \
                prefetch_l2(&ps.xo[bounce & 1][slot_in + FW_BLOCK]); prefetch_l2(&ps.xd[bounce & 1][slot_in + FW_BLOCK]); \
            }                                                                                                \
        }                                                                                                    \
        Winner w;                                                                                            \
        w.found = false; w.t = 0.0f; w.obj = -1; w.rank = -1; w.h.t = 0.0f; w.h.prim = 0;                    \
        w.h.b0 = w.h.b1 = w.h.b2 = 0.0f;                                                                     \
        int mine = -1, material = -1;
#define FW_EXTEND_EPILOGUE(NQ_OUT)                                                                         \
        if (valid && mine < 0) mine = classify_winner(S, w, material);                                       \
        enqueue_hit<NQ_OUT>(ps, s_fill, blockIdx.x * ps.seg_cap, mine, o, d, path, w, material);             \
    }                                                                                                        \
    seg_close<NQ_OUT>(s_fill, ps, counter_row(ps, bounce, 0), blockIdx.x);

}  // namespace fw
