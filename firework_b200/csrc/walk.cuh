// Collect / test traversal for BVH scenes (Renderer.use_bvh == true): the closest-hit query of render.rs:19 ->
// bvh.rs:115-151 restructured so that every instruction of the hot loop is useful for (almost) every lane of a warp.
//
// The lock-step kernels (kernels_extend.cu) run "walk to a leaf, test its items, pop" per lane; lanes of a warp are in
// different phases, so box code ran with ~6-8 of 32 lanes on mesh walks and ~18 on sphere scenes (ncu, profiles/r01f).
// Here the three phases are separated:
//   WALK   one loop iteration = one wide-node visit for every lane that has a ray (pop, four slab tests with the
//          reference's arithmetic aabb.rs:30-50, push the surviving interior children).  Surviving LEAF children are not
//          tested; the lane appends (lane, leaf) pairs to a small per-warp buffer in shared memory.
//   TEST   whenever the buffer holds 32 pairs the whole warp tests them, one pair per lane: the ray is fetched from the
//          owning lane's slot in shared memory, the leaf's 1-2 items go through the ordinary shape routines
//          (objects/*.rs restated in intersect.cuh), and hits are merged into the owning ray's 64-bit key with
//          atomicMin — key = (t bits, ~rank, ~primitive), i.e. exactly "smallest t, ties to the later leaf"
//          (bvh.rs:128,141).  The walking lane reads its key for the culling bound, so culling is only delayed by a few
//          iterations, never wrong (a culled subtree can not hold the winner).
//   REFILL warps are persistent inside their segment: when enough lanes have run out of nodes the warp flushes its
//          pairs, retires the finished rays and fetches new ones from the segment's queue (shared cursor).  With no
//          item / enter / exit code left inside the walk loop, refilled lanes do not serialise against the others (the
//          reason refilling did not pay for the lock-step kernels, profiles/r01_extend_variants.md).
// TriangleMesh objects are a second instance of the same machine: the top-level test phase runs the mesh's root-box test
// (scene.rs:242-253 + bvh.rs:117) and emits (ray, mesh) ENTRIES; walk_mesh_kernel walks one mesh tree per entry in the
// mesh's object space, tests triangles (mesh.rs:140-219) in its test phase and merges into the same per-ray key in
// global memory; classify_kernel then sorts the rays into the shade queues.  The barycentrics of the winning triangle
// are recomputed by finalize_hit (same arithmetic, once per ray) instead of travelling through the queues.
#pragma once
#include <cstdio>

#include "wavefront.cuh"

namespace fw {

#ifndef FW_WALK_MIN_BLOCKS
#define FW_WALK_MIN_BLOCKS 6      // __launch_bounds__ min blocks / SM of the walk kernels (register cap knob)
#endif
#ifndef FW_WALK_REFILL_IDLE
#define FW_WALK_REFILL_IDLE 12    // refill a warp when at least this many of its lanes have no node left to visit
#endif
#ifndef FW_WALK_CHECKS
#define FW_WALK_CHECKS 0          // 1 = bounds checks with printf + trap in the walk kernels (debug builds)
#endif
#define FW_WALK_CHECK(cond, ...) do { if (FW_WALK_CHECKS && !(cond)) { printf(__VA_ARGS__); __trap(); } } while (0)
constexpr int FW_WALK_STACK = 64;      // deferred interior children per lane (3 per wide level; checked at flatten)
constexpr int FW_WALK_RING = 256;      // pair buffer (power of two): < 32 left over + at most 4 new per lane = 159 pending
constexpr int FW_WALK_SLOTS = 32;      // entry slots per warp: one per lane
constexpr int FW_WALK_WARPS = FW_BLOCK / 32;
constexpr unsigned long long FW_KEY_NONE = ~0ull;

// key = t bits << 32 | ~rank << prim_bits | ~prim: atomicMin keeps the smallest t, then the largest rank, then the
// largest primitive slot — the merge rule of bvh.rs:120-146 as a total order (t > 0 always: t_min = 0.001).
FW_DEV unsigned long long pack_key(float t, int rank, int prim, int prim_bits) {
    uint32_t lo = ((uint32_t)(~rank) << prim_bits) | ((uint32_t)(~prim) & ((1u << prim_bits) - 1u));
    return ((unsigned long long)__float_as_uint(t) << 32) | lo;
}
FW_DEV float key_t(unsigned long long k) { return __uint_as_float((uint32_t)(k >> 32)); }
FW_DEV int key_rank(unsigned long long k, int prim_bits) { return (int)((~(uint32_t)k) >> prim_bits); }
FW_DEV int key_prim(unsigned long long k, int prim_bits) { return (int)((~(uint32_t)k) & ((1u << prim_bits) - 1u)); }
FW_DEV float key_bound(unsigned long long k) { return k == FW_KEY_NONE ? FW_FLT_MAX : cull_bound(key_t(k)); }

// Per-warp scratch in shared memory: the entries the warp currently owns (read by whichever lane tests one of their
// pairs), their keys, and the pair ring.
struct WalkWarp {
    unsigned long long key[FW_WALK_SLOTS];
    float ox[FW_WALK_SLOTS], oy[FW_WALK_SLOTS], oz[FW_WALK_SLOTS];   // ray origin in mesh space, permuted to (kx, ky, kz)
    uint32_t a0[FW_WALK_SLOTS], a1[FW_WALK_SLOTS];                    // first triangle slot of the mesh, top-level rank
    float su_x[FW_WALK_SLOTS], su_y[FW_WALK_SLOTS], su_z[FW_WALK_SLOTS];
    int su_k[FW_WALK_SLOTS];                                          // TriSetup of the ray in the mesh's space (mesh.rs:146-163)
    uint32_t pairs[FW_WALK_RING];                                     // (~leaf code) << 6 | owning slot
};

struct WalkAux {
    unsigned long long* tkey;   // [nseg][seg_cap] per-ray key of the current bounce (mesh scenes)
    uint4* entries;             // [nseg][ent_cap] (ray's slot in the segment's mesh queue, top-level rank of the mesh, its root
                                // node, its first triangle slot): everything the walker's fetch needs besides the ray
    uint32_t ent_cap;           // entries per segment
    int prim_bits;
};

// ---- culling that can not change the winner ---------------------------------------------------------------------
// A child box is culled against the best hit so far by the entry parameter of its kz-axis slab alone,
// (near_z - o_z) * (1 / d_z), kz = the axis Triangle::hit permutes to z (mesh.rs:146-153).  Every accepted hit satisfies
// t >= min_i z_i up to a few ulp, z_i = (p_i.z - o.z) * (1 / d.z) being computed from a vertex inside the box with the same
// subtraction, the same reciprocal and monotonic rounding, so t >= that slab entry: a box skipped because the entry exceeds
// best_t + margin can not hold the winner.  The set of boxes skipped then depends on timing, the winner does not — results
// are the reference's exhaustive traversal (bvh.rs:134-146), bit for bit and run to run.
// The box-entry parameter of the full slab test (what the lock-step kernels cull by) is NOT safe here: a triangle seen
// nearly edge-on is accepted with barycentrics that are rounding noise, and its t = sum(b_i z_i) (mesh.rs:188-196) can then
// land anywhere inside the triangle's depth range along kz — below the entry parameter of its own leaf box.  Such a hit is
// lost if an unrelated hit culled the leaf first (measured: ~3e-8 of the rays on suzanne, and WHICH is lost depends on
// scheduling once warps fetch work dynamically; profiles/r02_variants.md §2).
// The slab test itself is axis-order independent (max / min of the same six products), so the walker keeps the ray
// permuted to (kx, ky, kz) and loads the node rows in that order; the kz product comes out of the test for free.
#ifndef FW_WALK_TEST_AT
#define FW_WALK_TEST_AT 32   // pairs gathered by a warp before it runs a test phase (fewer: bounds shrink sooner, test lanes idle)
#endif

// One deferred interior child on a lane's stack: (cull distance, node) in one 64-bit word — one local-memory access per
// push / pop instead of two.
FW_DEV unsigned long long stack_entry(float dist, int node) {
    return ((unsigned long long)__float_as_uint(dist) << 32) | (uint32_t)node;
}

// Row byte offsets inside a wide node for a ray whose axes are permuted to (kx, ky, kz): near / far plane rows of each
// permuted axis, one byte each (near plane = max row where the direction is negative, see wide_visit).
FW_DEV void walk_rows(int kz, float3 inv_perm, uint32_t& near_pack, uint32_t& far_pack) {
    const int kx = kz == 2 ? 0 : kz + 1, ky = kx == 2 ? 0 : kx + 1;
    const uint32_t s0 = inv_perm.x < 0.0f ? 48u : 0u, s1 = inv_perm.y < 0.0f ? 48u : 0u, s2 = inv_perm.z < 0.0f ? 48u : 0u;
    near_pack = (16u * kx + s0) | ((16u * ky + s1) << 8) | ((16u * kz + s2) << 16);
    far_pack = (16u * kx + 48u - s0) | ((16u * ky + 48u - s1) << 8) | ((16u * kz + 48u - s2) << 16);
}

// One wide-node visit for the walk loop; o / inv are the ray permuted to (kx, ky, kz).  Children that survive the slab test
// (aabb.rs:30-50 arithmetic) and the cull are split into leaves (returned in l0..l3 for the caller to emit) and interior
// nodes (nearest becomes `node`, the rest are pushed onto the lane's stack `stk` with their cull distance).
FW_DEV void walk_visit(const float4* __restrict__ nodes, int& node, float3 o, float3 inv, uint32_t near_pack, uint32_t far_pack,
                       float bound, unsigned long long* stk, int& sp, bool& l0, bool& l1, bool& l2, bool& l3, int4& cc) {
    const float tmin = 0.001f, tmax = 2e9f;   // render.rs:19
    const float4* n = &nodes[8 * node];
    const uintptr_t nb = reinterpret_cast<uintptr_t>(n);   // 128-byte aligned: row offsets are OR-ed in
    auto row = [nb](uint32_t byte_off) { return reinterpret_cast<const float4*>(nb | (uintptr_t)byte_off); };
    const float4 nx = __ldg(row(near_pack & 0xffu)), ny = __ldg(row((near_pack >> 8) & 0xffu)), nz = __ldg(row(near_pack >> 16));
    const float4 fx = __ldg(row(far_pack & 0xffu)), fy = __ldg(row((far_pack >> 8) & 0xffu)), fz = __ldg(row(far_pack >> 16));
    cc = __ldg(reinterpret_cast<const int4*>(n + 6));
    float e0, e1, e2, e3;   // box entry (all three slabs)
    float z0, z1, z2, z3;   // entry of the kz slab alone
    auto slab = [&](float cnx, float cny, float cnz, float cfx, float cfy, float cfz, float& te, float& tz) {
        tz = (cnz - o.z) * inv.z;
        float lo = fmaxf(fmaxf(fmaxf(tmin, (cnx - o.x) * inv.x), (cny - o.y) * inv.y), tz);
        float hi = fminf(fminf(fminf(tmax, (cfx - o.x) * inv.x), (cfy - o.y) * inv.y), (cfz - o.z) * inv.z);
        te = lo;
        return hi > lo;
    };
    bool h0 = slab(nx.x, ny.x, nz.x, fx.x, fy.x, fz.x, e0, z0);
    bool h1 = slab(nx.y, ny.y, nz.y, fx.y, fy.y, fz.y, e1, z1);
    bool h2 = slab(nx.z, ny.z, nz.z, fx.z, fy.z, fz.z, e2, z2);
    bool h3 = slab(nx.w, ny.w, nz.w, fx.w, fy.w, fz.w, e3, z3);
    // cull / order distance (a NaN product, 0 * inf, must not drop the child: fmaxf returns the other operand)
    float t0 = fmaxf(z0, -FW_FLT_MAX), t1 = fmaxf(z1, -FW_FLT_MAX), t2 = fmaxf(z2, -FW_FLT_MAX), t3 = fmaxf(z3, -FW_FLT_MAX);
    h0 = h0 && !(t0 > bound); h1 = h1 && !(t1 > bound); h2 = h2 && !(t2 > bound); h3 = h3 && !(t3 > bound);
    // leaf children; empty slots (code FW_CODE_EXIT, inverted box) are excluded explicitly: a direction with NaN / infinite
    // components (scatter off a near-zero interpolated normal) passes EVERY slab test, f32::max / min ignoring NaN
    const int none = FW_CODE_EXIT;
    l0 = h0 && cc.x < 0 && cc.x != none; l1 = h1 && cc.y < 0 && cc.y != none;
    l2 = h2 && cc.z < 0 && cc.z != none; l3 = h3 && cc.w < 0 && cc.w != none;
    const float miss = __int_as_float(0x7f800000);
    t0 = (h0 && cc.x >= 0) ? t0 : miss; t1 = (h1 && cc.y >= 0) ? t1 : miss;
    t2 = (h2 && cc.z >= 0) ? t2 : miss; t3 = (h3 && cc.w >= 0) ? t3 : miss;
    int c0 = cc.x, c1 = cc.y, c2 = cc.z, c3 = cc.w;
    // visit order by the true box entry (all three slabs: a better front-to-back proxy than the kz slab, teapot +1.8 %),
    // culling still by the kz slab alone: the order only decides how soon the bound shrinks, never which hit wins
    float k0 = t0 < miss ? e0 : miss, k1 = t1 < miss ? e1 : miss, k2 = t2 < miss ? e2 : miss, k3 = t3 < miss ? e3 : miss;
    auto cswap3 = [](float& ka, int& ca, float& da, float& kb, int& cb, float& db) {
        if (kb < ka) { float k = ka; ka = kb; kb = k; int c = ca; ca = cb; cb = c; float d = da; da = db; db = d; }
    };
    cswap3(k0, c0, t0, k1, c1, t1);
    cswap3(k2, c2, t2, k3, c3, t3);
    cswap3(k0, c0, t0, k2, c2, t2);
    FW_WALK_CHECK(sp + 3 <= FW_WALK_STACK, "walk stack overflow sp=%d node=%d\n", sp, node);
    if (k3 < miss) stk[sp++] = stack_entry(t3, c3);
    if (k2 < miss) stk[sp++] = stack_entry(t2, c2);
    if (k1 < miss) stk[sp++] = stack_entry(t1, c1);
    node = (k0 < miss) ? c0 : -1;
}

// Appends the leaf children a lane found (l0..l3 of cc) for its entry slot `slot` to the warp's pair ring; returns the new
// tail.  All 32 lanes must call (lanes without work pass false flags).
FW_DEV uint32_t walk_emit(WalkWarp& W, uint32_t tail, uint32_t slot, bool l0, bool l1, bool l2, bool l3, int4 cc) {
    const unsigned lane = threadIdx.x & 31u, lt = (1u << lane) - 1u;
    const int c = (int)l0 + (int)l1 + (int)l2 + (int)l3;
    const unsigned b0 = __ballot_sync(0xffffffffu, c & 1), b1 = __ballot_sync(0xffffffffu, c & 2), b2 = __ballot_sync(0xffffffffu, c & 4);
    if ((b0 | b1 | b2) == 0u) return tail;
    uint32_t off = tail + __popc(b0 & lt) + 2 * __popc(b1 & lt) + 4 * __popc(b2 & lt);
    const uint32_t m = FW_WALK_RING - 1;
    if (l0) W.pairs[off++ & m] = ((uint32_t)(~cc.x) << 6) | slot;
    if (l1) W.pairs[off++ & m] = ((uint32_t)(~cc.y) << 6) | slot;
    if (l2) W.pairs[off++ & m] = ((uint32_t)(~cc.z) << 6) | slot;
    if (l3) W.pairs[off++ & m] = ((uint32_t)(~cc.w) << 6) | slot;
    return tail + __popc(b0) + 2 * __popc(b1) + 4 * __popc(b2);
}

}  // namespace fw
