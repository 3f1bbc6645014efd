// Extend kernels: closest hit for every queued ray (render.rs:19 -> bvh.rs:115-151 / scene.rs:137-149).
#include "launch.h"
#include "walk.cuh"

namespace fw {

// What the mesh walk needs of a ray that pass 1 put into mesh-queue slot `slot` of segment `seg` because it must enter a
// mesh (`pending` != 0): its pass-1 winner as a 64-bit key (walk.cuh pack_key), and one (slot in the segment, mesh rank,
// mesh root node, first triangle slot) entry per mesh root box it hit.
FW_DEV void put_mesh_entries(const DeviceScene& S, const WalkAux& aux, uint32_t* s_fill, uint32_t seg, uint32_t seg_base, uint32_t slot,
                             uint32_t pending, const Winner& w) {
    aux.tkey[slot] = w.found ? pack_key(w.t, w.rank, w.h.prim, aux.prim_bits) : FW_KEY_NONE;
    uint32_t m = pending;
    while (m) {
        const int ord = __ffs(m) - 1;
        m &= m - 1u;
        const uint32_t e = atomicAdd(&s_fill[FW_Q_ENTRY], 1u);
        FW_WALK_CHECK(e < aux.ent_cap && ord < FW_MAX_WALK_MESHES, "entry overflow e=%u cap=%u ord=%d\n", e, aux.ent_cap, ord);
        aux.entries[(size_t)seg * aux.ent_cap + e] = make_uint4(slot - seg_base, (uint32_t)S.mesh_rank[ord], (uint32_t)S.mesh_root[ord], (uint32_t)S.mesh_tri0[ord]);
    }
}

// Two-pass extend for BVH scenes with TriangleMesh objects (see UnifiedWalker PHASE).  Pass 1 settles every ray
// against the non-mesh objects and the mesh root boxes; rays that must enter a mesh are compacted into the mesh
// queue (with the pass-1 winner and its rank) and finished by pass 2, where every lane of a warp is doing real
// mesh traversal.
// ENTRIES: the mesh walk (kernels_walk.cu) finishes the bounce instead of pass 2: every ray that must enter a mesh also
// gets its key and entries (put_mesh_entries).
template <bool NESTED, bool ENTRIES, bool LIST>
__global__ void __launch_bounds__(FW_BLOCK, FW_EXTEND_MIN_BLOCKS) extend_pass1_kernel(DeviceScene S, PathState ps, Batch b, uint2 seed,
                                                                                uint32_t bounce, WalkAux aux) {
    __shared__ uint32_t s_fill[FW_NUM_QUEUES];
    const uint32_t seg = blockIdx.x;
    const uint32_t in_count = counter_row(ps, bounce, FW_Q_EXTEND)[seg];
    seg_open<FW_NUM_QUEUES>(s_fill, ps, counter_row(ps, bounce, 0), seg);
    const uint32_t seg_base = seg * ps.seg_cap;
    for (uint32_t e0 = 0; e0 < in_count; e0 += FW_BLOCK) {
        const bool valid = e0 + threadIdx.x < in_count;
        uint32_t path = 0, pending = 0u;
        float3 o = f3(1e30f, 1e30f, 1e30f), d = f3(1.0f, 1.0f, 1.0f);
        Winner w;
        w.found = false; w.t = 0.0f; w.obj = -1; w.rank = -1; w.h.t = 0.0f; w.h.prim = 0;
        w.h.b0 = w.h.b1 = w.h.b2 = 0.0f;
        int mine = -1, material = -1;
        if (valid) {
            const size_t slot_in = (size_t)seg_base + e0 + threadIdx.x;
            float4 ro = ld_stream(&ps.xo[bounce & 1][slot_in]), rd = ld_stream(&ps.xd[bounce & 1][slot_in]);
            o = f3(ro); d = f3(rd); path = __float_as_uint(ro.w);
            RngKey key{seed, 0u, 0u, bounce};
            batch_path<LIST>(b, path, key.pixel, key.sample);
            UnifiedWalker<false, NESTED, true, 1> wk;
            int stack_code[FW_STACK];
            float stack_te[FW_STACK];
            if (wk.init(S, o, d, stack_code, stack_te, nullptr)) {
                while (wk.step(S, key, nullptr)) {
                }
            }
            w = wk.w;
            pending = wk.pending;
            if (pending) mine = FW_Q_MESH;
            else mine = classify_winner(S, w, material);
        }
        const uint32_t slot = enqueue_hit<FW_Q_MESH + 1>(ps, s_fill, seg_base, mine, o, d, path, w, material);
        if (ENTRIES && pending) put_mesh_entries(S, aux, s_fill, seg, seg_base, slot, pending, w);
    }
    seg_close<FW_NUM_QUEUES>(s_fill, ps, counter_row(ps, bounce, 0), seg);
}
// The same pass for scenes whose top-level tree has only a handful of leaves (a floor, a light, a few meshes): no walk at
// all.  A leaf of the reference's tree is reached iff its own box test passes (every ancestor's box contains it and the
// slab arithmetic is monotonic in the box planes), so the leaves are scanned in DFS order — every lane of the warp at the
// same leaf — and hits are merged by the (t, rank) rule of bvh.rs:120-146, which in rank order is "later wins unless
// strictly farther".  No stack, no traversal divergence; always with ENTRIES (it only serves the mesh walk).
template <bool NESTED, bool LIST>
__global__ void __launch_bounds__(FW_BLOCK, FW_EXTEND_MIN_BLOCKS) extend_pass1_small_kernel(DeviceScene S, PathState ps, Batch b, uint2 seed,
                                                                                      uint32_t bounce, WalkAux aux) {
    __shared__ uint32_t s_fill[FW_NUM_QUEUES];
    const uint32_t seg = blockIdx.x;
    const uint32_t in_count = counter_row(ps, bounce, FW_Q_EXTEND)[seg];
    seg_open<FW_NUM_QUEUES>(s_fill, ps, counter_row(ps, bounce, 0), seg);
    const uint32_t seg_base = seg * ps.seg_cap;
    const float tmin = 0.001f, tmax = 2e9f;   // render.rs:19
    for (uint32_t e0 = 0; e0 < in_count; e0 += FW_BLOCK) {
        const bool valid = e0 + threadIdx.x < in_count;
        uint32_t path = 0, pending = 0u;
        float3 o = f3(1e30f, 1e30f, 1e30f), d = f3(1.0f, 1.0f, 1.0f);
        Winner w;
        w.found = false; w.t = 0.0f; w.obj = -1; w.rank = -1; w.h.t = 0.0f; w.h.prim = 0;
        w.h.b0 = w.h.b1 = w.h.b2 = 0.0f;
        int mine = -1, material = -1;
        if (valid) {
            const size_t slot_in = (size_t)seg_base + e0 + threadIdx.x;
            float4 ro = ld_stream(&ps.xo[bounce & 1][slot_in]), rd = ld_stream(&ps.xd[bounce & 1][slot_in]);
            o = f3(ro); d = f3(rd); path = __float_as_uint(ro.w);
            if (e0 + FW_BLOCK + threadIdx.x < in_count) {
                prefetch_l2(&ps.xo[bounce & 1][slot_in + FW_BLOCK]); prefetch_l2(&ps.xd[bounce & 1][slot_in + FW_BLOCK]);
            }
            if (nan_direction(d)) {
                nan_direction_winner(S.nan_bvh_obj, S.nan_bvh_prim, w);
            } else {
                RngKey key{seed, 0u, 0u, bounce};
                if (S.has_medium) batch_path<LIST>(b, path, key.pixel, key.sample);
                const float3 inv = f3(1.0f / d.x, 1.0f / d.y, 1.0f / d.z);
                float bnd = FW_FLT_MAX;
                for (int l = 0; l < S.n_top_leaves; ++l) {
                    const float4 lo = __ldg(&S.top_leaves[2 * l]), hi = __ldg(&S.top_leaves[2 * l + 1]);
                    float te;
                    if (!slab_test(lo, hi, o, inv, tmin, tmax, te)) continue;
                    const int first = as_int(lo.w), count = as_int(hi.w);
                    for (int k = 0; k < count; ++k) {
                        const int rank = first + k;
                        const float4 posr = __ldg(&S.leaf_posr[rank]);
                        const int4 meta = __ldg(&S.leaf_meta[rank]);
                        if ((meta.x & OBJ_KIND_MASK) == SH_MESH) {
                            if (mesh_root_box_hit(S, posr, meta, o, d, bnd)) pending |= 1u << ((meta.x >> OBJ_MESH_ORD_SHIFT) & (FW_MAX_WALK_MESHES - 1));
                            continue;
                        }
                        ObjHit h;
                        if (object_test_loaded<false, NESTED>(S, meta.w, posr, meta, o, d, tmin, tmax, bnd, key, h, nullptr)) {
                            if (!w.found || !(w.t < h.t)) {   // ranks ascend: the later item wins unless it is strictly farther
                                w.found = true; w.t = h.t; w.obj = meta.w; w.rank = rank; w.h = h;
                                bnd = top_bound(S, h.t);
                            }
                        }
                    }
                }
            }
            if (pending) mine = FW_Q_MESH;
            else mine = classify_winner(S, w, material);
        }
        const uint32_t slot = enqueue_hit<FW_Q_MESH + 1>(ps, s_fill, seg_base, mine, o, d, path, w, material);
        if (pending) put_mesh_entries(S, aux, s_fill, seg, seg_base, slot, pending, w);
    }
    seg_close<FW_NUM_QUEUES>(s_fill, ps, counter_row(ps, bounce, 0), seg);
}

template <bool NESTED, bool LIST>
__global__ void __launch_bounds__(FW_BLOCK, FW_EXTEND_MIN_BLOCKS) extend_pass2_kernel(DeviceScene S, PathState ps, Batch b, uint2 seed,
                                                                                uint32_t bounce) {
    __shared__ uint32_t s_fill[FW_NUM_QUEUES];
    const uint32_t in_count = counter_row(ps, bounce, FW_Q_MESH)[blockIdx.x];
    if (in_count == 0) return;  // block-uniform
    seg_open<MAT_NUM_QUEUES>(s_fill, ps, counter_row(ps, bounce, 0), blockIdx.x);   // continues pass 1's material queues
    for (uint32_t e0 = 0; e0 < in_count; e0 += FW_BLOCK) {
        const bool valid = e0 + threadIdx.x < in_count;
        int mine = -1, material = -1;
        HitIn h;
        h.path = 0; h.o = h.d = f3(0.0f, 0.0f, 0.0f);
        h.w.found = false; h.w.t = 0.0f; h.w.obj = -1; h.w.rank = -1; h.w.h.t = 0.0f; h.w.h.prim = 0;
        h.w.h.b0 = h.w.h.b1 = h.w.h.b2 = 0.0f;
        if (valid) {
            h = get_hit<FW_Q_MESH>(ps, blockIdx.x * ps.seg_cap + e0 + threadIdx.x);
            RngKey key{seed, 0u, 0u, bounce};
            batch_path<LIST>(b, h.path, key.pixel, key.sample);
            UnifiedWalker<false, NESTED, true, 2> wk;
            wk.w = h.w;   // the pass-1 winner (a non-mesh object) and its rank
            wk.w.h.b0 = wk.w.h.b1 = wk.w.h.b2 = 0.0f;
            int stack_code[FW_STACK];
            float stack_te[FW_STACK];
            if (wk.init(S, h.o, h.d, stack_code, stack_te, nullptr)) {
                while (wk.step(S, key, nullptr)) {
                }
            }
            h.w = wk.w;
            mine = classify_winner(S, h.w, material);
        }
        enqueue_hit<MAT_NUM_QUEUES>(ps, s_fill, blockIdx.x * ps.seg_cap, mine, h.o, h.d, h.path, h.w, material);
    }
    seg_close<MAT_NUM_QUEUES>(s_fill, ps, counter_row(ps, bounce, 0), blockIdx.x);
}

template <bool NESTED, bool MESHES, bool LIST>
__global__ void __launch_bounds__(FW_BLOCK, FW_EXTEND_MIN_BLOCKS) extend_bvh_simple_kernel(DeviceScene S, PathState ps, Batch b, uint2 seed,
                                                                                     uint32_t bounce) {
    FW_EXTEND_PROLOGUE(MAT_NUM_QUEUES)
        if (valid) {
            RngKey key{seed, 0u, 0u, bounce};
            batch_path<LIST>(b, path, key.pixel, key.sample);
            trace_unified<false, NESTED, MESHES>(S, o, d, key, w, nullptr);
        }
    FW_EXTEND_EPILOGUE(MAT_NUM_QUEUES)
}

// Linear-scan scenes (Renderer.use_bvh == false, scene.rs:137-149): every ray tests every object in scene
// order, so there is no traversal-length divergence to balance.
// NESTED: the scene contains a TriangleMesh (its own BVH is walked inside the object test).
// This object-loop form serves scenes whose LinProgram does not fit kernel-parameter space.
template <bool NESTED, bool LIST>
__global__ void __launch_bounds__(FW_BLOCK) extend_linear_kernel(DeviceScene S, PathState ps, Batch b, uint2 seed, uint32_t bounce) {
    FW_EXTEND_PROLOGUE(MAT_NUM_QUEUES)
        if (valid) {
            RngKey key{seed, 0u, 0u, bounce};
            batch_path<LIST>(b, path, key.pixel, key.sample);
            trace_linear_scan<false, NESTED>(S, o, d, key, w, nullptr);
        }
    FW_EXTEND_EPILOGUE(MAT_NUM_QUEUES)
}

// The same query driven by the scene's LinProgram in kernel-parameter space (intersect.cuh trace_linear_prog):
// no per-lane loads of scene records, uniform item dispatch.  Every lane of a warp runs the program (lanes past
// the end of the segment trace a dummy ray and drop the result) so that the PRETEST vote sees the whole warp.
template <bool GENERIC, bool NESTED, bool PRETEST, bool SHDIV, bool LIST>
__global__ void __launch_bounds__(FW_BLOCK) extend_linear_prog_kernel(const __grid_constant__ LinProgram P, DeviceScene S, PathState ps,
                                                                      Batch b, uint2 seed, uint32_t bounce) {
    FW_EXTEND_PROLOGUE(MAT_NUM_QUEUES)
        RngKey key{seed, 0u, 0u, bounce};
        if (GENERIC) batch_path<LIST>(b, path, key.pixel, key.sample);
        trace_linear_prog<false, GENERIC, NESTED, PRETEST, SHDIV>(P, S, o, d, key, w, nullptr);
    FW_EXTEND_EPILOGUE(MAT_NUM_QUEUES)
}

// ---- launchers -------------------------------------------------------------------------------------------
template <bool LIST>
static int launch_extend_t(const ExtendPlan& plan, bool use_bvh, const LinProgram& P, const DeviceScene& S, const PathState& ps,
                           const Batch& b, uint2 seed, uint32_t bounce, cudaStream_t st) {
    const unsigned G = ps.nseg;   // one block per segment
    if (use_bvh && plan.has_top_mesh) {   // scenes the mesh walk does not serve
        WalkAux none{};
        if (plan.has_medium_mesh) {
            extend_pass1_kernel<true, false, LIST><<<G, FW_BLOCK, 0, st>>>(S, ps, b, seed, bounce, none);
            extend_pass2_kernel<true, LIST><<<G, FW_BLOCK, 0, st>>>(S, ps, b, seed, bounce);
        } else {
            extend_pass1_kernel<false, false, LIST><<<G, FW_BLOCK, 0, st>>>(S, ps, b, seed, bounce, none);
            extend_pass2_kernel<false, LIST><<<G, FW_BLOCK, 0, st>>>(S, ps, b, seed, bounce);
        }
        return 2;
    }
    if (use_bvh) {   // no top-level mesh: a mesh, if any, sits inside a ConstantMedium
        if (plan.has_medium_mesh)
            extend_bvh_simple_kernel<true, true, LIST><<<G, FW_BLOCK, 0, st>>>(S, ps, b, seed, bounce);
        else
            extend_bvh_simple_kernel<false, false, LIST><<<G, FW_BLOCK, 0, st>>>(S, ps, b, seed, bounce);
    } else if (plan.lin_prog_ok) {
        if (plan.lin_generic) {
            if (plan.has_mesh)
                extend_linear_prog_kernel<true, true, false, false, LIST><<<G, FW_BLOCK, 0, st>>>(P, S, ps, b, seed, bounce);
            else
                extend_linear_prog_kernel<true, false, false, false, LIST><<<G, FW_BLOCK, 0, st>>>(P, S, ps, b, seed, bounce);
        } else if (plan.lin_rect_tests >= 8) {   // rectangle-heavy: shared-reciprocal division (SHDIV)
            // coherent primary rays: whole warps skip Rect3d boxes they do not enter (PRETEST)
            if (bounce == 0) extend_linear_prog_kernel<false, false, true, true, LIST><<<G, FW_BLOCK, 0, st>>>(P, S, ps, b, seed, bounce);
            else extend_linear_prog_kernel<false, false, false, true, LIST><<<G, FW_BLOCK, 0, st>>>(P, S, ps, b, seed, bounce);
        } else {
            extend_linear_prog_kernel<false, false, false, false, LIST><<<G, FW_BLOCK, 0, st>>>(P, S, ps, b, seed, bounce);
        }
    } else if (plan.has_mesh) {
        extend_linear_kernel<true, LIST><<<G, FW_BLOCK, 0, st>>>(S, ps, b, seed, bounce);
    } else {
        extend_linear_kernel<false, LIST><<<G, FW_BLOCK, 0, st>>>(S, ps, b, seed, bounce);
    }
    return 1;
}
template <bool LIST>
static void launch_extend_pass1_entries_t(bool small_top, bool nested, const DeviceScene& S, const PathState& ps, const Batch& b, uint2 seed,
                                          uint32_t bounce, const WalkAuxHost& ax, cudaStream_t st) {
    WalkAux aux;
    aux.tkey = ax.tkey; aux.entries = reinterpret_cast<uint4*>(ax.entries); aux.ent_cap = ax.ent_cap; aux.prim_bits = ax.prim_bits;
    if (small_top) {
        if (nested) extend_pass1_small_kernel<true, LIST><<<ps.nseg, FW_BLOCK, 0, st>>>(S, ps, b, seed, bounce, aux);
        else extend_pass1_small_kernel<false, LIST><<<ps.nseg, FW_BLOCK, 0, st>>>(S, ps, b, seed, bounce, aux);
        return;
    }
    if (nested) extend_pass1_kernel<true, true, LIST><<<ps.nseg, FW_BLOCK, 0, st>>>(S, ps, b, seed, bounce, aux);
    else extend_pass1_kernel<false, true, LIST><<<ps.nseg, FW_BLOCK, 0, st>>>(S, ps, b, seed, bounce, aux);
}

// Batches over a pixel list (b.pixels set: adaptive rounds) run the LIST instantiations.
int launch_extend(const ExtendPlan& plan, bool use_bvh, const LinProgram& P, const DeviceScene& S, const PathState& ps,
                  const Batch& b, uint2 seed, uint32_t bounce, cudaStream_t st) {
    return b.pixels ? launch_extend_t<true>(plan, use_bvh, P, S, ps, b, seed, bounce, st)
                    : launch_extend_t<false>(plan, use_bvh, P, S, ps, b, seed, bounce, st);
}
void launch_extend_pass1_entries(bool small_top, bool nested, const DeviceScene& S, const PathState& ps, const Batch& b, uint2 seed, uint32_t bounce,
                                 const WalkAuxHost& ax, cudaStream_t st) {
    if (b.pixels) launch_extend_pass1_entries_t<true>(small_top, nested, S, ps, b, seed, bounce, ax, st);
    else launch_extend_pass1_entries_t<false>(small_top, nested, S, ps, b, seed, bounce, ax, st);
}

}  // namespace fw
