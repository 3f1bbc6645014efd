// Collect / test traversal of TriangleMesh trees (see walk.cuh for the design): walk_mesh_kernel, classify_mesh_kernel.
// extend_pass1_kernel<.., ENTRIES> (kernels_extend.cu) feeds them: mesh queue records, per-ray keys and (ray, mesh) entries.
#include "launch.h"
#include "walk.cuh"

namespace fw {

// Winner of a ray from its final key (found / t / object / rank / primitive).
FW_DEV void winner_from_key(const DeviceScene& S, unsigned long long k, int prim_bits, Winner& w) {
    w.found = k != FW_KEY_NONE;
    w.t = 0.0f; w.obj = -1; w.rank = -1;
    w.h.t = 0.0f; w.h.prim = 0; w.h.b0 = w.h.b1 = w.h.b2 = 0.0f;
    if (w.found) {
        w.t = w.h.t = key_t(k);
        w.rank = key_rank(k, prim_bits);
        w.h.prim = key_prim(k, prim_bits);
        w.obj = __ldg(&S.leaf_meta[w.rank]).w;
    }
}

// ---- mesh level ------------------------------------------------------------------------------------------------
// One work item = one (ray, mesh) entry: the mesh's tree is walked in the mesh's object space (scene.rs:242-253),
// triangles are tested in the test phase (mesh.rs:140-219), and the entry's best (t, rank, slot) is merged into the
// ray's key in global memory.
__global__ void __launch_bounds__(FW_BLOCK, FW_WALK_MIN_BLOCKS) walk_mesh_kernel(DeviceScene S, PathState ps, uint32_t bounce,
                                                                                 WalkAux aux) {
    __shared__ uint32_t s_cursor;
    __shared__ WalkWarp s_w[FW_WALK_WARPS];
    const uint32_t seg = blockIdx.x;
    const uint32_t in_count = counter_row(ps, bounce, FW_Q_ENTRY)[seg];
    if (in_count == 0) return;   // block-uniform
    if (threadIdx.x == 0) s_cursor = 0;
    __syncthreads();
    WalkWarp& W = s_w[threadIdx.x >> 5];
    const unsigned lane = threadIdx.x & 31u, lt = (1u << lane) - 1u;
    const size_t seg_base = (size_t)seg * ps.seg_cap;
    const float4* __restrict__ qo = ps.hq[FW_Q_MESH].o + seg_base;   // the rays that enter a mesh (pass 1)
    const float4* __restrict__ qd = ps.hq[FW_Q_MESH].d + seg_base;
    const uint4* __restrict__ ents = aux.entries + (size_t)seg * aux.ent_cap;
    unsigned long long* __restrict__ tkey = aux.tkey + seg_base;
    const float tmin = 0.001f, tmax = 2e9f;
    const int pb = aux.prim_bits;

    bool has_ray = false, active = false;
    float3 o = f3(0.0f, 0.0f, 0.0f), inv = f3(1.0f, 1.0f, 1.0f);   // the entry's ray in mesh space, permuted to (kx, ky, kz)
    uint32_t near_pack = 0, far_pack = 0;                           // node row offsets for that permutation (walk_rows)
    int node = -1, sp = 0;
    uint32_t slot_in = 0;
    unsigned long long stk[FW_WALK_STACK];   // deferred interior children: (cull distance, node)
    int npairs = 0;
    bool input_left = true;

    for (;;) {
        unsigned act = __ballot_sync(0xffffffffu, active);
        const bool want_refill = (input_left && 32 - __popc(act) >= FW_WALK_REFILL_IDLE) || act == 0u;
        if (npairs >= FW_WALK_TEST_AT || (want_refill && npairs > 0)) {
            // ---- TEST: one pair per lane, the leaf's 1-2 triangles against the owning entry's ray (bvh.rs:119-133 over
            // Triangle items, mesh.rs:140-219)
            const int n = npairs < 32 ? npairs : 32;
            __syncwarp();
            if ((int)lane < n) {
                const uint32_t pr = W.pairs[npairs - n + lane];
                const unsigned src = pr & 63u;
                const int packed = (int)(pr >> 6);
                const int first = packed >> 1, count = (packed & 1) + 1;
                const float3 ro = f3(W.ox[src], W.oy[src], W.oz[src]);
                TriSetup su;
                su.kz = W.su_k[src]; su.sx = W.su_x[src]; su.sy = W.su_y[src]; su.sz = W.su_z[src];
                const int tri_first = (int)W.a0[src], rank = (int)W.a1[src];
                // vertices from the copy permuted for this ray's dominant axis; the origin was stored permuted at fetch
                FW_WALK_CHECK(su.kz >= 0 && su.kz < 3 && tri_first >= 0 && first >= 0 && tri_first + first + count <= S.n_tris,
                              "bad pair kz=%d tri_first=%d first=%d count=%d n_tris=%d pr=%08x\n", su.kz, tri_first, first, count, S.n_tris, pr);
                const float4* tv = S.tri_perm + ((size_t)su.kz * S.n_tris + tri_first) * 3;
                for (int k = 0; k < count; ++k) {
                    const int slot = first + k;
                    const float4* v = &tv[3 * slot];
                    const float4 q0 = __ldg(v), q1 = __ldg(v + 1), q2 = __ldg(v + 2);
                    float t, c0, c1, c2;
                    if (triangle_test_perm(f3(q0), f3(q1), f3(q2), ro, su, tmin, tmax, t, c0, c1, c2))
                        atomicMin(&W.key[src], pack_key(t, rank, slot, pb));
                }
            }
            npairs -= n;
            __syncwarp();
            continue;
        }
        if (want_refill) {
            if (has_ray && !active) {   // retire: merge this entry's best into the ray's key
                const unsigned long long k = W.key[lane];
                if (k != FW_KEY_NONE) atomicMin(&tkey[slot_in], k);
                has_ray = false;
            }
            if (input_left) {
                const unsigned want = __ballot_sync(0xffffffffu, !has_ray);
                uint32_t base = 0;
                if (lane == 0) base = atomicAdd(&s_cursor, (uint32_t)__popc(want));
                base = __shfl_sync(0xffffffffu, base, 0);
                if (!has_ray) {
                    const uint32_t e = base + __popc(want & lt);
                    if (e < in_count) {
                        const uint4 en = __ldg(&ents[e]);
                        slot_in = en.x;
                        const int rank = (int)en.y;
                        const float4 ro = __ldg(&qo[slot_in]), rd = __ldg(&qd[slot_in]);
                        const float4 posr = __ldg(&S.leaf_posr[rank]);
                        const int4 meta = __ldg(&S.leaf_meta[rank]);
                        float3 oo = f3(ro) - f3(posr), od = f3(rd);
                        if (meta.x & OBJ_ROTATED) {   // scene.rs:242-249
                            const float4* m = &S.obj_irot[3 * meta.w];
                            float4 r0 = __ldg(m), r1 = __ldg(m + 1), r2 = __ldg(m + 2);
                            od = mat_mul(r0, r1, r2, f3(rd));
                            oo = mat_mul(r0, r1, r2, oo);
                        }
                        const int2 m0 = make_int2((int)en.z, (int)en.w);   // the mesh's root node, its first triangle slot
                        const TriSetup su = tri_setup(od);
                        {   // walker and test phase both use the ray permuted to (kx, ky, kz) order (mesh.rs:146-153)
                            const int kx = su.kz == 2 ? 0 : su.kz + 1, ky = kx == 2 ? 0 : kx + 1;
                            o = f3(comp3(oo, kx), comp3(oo, ky), comp3(oo, su.kz));
                            const float3 dp = f3(comp3(od, kx), comp3(od, ky), comp3(od, su.kz));
                            inv = f3(1.0f / dp.x, 1.0f / dp.y, 1.0f / dp.z);
                            walk_rows(su.kz, inv, near_pack, far_pack);
                            W.ox[lane] = o.x; W.oy[lane] = o.y; W.oz[lane] = o.z;
                        }
                        W.su_k[lane] = su.kz; W.su_x[lane] = su.sx; W.su_y[lane] = su.sy; W.su_z[lane] = su.sz;
                        W.a0[lane] = (uint32_t)m0.y;   // first triangle slot
                        W.a1[lane] = (uint32_t)rank;
                        // the ray's best so far (top-level winner, or an earlier entry's triangle): only a culling bound here
                        W.key[lane] = *reinterpret_cast<volatile unsigned long long*>(&tkey[slot_in]);
                        has_ray = true;
                        active = true;
                        sp = 0;
                        FW_WALK_CHECK(m0.x >= 0 && m0.x < S.n_nodes && (meta.x & OBJ_KIND_MASK) == SH_MESH, "bad mesh root %d kind %d rank %d\n", m0.x, meta.x & OBJ_KIND_MASK, rank);
                        node = m0.x;   // the mesh's root (a wide node: checked at flatten); its box was tested at top level
                    }
                }
                if (base + (uint32_t)__popc(want) >= in_count) input_left = false;
            }
            act = __ballot_sync(0xffffffffu, active);
            if (act == 0u) {
                if (!input_left && __ballot_sync(0xffffffffu, has_ray) == 0u) break;
                continue;
            }
        }
        bool l0 = false, l1 = false, l2 = false, l3 = false;
        int4 cc = make_int4(0, 0, 0, 0);
        if (active) {
            const float bnd = key_bound(W.key[lane]);
            if (node < 0) {
                for (;;) {
                    if (sp == 0) { active = false; break; }
                    const unsigned long long e = stk[--sp];
                    if (!(__uint_as_float((uint32_t)(e >> 32)) > bnd)) { node = (int)(uint32_t)e; break; }
                }
            }
            FW_WALK_CHECK(!active || (node >= 0 && node < S.n_nodes), "bad node %d sp %d\n", node, sp);
            if (active) walk_visit(S.nodes, node, o, inv, near_pack, far_pack, bnd, stk, sp, l0, l1, l2, l3, cc);
        }
        npairs = (int)walk_emit(W, (uint32_t)npairs, lane, l0, l1, l2, l3, cc);
    }
}

// ---- classification of the rays that entered a mesh ------------------------------------------------------------------
// Final key (pass-1 winner merged with every mesh entry's best triangle) -> winner -> its material's shade queue or the
// miss queue; continues the material queues pass 1 started.
__global__ void __launch_bounds__(FW_BLOCK) classify_mesh_kernel(DeviceScene S, PathState ps, uint32_t bounce, WalkAux aux) {
    __shared__ uint32_t s_fill[FW_NUM_QUEUES];
    const uint32_t seg = blockIdx.x;
    const uint32_t in_count = counter_row(ps, bounce, FW_Q_MESH)[seg];
    if (in_count == 0) return;
    seg_open<MAT_NUM_QUEUES>(s_fill, ps, counter_row(ps, bounce, 0), seg);
    const size_t seg_base = (size_t)seg * ps.seg_cap;
    for (uint32_t e0 = 0; e0 < in_count; e0 += FW_BLOCK) {
        const uint32_t e = e0 + threadIdx.x;
        Winner w;
        w.found = false; w.t = 0.0f; w.obj = -1; w.rank = -1; w.h.t = 0.0f; w.h.prim = 0; w.h.b0 = w.h.b1 = w.h.b2 = 0.0f;
        int mine = -1, material = -1;
        float3 o = f3(0.0f, 0.0f, 0.0f), d = o;
        uint32_t path = 0;
        if (e < in_count) {
            const float4 ro = ld_stream(&ps.hq[FW_Q_MESH].o[seg_base + e]), rd = ld_stream(&ps.hq[FW_Q_MESH].d[seg_base + e]);
            o = f3(ro); d = f3(rd); path = __float_as_uint(ro.w);
            winner_from_key(S, aux.tkey[seg_base + e], aux.prim_bits, w);
            FW_WALK_CHECK(!w.found || (w.rank >= 0 && w.rank < S.n_objects && w.h.prim >= 0 && w.h.prim < (1 << 24)), "bad key %016llx rank %d prim %d\n",
                          aux.tkey[seg_base + e], w.rank, w.h.prim);
            mine = classify_winner(S, w, material);
        }
        enqueue_hit<MAT_NUM_QUEUES>(ps, s_fill, blockIdx.x * ps.seg_cap, mine, o, d, path, w, material);
    }
    seg_close<MAT_NUM_QUEUES>(s_fill, ps, counter_row(ps, bounce, 0), seg);
}

// ---- launcher ----------------------------------------------------------------------------------------------------
void launch_extend_walk_part(int part, const ExtendPlan& plan, const DeviceScene& S, const PathState& ps, const Batch& b, uint2 seed,
                             uint32_t bounce, const WalkAuxHost& ax, cudaStream_t st) {
    WalkAux aux;
    aux.tkey = ax.tkey; aux.entries = reinterpret_cast<uint4*>(ax.entries); aux.ent_cap = ax.ent_cap; aux.prim_bits = ax.prim_bits;
    const unsigned G = ps.nseg;
    if (part == 0) launch_extend_pass1_entries(plan.small_top, plan.has_medium_mesh, S, ps, b, seed, bounce, ax, st);
    else if (part == 1) walk_mesh_kernel<<<G, FW_BLOCK, 0, st>>>(S, ps, bounce, aux);
    else classify_mesh_kernel<<<G, FW_BLOCK, 0, st>>>(S, ps, bounce, aux);
}

}  // namespace fw
