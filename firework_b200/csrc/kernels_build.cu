// BVH build on the device: stage (a), the reference's median-split leaf order, and stage (b), the SAH splits over those
// leaves, with scene_host.cpp's semantics exactly (DESIGN.md §8).  The host keeps the O(n) bookkeeping: it reads the
// tree shape of stage (a) from n alone, makes every node and its box from the returned orders and splits with the code a
// host build uses, and collapses the result (stage (c)).  So every bit of the flattened tree comes from the same host
// arithmetic as a host build; the device decides orders and splits only.
//
// Both stages are sorts of segments (tree nodes) of one array.  A segmented stable sort here is a rank-by-counting sort
// of 1024-element tiles in shared memory followed by merge passes that double the sorted run length; a merge places an
// element of the left run after the right run's elements with a SMALLER key and one of the right run after the left
// run's elements with a key that is not larger, so equal keys (including -0.0 / +0.0, which compare equal as they do
// under the host's `<`) keep their input order.  No value is decided by an atomic; the NaN flag is a plain store of 1.
#include <cuda_runtime.h>

#include <algorithm>
#include <cmath>
#include <cstring>
#include <string>
#include <vector>

#include "../../include/firework_b200.h"
#include "scene_host.h"

namespace fw {
namespace {

constexpr int kTile = 1024;   // elements per tile sort / local subtree block (one per thread)

struct Seg {
    int lo, n;
};

// Index of the segment with the largest lo <= p (segments sorted by lo).
__device__ __forceinline__ int find_seg(const Seg* __restrict__ segs, int nseg, int p) {
    int a = 0, b = nseg - 1;
    while (a < b) {
        const int m = (a + b + 1) >> 1;
        if (segs[m].lo <= p) a = m;
        else b = m - 1;
    }
    return a;
}

// Positions outside every segment (single-leaf SAH nodes) are skipped: their vals are not maintained.
template <typename K>
__global__ void gather_keys_kernel(const K* __restrict__ key_of, const int* __restrict__ vals, K* __restrict__ keys, int n,
                                   const Seg* __restrict__ segs, int nseg, int* __restrict__ nan_flag) {
    const int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= n) return;
    const Seg s = segs[find_seg(segs, nseg, p)];
    if (p < s.lo || p >= s.lo + s.n) return;
    const K k = key_of[vals[p]];
    keys[p] = k;
    if (nan_flag && k != k) *nan_flag = 1;   // bvh.rs:34 would panic
}

// One block per tile (lo, len) of a segment: stable rank = keys below + equal keys earlier.
template <typename K>
__global__ void __launch_bounds__(kTile) tile_sort_kernel(const K* __restrict__ kin, const int* __restrict__ vin, K* __restrict__ kout,
                                                          int* __restrict__ vout, const int2* __restrict__ tiles) {
    __shared__ K sk[kTile];
    const int2 t = tiles[blockIdx.x];
    const int i = threadIdx.x;
    if (i < t.y) sk[i] = kin[t.x + i];
    __syncthreads();
    if (i >= t.y) return;
    const K k = sk[i];
    int r = 0;
    for (int j = 0; j < t.y; ++j) {
        const K kj = sk[j];
        r += (kj < k) || (kj == k && j < i);
    }
    kout[t.x + r] = k;
    vout[t.x + r] = vin[t.x + i];
}

// Merges pairs of sorted runs of width w (counted from each segment's start).  Positions outside every segment are skipped.
template <typename K>
__global__ void merge_kernel(const K* __restrict__ kin, const int* __restrict__ vin, K* __restrict__ kout, int* __restrict__ vout, int n,
                             const Seg* __restrict__ segs, int nseg, int w) {
    const int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= n) return;
    const Seg s = segs[find_seg(segs, nseg, p)];
    if (p < s.lo || p >= s.lo + s.n) return;
    const int i = p - s.lo, r = i / w, pr = r ^ 1, pb = pr * w;
    const K k = kin[p];
    int cnt = 0;
    if (pb < s.n) {
        const K* B = kin + s.lo + pb;
        int a = 0, b = min(pb + w, s.n) - pb;
        if (!(r & 1)) {   // left run: right-run keys strictly below
            while (a < b) { const int m = (a + b) >> 1; if (B[m] < k) a = m + 1; else b = m; }
        } else {          // right run: left-run keys not above
            while (a < b) { const int m = (a + b) >> 1; if (!(k < B[m])) a = m + 1; else b = m; }
        }
        cnt = a;
    }
    const int o = s.lo + min(r, pr) * w + (i - r * w) + cnt;
    kout[o] = k;
    vout[o] = vin[p];
}

// Stage (a) below the level where every node fits one block: one block per node finishes its subtree, level by level,
// in shared memory.  A node of 1 or 2 items is a leaf and is still sorted (and NaN-checked) at its own depth.
__global__ void __launch_bounds__(kTile) leaf_local_kernel(const float* __restrict__ cx, const float* __restrict__ cy,
                                                           const float* __restrict__ cz, int* __restrict__ order,
                                                           const Seg* __restrict__ segs, int depth0, int* __restrict__ nan_flag) {
    __shared__ int sid[kTile], sid2[kTile];
    __shared__ float sk[kTile];
    const Seg s = segs[blockIdx.x];
    const int i = threadIdx.x;
    sid[i] = i < s.n ? order[s.lo + i] : 0;
    sid2[i] = 0;   // only ever holds item ids, even if a NaN key breaks the ranks
    __syncthreads();
    for (int d = depth0;; ++d) {
        int lo = 0, m = s.n;
        bool active = i < s.n;
        for (int e = depth0; active && e < d; ++e) {
            if (m <= 2) { active = false; break; }
            const int h = m / 2;
            if (i < lo + h) m = h;
            else { lo += h; m -= h; }
        }
        const int axis = d % 3;
        const float* c = axis == 0 ? cx : axis == 1 ? cy : cz;
        float k = 0.0f;
        if (active) {
            k = c[sid[i]];
            sk[i] = k;
            if (k != k) *nan_flag = 1;
        }
        if (!__syncthreads_or(active)) break;
        if (active) {
            int r = lo;
            for (int j = lo; j < lo + m; ++j) {
                const float kj = sk[j];
                r += (kj < k) || (kj == k && j < i);
            }
            sid2[r] = sid[i];
        }
        __syncthreads();
        if (active) sid[i] = sid2[i];
        __syncthreads();
    }
    if (i < s.n) order[s.lo + i] = sid[i];
}

__global__ void centres_f32_kernel(const float* __restrict__ boxes, float* __restrict__ c, int n) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    for (int a = 0; a < 3; ++a) c[(size_t)a * n + i] = 0.5f * boxes[6 * (size_t)i + a] + 0.5f * boxes[6 * (size_t)i + 3 + a];   // aabb.rs:59-61
}

// ---- stage (b) ------------------------------------------------------------------------------------------------------

__global__ void centres_f64_kernel(const float* __restrict__ boxes, double* __restrict__ c, int n) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    for (int a = 0; a < 3; ++a) {
        const double v = 0.5 * ((double)boxes[6 * (size_t)i + a] + boxes[6 * (size_t)i + 3 + a]);
        c[(size_t)a * n + i] = v == v ? v : INFINITY;
    }
}

// Union of leaf boxes and their item count; cnt == 0 is the empty set (every leaf holds 1 or 2 items).  Min / max are
// exact, so any association gives the values the host's sequential sweep gives; the signs of zeros and NaN payloads may
// differ, and area() below cannot see either.
struct Agg {
    float lo[3], hi[3];
    int cnt;
};
__device__ __forceinline__ Agg comb(const Agg& a, const Agg& b) {
    if (!a.cnt) return b;
    if (!b.cnt) return a;
    Agg r;
    for (int q = 0; q < 3; ++q) { r.lo[q] = fminf(a.lo[q], b.lo[q]); r.hi[q] = fmaxf(a.hi[q], b.hi[q]); }
    r.cnt = a.cnt + b.cnt;
    return r;
}
__device__ __forceinline__ Agg shfl_up(const Agg& v, int off) {
    Agg r;
    for (int q = 0; q < 3; ++q) { r.lo[q] = __shfl_up_sync(~0u, v.lo[q], off); r.hi[q] = __shfl_up_sync(~0u, v.hi[q], off); }
    r.cnt = __shfl_up_sync(~0u, v.cnt, off);
    return r;
}
__device__ __forceinline__ Agg leaf_agg(const float* __restrict__ boxes, const int* __restrict__ counts, int leaf) {
    Agg r;
    for (int q = 0; q < 3; ++q) { r.lo[q] = boxes[6 * (size_t)leaf + q]; r.hi[q] = boxes[6 * (size_t)leaf + 3 + q]; }
    r.cnt = counts[leaf];
    return r;
}
__device__ __forceinline__ double area(const Agg& x) {   // scene_host.cpp half_area, std::max included
    double dx = (double)x.hi[0] - x.lo[0], dy = (double)x.hi[1] - x.lo[1], dz = (double)x.hi[2] - x.lo[2];
    dx = dx < 0.0 ? 0.0 : dx;
    dy = dy < 0.0 ? 0.0 : dy;
    dz = dz < 0.0 ? 0.0 : dz;
    return dx * dy + dy * dz + dz * dx;
}

// Inclusive scan over the block's threads (blockDim.x == kTile).
__device__ Agg block_scan(Agg v, Agg* warp_tot) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (int off = 1; off < 32; off <<= 1) {
        const Agg o = shfl_up(v, off);
        if (lane >= off) v = comb(o, v);
    }
    if (lane == 31) warp_tot[warp] = v;
    __syncthreads();
    if (warp == 0) {
        Agg t = warp_tot[lane];
        for (int off = 1; off < 32; off <<= 1) {
            const Agg o = shfl_up(t, off);
            if (lane >= off) t = comb(o, t);
        }
        warp_tot[lane] = t;
    }
    __syncthreads();
    if (warp > 0) v = comb(warp_tot[warp - 1], v);
    __syncthreads();
    return v;
}

struct SahTile {
    int seg, lo, len, first;   // segment index, first position, element count, index of the segment's first tile
};
struct SahSeg {
    int lo, n, depth, tile0, ntiles;
};
struct Best {
    double cost;
    int k;
};
__device__ __forceinline__ bool better(const Best& a, const Best& b) {   // a valid cost below b's, or equal at a smaller k
    return a.k >= 0 && (b.k < 0 || a.cost < b.cost || (a.cost == b.cost && a.k < b.k));
}

// Per tile and axis (blockIdx.y): union of its leaves in ord[axis] order.
__global__ void __launch_bounds__(kTile) sah_tile_reduce_kernel(const int* __restrict__ ord, const float* __restrict__ boxes,
                                                                const int* __restrict__ counts, const SahTile* __restrict__ tiles,
                                                                int ntiles, int nl, Agg* __restrict__ agg) {
    __shared__ Agg warp_tot[32];
    const SahTile t = tiles[blockIdx.x];
    const int a = blockIdx.y;
    Agg v;
    v.cnt = 0;
    if ((int)threadIdx.x < t.len) v = leaf_agg(boxes, counts, ord[(size_t)a * nl + t.lo + threadIdx.x]);
    v = block_scan(v, warp_tot);
    if (threadIdx.x == kTile - 1) agg[(size_t)a * ntiles + blockIdx.x] = v;
}

// Per segment and axis: exclusive prefix / suffix carries of its tiles, in tile order.
__global__ void sah_seg_scan_kernel(const SahSeg* __restrict__ segs, int nseg, int ntiles, const Agg* __restrict__ agg,
                                    Agg* __restrict__ pre, Agg* __restrict__ suf) {
    const int s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= nseg * 3) return;
    const int a = s / nseg;
    const SahSeg g = segs[s % nseg];
    const size_t base = (size_t)a * ntiles;
    Agg acc;
    acc.cnt = 0;
    for (int t = g.tile0; t < g.tile0 + g.ntiles; ++t) { pre[base + t] = acc; acc = comb(acc, agg[base + t]); }
    acc.cnt = 0;
    for (int t = g.tile0 + g.ntiles - 1; t >= g.tile0; --t) { suf[base + t] = acc; acc = comb(acc, agg[base + t]); }
}

// Per tile and axis: the SAH cost of every split k = i + 1 whose left side ends at this tile's element i, and the tile's
// best (lowest cost, then lowest k).
__global__ void __launch_bounds__(kTile) sah_tile_cost_kernel(const int* __restrict__ ord, const float* __restrict__ boxes,
                                                              const int* __restrict__ counts, const SahTile* __restrict__ tiles,
                                                              const SahSeg* __restrict__ segs, int ntiles, int nl,
                                                              const Agg* __restrict__ pre, const Agg* __restrict__ suf,
                                                              Best* __restrict__ best, int max_depth) {
    __shared__ Agg warp_tot[32];
    __shared__ Agg sfx[kTile + 1];
    __shared__ Best wbest[32];
    const SahTile t = tiles[blockIdx.x];
    const SahSeg g = segs[t.seg];
    const int a = blockIdx.y, i = threadIdx.x;
    const size_t ti = (size_t)a * ntiles + blockIdx.x;
    Agg v;
    v.cnt = 0;
    if (i < t.len) v = leaf_agg(boxes, counts, ord[(size_t)a * nl + t.lo + i]);
    const Agg p = comb(pre[ti], block_scan(v, warp_tot));          // leaves [0, pos] of the segment
    Agg r;                                                          // suffix from the tile's far end, built in reverse
    r.cnt = 0;
    const int j = kTile - 1 - i;
    if (j < t.len) r = leaf_agg(boxes, counts, ord[(size_t)a * nl + t.lo + j]);
    r = block_scan(r, warp_tot);
    sfx[j] = comb(r, suf[ti]);                                      // leaves [pos j, end) of the segment
    if (i == 0) sfx[kTile] = suf[ti];
    __syncthreads();
    const int total = comb(pre[ti], sfx[0]).cnt;
    int levels_needed = 0;
    while ((1 << levels_needed) < g.n) ++levels_needed;
    const bool balanced = g.depth + levels_needed >= max_depth;
    const int k = t.lo - g.lo + i + 1;
    Best b{INFINITY, -1};
    if (i < t.len && k < g.n && (!balanced || k == g.n / 2)) {
        const Agg right = i + 1 < t.len ? sfx[i + 1] : sfx[kTile];
        const double cost = area(p) * p.cnt + area(right) * (total - p.cnt);
        if (cost < INFINITY) b = Best{cost, k};
    }
    for (int off = 16; off > 0; off >>= 1) {
        const Best o{__shfl_down_sync(~0u, b.cost, off), __shfl_down_sync(~0u, b.k, off)};
        if (better(o, b)) b = o;
    }
    if ((i & 31) == 0) wbest[i >> 5] = b;
    __syncthreads();
    if (i < 32) {
        b = wbest[i];
        for (int off = 16; off > 0; off >>= 1) {
            const Best o{__shfl_down_sync(~0u, b.cost, off), __shfl_down_sync(~0u, b.k, off)};
            if (better(o, b)) b = o;
        }
        if (i == 0) best[ti] = b;
    }
}

// Per segment: the first strictly smaller cost in (axis, k) order; (2, n / 2) when none is finite.
__global__ void sah_pick_kernel(const SahSeg* __restrict__ segs, int nseg, int ntiles, const Best* __restrict__ best,
                                int2* __restrict__ split) {
    const int s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= nseg) return;
    const SahSeg g = segs[s];
    Best b{INFINITY, -1};
    int axis = -1;
    for (int a = 0; a < 3; ++a)
        for (int t = g.tile0; t < g.tile0 + g.ntiles; ++t) {
            const Best c = best[(size_t)a * ntiles + t];
            if (c.k >= 0 && c.cost < b.cost) { b = c; axis = a; }
        }
    split[s] = axis < 0 ? make_int2(2, g.n / 2) : make_int2(axis, b.k);
}

// The children take ord[best axis] as their order.
__global__ void sah_apply_kernel(const int* __restrict__ ord, int* __restrict__ leaves, int nl, const Seg* __restrict__ segs, int nseg,
                                 const int2* __restrict__ split) {
    const int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= nl) return;
    const int s = find_seg(segs, nseg, p);
    if (p < segs[s].lo || p >= segs[s].lo + segs[s].n) return;
    leaves[p] = ord[(size_t)split[s].x * nl + p];
}

// ---- host side --------------------------------------------------------------------------------------------------------

struct Err {
    std::string* msg;
    bool ok = true;
    bool operator()(cudaError_t e, const char* what) {
        if (e != cudaSuccess && ok) {
            ok = false;
            *msg = std::string("device BVH build: ") + what + ": " + cudaGetErrorString(e);
        }
        return ok;
    }
};
#define FWB(call) if (!chk((call), #call)) return false

// Scratch on one stream; stream-ordered allocations come back from the device's pool.
struct Session {
    int prev_device = -1;
    cudaStream_t stream = nullptr;
    std::vector<void*> bufs;
    ~Session() {
        if (stream) {
            for (void* p : bufs) cudaFreeAsync(p, stream);
            cudaStreamSynchronize(stream);
            cudaStreamDestroy(stream);
        }
        if (prev_device >= 0) cudaSetDevice(prev_device);
    }
    template <typename T>
    cudaError_t alloc(T** p, size_t count) {
        void* q = nullptr;
        cudaError_t e = cudaMallocAsync(&q, std::max<size_t>(count * sizeof(T), 16), stream);
        if (e == cudaSuccess) bufs.push_back(q);
        *p = (T*)q;
        return e;
    }
};

bool open_session(Session& S, int device, Err& chk) {
    int cur = 0;
    FWB(cudaGetDevice(&cur));
    S.prev_device = cur;
    FWB(cudaSetDevice(device));
    FWB(cudaStreamCreateWithFlags(&S.stream, cudaStreamNonBlocking));
    return true;
}

inline unsigned blocks(size_t n, unsigned b = 256) { return (unsigned)((n + b - 1) / b); }

// Stable sort of every segment of (keys, vals); the result ends in (keys, vals).  kt / vt are scratch of the same size.
template <typename K>
bool sort_segments(Session& S, Err& chk, K*& keys, int*& vals, K*& kt, int*& vt, int n, const std::vector<Seg>& segs, Seg* d_segs,
                   int2* d_tiles) {
    std::vector<int2> tiles;
    int max_n = 0;
    for (const Seg& s : segs) {
        max_n = std::max(max_n, s.n);
        for (int t = 0; t < s.n; t += kTile) tiles.push_back(make_int2(s.lo + t, std::min(kTile, s.n - t)));
    }
    FWB(cudaMemcpyAsync(d_segs, segs.data(), segs.size() * sizeof(Seg), cudaMemcpyHostToDevice, S.stream));
    FWB(cudaMemcpyAsync(d_tiles, tiles.data(), tiles.size() * sizeof(int2), cudaMemcpyHostToDevice, S.stream));
    tile_sort_kernel<K><<<(unsigned)tiles.size(), kTile, 0, S.stream>>>(keys, vals, kt, vt, d_tiles);
    std::swap(keys, kt);
    std::swap(vals, vt);
    for (int w = kTile; w < max_n; w *= 2) {
        merge_kernel<K><<<blocks(n), 256, 0, S.stream>>>(keys, vals, kt, vt, n, d_segs, (int)segs.size(), w);
        std::swap(keys, kt);
        std::swap(vals, vt);
    }
    FWB(cudaGetLastError());
    return true;
}

}  // namespace

bool bvh_leaf_order_device(int device, const std::vector<Box>& boxes, std::vector<int>& order, bool& nan, std::string& err) {
    Err chk{&err};
    Session S;
    if (!open_session(S, device, chk)) return false;
    const int n = (int)boxes.size();
    float *d_boxes, *d_c, *d_keys, *d_kt;
    int *d_order, *d_vt, *d_nan;
    Seg* d_segs;
    int2* d_tiles;
    // nodes per level: 2^depth while they exceed a tile (at most n / kTile of them); tiles: n / kTile + one per node
    const size_t max_segs = 2 * (size_t)n / kTile + 2;
    FWB(S.alloc(&d_boxes, 6 * (size_t)n));
    FWB(S.alloc(&d_c, 3 * (size_t)n));
    FWB(S.alloc(&d_keys, n));
    FWB(S.alloc(&d_kt, n));
    FWB(S.alloc(&d_order, n));
    FWB(S.alloc(&d_vt, n));
    FWB(S.alloc(&d_nan, 1));
    FWB(S.alloc(&d_segs, max_segs));
    FWB(S.alloc(&d_tiles, 2 * max_segs));
    order.resize(n);
    for (int i = 0; i < n; ++i) order[i] = i;
    FWB(cudaMemcpyAsync(d_boxes, boxes.data(), sizeof(Box) * (size_t)n, cudaMemcpyHostToDevice, S.stream));
    FWB(cudaMemcpyAsync(d_order, order.data(), sizeof(int) * (size_t)n, cudaMemcpyHostToDevice, S.stream));
    FWB(cudaMemsetAsync(d_vt, 0, sizeof(int) * (size_t)n, S.stream));   // only item ids, even if a NaN key breaks the merge
    FWB(cudaMemsetAsync(d_nan, 0, sizeof(int), S.stream));
    centres_f32_kernel<<<blocks(n), 256, 0, S.stream>>>(d_boxes, d_c, n);
    // Levels whose nodes exceed a tile: global sorts.  Node sizes of one level differ by at most one, so they are all
    // interior there.
    std::vector<Seg> segs{Seg{0, n}};
    int depth = 0;
    while (segs.back().n > kTile) {   // the last node of a level is one of its largest
        FWB(cudaMemcpyAsync(d_segs, segs.data(), segs.size() * sizeof(Seg), cudaMemcpyHostToDevice, S.stream));
        gather_keys_kernel<float><<<blocks(n), 256, 0, S.stream>>>(d_c + (size_t)(depth % 3) * n, d_order, d_keys, n, d_segs,
                                                                   (int)segs.size(), d_nan);
        if (!sort_segments<float>(S, chk, d_keys, d_order, d_kt, d_vt, n, segs, d_segs, d_tiles)) return false;
        std::vector<Seg> next;
        for (const Seg& s : segs) {
            next.push_back(Seg{s.lo, s.n / 2});
            next.push_back(Seg{s.lo + s.n / 2, s.n - s.n / 2});
        }
        segs.swap(next);
        ++depth;
    }
    FWB(cudaMemcpyAsync(d_segs, segs.data(), segs.size() * sizeof(Seg), cudaMemcpyHostToDevice, S.stream));
    leaf_local_kernel<<<(unsigned)segs.size(), kTile, 0, S.stream>>>(d_c, d_c + n, d_c + 2 * (size_t)n, d_order, d_segs, depth, d_nan);
    FWB(cudaGetLastError());
    int h_nan = 0;
    FWB(cudaMemcpyAsync(order.data(), d_order, sizeof(int) * (size_t)n, cudaMemcpyDeviceToHost, S.stream));
    FWB(cudaMemcpyAsync(&h_nan, d_nan, sizeof(int), cudaMemcpyDeviceToHost, S.stream));
    FWB(cudaStreamSynchronize(S.stream));
    nan = h_nan != 0;
    return true;
}

bool bvh_sah_device(int device, const std::vector<Box>& leaf_boxes, const std::vector<int>& leaf_counts, int max_depth,
                    std::vector<SahRec>& recs, std::vector<int>& leaf_order, std::string& err) {
    Err chk{&err};
    Session S;
    if (!open_session(S, device, chk)) return false;
    const int nl = (int)leaf_boxes.size();
    recs.clear();
    leaf_order.resize(nl);
    for (int i = 0; i < nl; ++i) leaf_order[i] = i;
    float* d_boxes;
    double *d_ctr, *d_keys, *d_kt;
    int *d_counts, *d_leaves, *d_ord, *d_vals, *d_vt;
    Seg* d_segs;
    int2 *d_tiles, *d_split;
    SahSeg* d_sseg;
    SahTile* d_stile;
    Agg *d_agg, *d_pre, *d_suf;
    Best* d_best;
    // a level holds at most nl / 2 nodes of 2 or more leaves and nl / 2 + nl / kTile tiles
    const size_t max_segs = (size_t)nl / 2 + 1, max_tiles = (size_t)nl / 2 + (size_t)nl / kTile + 2;
    FWB(S.alloc(&d_boxes, 6 * (size_t)nl));
    FWB(S.alloc(&d_counts, nl));
    FWB(S.alloc(&d_ctr, 3 * (size_t)nl));
    FWB(S.alloc(&d_keys, nl));
    FWB(S.alloc(&d_kt, nl));
    FWB(S.alloc(&d_leaves, nl));
    FWB(S.alloc(&d_ord, 3 * (size_t)nl));
    FWB(S.alloc(&d_vals, nl));
    FWB(S.alloc(&d_vt, nl));
    FWB(S.alloc(&d_segs, max_segs));
    FWB(S.alloc(&d_tiles, max_tiles));
    FWB(S.alloc(&d_split, max_segs));
    FWB(S.alloc(&d_sseg, max_segs));
    FWB(S.alloc(&d_stile, max_tiles));
    FWB(S.alloc(&d_agg, 3 * max_tiles));
    FWB(S.alloc(&d_pre, 3 * max_tiles));
    FWB(S.alloc(&d_suf, 3 * max_tiles));
    FWB(S.alloc(&d_best, 3 * max_tiles));
    FWB(cudaMemcpyAsync(d_boxes, leaf_boxes.data(), sizeof(Box) * (size_t)nl, cudaMemcpyHostToDevice, S.stream));
    FWB(cudaMemcpyAsync(d_counts, leaf_counts.data(), sizeof(int) * (size_t)nl, cudaMemcpyHostToDevice, S.stream));
    FWB(cudaMemcpyAsync(d_leaves, leaf_order.data(), sizeof(int) * (size_t)nl, cudaMemcpyHostToDevice, S.stream));
    centres_f64_kernel<<<blocks(nl), 256, 0, S.stream>>>(d_boxes, d_ctr, nl);
    // One level of the SAH recursion per pass; a node is (lo, n, depth) plus the record slot its parent keeps for it.
    struct Pending { int lo, n, depth, parent, side; };
    std::vector<Pending> level{Pending{0, nl, 0, -1, 0}};
    int root_ref = 0;
    auto link = [&](const Pending& p, int ref) {
        if (p.parent < 0) root_ref = ref;
        else if (p.side == 0) recs[p.parent].left = ref;
        else recs[p.parent].right = ref;
    };
    std::vector<int2> split;
    while (!level.empty()) {
        std::vector<Pending> work;
        for (const Pending& p : level) {
            if (p.n == 1) link(p, ~p.lo);   // a single leaf; its id is leaf_order[lo] once the parent's order is final
            else work.push_back(p);
        }
        if (work.empty()) break;
        std::vector<Seg> segs;
        std::vector<SahSeg> ssegs;
        std::vector<SahTile> stiles;
        for (const Pending& p : work) {
            segs.push_back(Seg{p.lo, p.n});
            const int t0 = (int)stiles.size();
            for (int t = 0; t < p.n; t += kTile) stiles.push_back(SahTile{(int)ssegs.size(), p.lo + t, std::min(kTile, p.n - t), t0});
            ssegs.push_back(SahSeg{p.lo, p.n, p.depth, t0, (int)stiles.size() - t0});
        }
        const int nseg = (int)segs.size(), ntiles = (int)stiles.size();
        FWB(cudaMemcpyAsync(d_sseg, ssegs.data(), ssegs.size() * sizeof(SahSeg), cudaMemcpyHostToDevice, S.stream));
        FWB(cudaMemcpyAsync(d_stile, stiles.data(), stiles.size() * sizeof(SahTile), cudaMemcpyHostToDevice, S.stream));
        // ord[0] = leaves by x, ord[1] = ord[0] by y, ord[2] = ord[1] by z, each stable
        for (int a = 0; a < 3; ++a) {
            const int* src = a == 0 ? d_leaves : d_ord + (size_t)(a - 1) * nl;
            FWB(cudaMemcpyAsync(d_vals, src, sizeof(int) * (size_t)nl, cudaMemcpyDeviceToDevice, S.stream));
            FWB(cudaMemcpyAsync(d_segs, segs.data(), segs.size() * sizeof(Seg), cudaMemcpyHostToDevice, S.stream));
            gather_keys_kernel<double><<<blocks(nl), 256, 0, S.stream>>>(d_ctr + (size_t)a * nl, d_vals, d_keys, nl, d_segs, nseg, nullptr);
            if (!sort_segments<double>(S, chk, d_keys, d_vals, d_kt, d_vt, nl, segs, d_segs, d_tiles)) return false;
            FWB(cudaMemcpyAsync(d_ord + (size_t)a * nl, d_vals, sizeof(int) * (size_t)nl, cudaMemcpyDeviceToDevice, S.stream));
        }
        sah_tile_reduce_kernel<<<dim3(ntiles, 3), kTile, 0, S.stream>>>(d_ord, d_boxes, d_counts, d_stile, ntiles, nl, d_agg);
        sah_seg_scan_kernel<<<blocks(3 * (size_t)nseg), 256, 0, S.stream>>>(d_sseg, nseg, ntiles, d_agg, d_pre, d_suf);
        sah_tile_cost_kernel<<<dim3(ntiles, 3), kTile, 0, S.stream>>>(d_ord, d_boxes, d_counts, d_stile, d_sseg, ntiles, nl, d_pre, d_suf,
                                                                      d_best, max_depth);
        sah_pick_kernel<<<blocks(nseg), 256, 0, S.stream>>>(d_sseg, nseg, ntiles, d_best, d_split);
        sah_apply_kernel<<<blocks(nl), 256, 0, S.stream>>>(d_ord, d_leaves, nl, d_segs, nseg, d_split);
        FWB(cudaGetLastError());
        split.resize(nseg);
        FWB(cudaMemcpyAsync(split.data(), d_split, sizeof(int2) * (size_t)nseg, cudaMemcpyDeviceToHost, S.stream));
        FWB(cudaStreamSynchronize(S.stream));
        std::vector<Pending> next;
        for (int s = 0; s < nseg; ++s) {
            const Pending& p = work[s];
            const int id = (int)recs.size();
            recs.push_back(SahRec{p.depth, 0, 0, split[s].y});
            link(p, id);
            const int k = split[s].y;
            next.push_back(Pending{p.lo, k, p.depth + 1, id, 0});
            next.push_back(Pending{p.lo + k, p.n - k, p.depth + 1, id, 1});
        }
        level.swap(next);
    }
    FWB(cudaMemcpyAsync(leaf_order.data(), d_leaves, sizeof(int) * (size_t)nl, cudaMemcpyDeviceToHost, S.stream));
    FWB(cudaStreamSynchronize(S.stream));
    // a root that is itself one leaf is returned as record -1 with the leaf in leaf_order[0]
    if (root_ref < 0) recs.clear();
    return true;
}

}  // namespace fw
