// C ABI implementation (include/firework_b200.h): scene lifecycle, upload, wavefront orchestration, probes.
#include <cuda_runtime.h>

#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <fstream>
#include <mutex>
#include <sstream>
#include <thread>
#include <string>
#include <vector>

#include "api_internal.h"

using namespace fw;

static thread_local std::string g_last_error;

// Pinned staging for equirect HDR maps (128 MiB as float4 at 4096 x 2048): fw_scene_set_hdr expands the caller's RGB
// texels straight into it (one multi-threaded pass), fw_scene_commit copies from it into the CUDA array.  The buffers
// are process-wide and grow-only; a scene holds one from set_hdr until its commit / destroy.
static std::mutex g_staging_mutex;
static std::vector<HdrStaging*> g_staging;
static HdrStaging* staging_acquire(size_t floats) {
    std::lock_guard<std::mutex> lk(g_staging_mutex);
    HdrStaging* best = nullptr;
    for (HdrStaging* h : g_staging)
        if (!h->in_use && (!best || h->floats > best->floats)) best = h;
    if (!best) { best = new HdrStaging(); g_staging.push_back(best); }
    if (best->floats < floats) {
        if (best->p) cudaFreeHost(best->p);
        best->p = nullptr; best->floats = 0;
        if (cudaMallocHost(&best->p, floats * sizeof(float)) != cudaSuccess) {   // no device / no pinned memory:
            cudaGetLastError();                                                // plain host memory still works
            best->p = nullptr;
            return nullptr;
        }
        best->floats = floats;
    }
    best->in_use = true;
    return best;
}
static void staging_release(HdrStaging* h) {
    if (!h) return;
    if (h->plain) { free(h->p); delete h; return; }
    std::lock_guard<std::mutex> lk(g_staging_mutex);
    h->in_use = false;
}
static void expand_rgb_to_rgba(const float* rgb, float* rgba, size_t texels) {
    unsigned nt = std::max(1u, std::min(8u, std::thread::hardware_concurrency()));
    if (texels < (1u << 18)) nt = 1;
    auto work = [=](size_t a, size_t b) {
        for (size_t p = a; p < b; ++p) {
            rgba[4 * p] = rgb[3 * p]; rgba[4 * p + 1] = rgb[3 * p + 1]; rgba[4 * p + 2] = rgb[3 * p + 2]; rgba[4 * p + 3] = 0.0f;
        }
    };
    std::vector<std::thread> th;
    size_t chunk = (texels + nt - 1) / nt;
    for (unsigned t = 1; t < nt; ++t) th.emplace_back(work, std::min(texels, t * chunk), std::min(texels, (t + 1) * chunk));
    work(0, std::min(texels, chunk));
    for (auto& t : th) t.join();
}
int fw::set_error(int code, const std::string& msg) {
    g_last_error = msg;
    return code;
}
int fw::set_last_error(int code, const std::string& msg) { return set_error(code, msg); }

static_assert(sizeof(fw_params) == sizeof(RenderParamsHost), "fw_params layout");
static_assert(sizeof(ShapeRec) == 48 && sizeof(MeshRec) == 64 && sizeof(MatRec) == 32 && sizeof(TexRec) == 32, "rec sizes");

static std::mutex g_ctx_mutex;
static std::vector<RenderCtx*> g_ctx_cache;

// ----------------------------------------------------------------------------------------------------------
// texture store: device-resident textures, process-wide, addressed by the content of the texels
// ----------------------------------------------------------------------------------------------------------
// A renderer that is handed the same environment map or image texture scene after scene (the usual case: one HDRI, many
// frames) spends more time copying 100 MB of texels to pinned memory and over PCIe than it spends rendering a small
// image.  fw_scene_set_image / fw_scene_set_hdr hash the caller's texels (128 bits, multi-threaded: ~1 ms per 100 MB);
// when an array with that content is already resident the host copy is skipped, and a commit onto the same device shares
// the array (textures are read-only).  FW_TEXTURE_CACHE=0 disables the lookup: every scene copies and uploads.
static std::mutex g_tex_mutex;
static std::vector<TexEntry*> g_tex;
static uint64_t g_tex_tick = 0, g_tex_hits = 0, g_tex_fills = 0;
static constexpr size_t kTexIdlePerDevice = 8;   // idle (unreferenced) arrays kept per device

static bool tex_store_enabled() {
    const char* e = getenv("FW_TEXTURE_CACHE");
    return !(e && e[0] == '0');
}
static inline uint64_t mix64(uint64_t a, uint64_t b) {
    __uint128_t m = (__uint128_t)a * b;
    return (uint64_t)m ^ (uint64_t)(m >> 64);
}
// Two interleaved multiply-fold chains over 32-byte blocks (each 8-byte word enters exactly one multiplication);
// not cryptographic — it guards against accidental reuse, the caller is trusted.
static void hash_span(const unsigned char* p, size_t n, uint64_t out[2]) {
    const uint64_t k0 = 0xa0761d6478bd642full, k1 = 0xe7037ed1a0b428dbull, k2 = 0x8ebc6af09c88c6e3ull, k3 = 0x589965cc75374cc3ull;
    uint64_t s0 = k0 ^ n, s1 = k1 + n;
    size_t i = 0;
    for (; i + 32 <= n; i += 32) {
        uint64_t w[4];
        memcpy(w, p + i, 32);
        s0 = mix64(w[0] ^ k2, w[1] ^ s0);
        s1 = mix64(w[2] ^ k3, w[3] ^ s1);
    }
    if (i < n) {
        uint64_t w[4] = {0, 0, 0, 0};
        memcpy(w, p + i, n - i);
        s0 = mix64(w[0] ^ k2, w[1] ^ s0);
        s1 = mix64(w[2] ^ k3, w[3] ^ s1);
    }
    out[0] = mix64(s0 ^ k1, s1 ^ k2);
    out[1] = mix64(s1 ^ k0, s0 + k3);
}
static AssetKey hash_texels(const void* data, size_t bytes, uint32_t w, uint32_t h, int kind) {
    AssetKey key;
    const unsigned char* p = static_cast<const unsigned char*>(data);
    const size_t piece = (size_t)1 << 20;
    const size_t n_pieces = std::max<size_t>(1, (bytes + piece - 1) / piece);
    std::vector<uint64_t> hs(2 * n_pieces);
    unsigned want = 16u;
    if (const char* e = getenv("FW_HASH_THREADS")) want = (unsigned)std::max(1, atoi(e));
    unsigned nt = (unsigned)std::min<size_t>(std::max(1u, std::min(want, std::thread::hardware_concurrency())), n_pieces);
    auto work = [&](unsigned t) {
        for (size_t k = t; k < n_pieces; k += nt) hash_span(p + k * piece, std::min(piece, bytes - k * piece), &hs[2 * k]);
    };
    std::vector<std::thread> th;
    for (unsigned t = 1; t < nt; ++t) th.emplace_back(work, t);
    work(0);
    for (auto& t : th) t.join();
    uint64_t a = 0x9e3779b97f4a7c15ull ^ w, b = 0xc2b2ae3d27d4eb4full ^ h ^ ((uint64_t)kind << 40);
    for (size_t k = 0; k < n_pieces; ++k) {   // piece order matters
        a = mix64(a ^ hs[2 * k], 0xd6e8feb86659fd93ull) + b;
        b = mix64(b ^ hs[2 * k + 1], 0xa0761d6478bd642full) + a;
    }
    key.hashed = true;
    key.hash[0] = a; key.hash[1] = b;
    return key;
}
static void tex_destroy(TexEntry* e) {
    cudaSetDevice(e->device);
    if (e->tex) cudaDestroyTextureObject(e->tex);
    if (e->arr) cudaFreeArray(e->arr);
    if (e->ready) cudaEventDestroy(e->ready);
    delete e;
}
// Resident entry with this content on any device (+1 reference), or null.
static TexEntry* tex_find_any(const AssetKey& key, uint32_t w, uint32_t h, bool is_float) {
    if (!key.hashed) return nullptr;
    std::lock_guard<std::mutex> lk(g_tex_mutex);
    for (TexEntry* e : g_tex)
        if (e->hashed && e->hash[0] == key.hash[0] && e->hash[1] == key.hash[1] && e->w == w && e->h == h && e->is_float == is_float) {
            ++e->refs;
            return e;
        }
    return nullptr;
}
static void tex_unref(TexEntry* e) {
    if (!e) return;
    std::lock_guard<std::mutex> lk(g_tex_mutex);
    --e->refs;
    e->last_use = ++g_tex_tick;
}
// The device state of a scene is gone (its stream was synchronised): drop its references, keep a few idle arrays.
static void tex_release(std::vector<TexEntry*>& used, int device) {
    std::lock_guard<std::mutex> lk(g_tex_mutex);
    for (TexEntry* e : used) { --e->refs; e->last_use = ++g_tex_tick; }
    used.clear();
    for (;;) {
        size_t idle = 0;
        size_t oldest = g_tex.size();
        for (size_t i = 0; i < g_tex.size(); ++i)
            if (g_tex[i]->device == device && g_tex[i]->refs == 0) {
                ++idle;
                if (oldest == g_tex.size() || g_tex[i]->last_use < g_tex[oldest]->last_use) oldest = i;
            }
        if (idle <= kTexIdlePerDevice) break;
        tex_destroy(g_tex[oldest]);
        g_tex.erase(g_tex.begin() + oldest);
    }
}


static int arena_alloc(fw_scene* sc, size_t bytes, void** out) {
    RenderCtx* c = sc->ctx;
    bytes = (bytes + 255) & ~(size_t)255;
    if (c->arena_used + bytes > c->arena_cap) {
        size_t cap = std::max<size_t>((size_t)8 << 20, 2 * (c->arena_used + bytes));
        char* slab = nullptr;
        FW_CUDA(cudaMalloc(&slab, cap));
        // tables already placed for this scene stay valid in the old slab until the scene is released
        if (c->arena) c->arena_retired.push_back(c->arena);
        c->arena = slab;
        c->arena_cap = cap;
        c->arena_used = 0;
    }
    *out = c->arena + c->arena_used;
    c->arena_used += bytes;
    return FW_OK;
}
// Small tables (a 500-object scene has seventeen of a few KB each) are gathered in a pinned staging buffer and go out as
// one copy per contiguous arena range: each cudaMemcpyAsync from pageable memory costs 5-10 us of driver time.
static constexpr size_t kStageCap = (size_t)4 << 20, kStageMaxTable = (size_t)256 << 10;
static int stage_flush(RenderCtx* c) {
    if (c->stage_len) {
        size_t n = c->stage_len;
        c->stage_len = 0;
        FW_CUDA(cudaMemcpyAsync(c->stage_dst, c->h_stage + c->stage_begin, n, cudaMemcpyHostToDevice, c->stream));
    }
    return FW_OK;
}
template <class T>
static int upload(fw_scene* sc, const std::vector<T>& host, const T** dev) {
    RenderCtx* c = sc->ctx;
    const size_t payload = host.size() * sizeof(T);
    size_t bytes = std::max<size_t>(payload, 64);
    void* p = nullptr;
    int rc = arena_alloc(sc, bytes, &p);
    if (rc != FW_OK) return rc;
    const size_t padded = (bytes + 255) & ~(size_t)255;   // what arena_alloc reserved
    if (!c->h_stage && !c->stage_failed) {
        if (cudaMallocHost(&c->h_stage, kStageCap) != cudaSuccess) { cudaGetLastError(); c->h_stage = nullptr; c->stage_failed = true; }
    }
    if (c->h_stage && padded <= kStageMaxTable) {
        if (c->stage_off + padded > kStageCap) {      // buffer full: wait for the copies that read it, start over
            if ((rc = stage_flush(c)) != FW_OK) return rc;
            FW_CUDA(cudaStreamSynchronize(c->stream));
            c->stage_off = 0;
        }
        if (!(c->stage_len > 0 && c->stage_dst + c->stage_len == static_cast<char*>(p))) {
            if ((rc = stage_flush(c)) != FW_OK) return rc;
            c->stage_begin = c->stage_off;
            c->stage_dst = static_cast<char*>(p);
        }
        char* h = c->h_stage + c->stage_off;
        if (payload) memcpy(h, host.data(), payload);
        if (padded > payload) memset(h + payload, 0, padded - payload);
        c->stage_off += padded;
        c->stage_len += padded;
    } else {
        if ((rc = stage_flush(c)) != FW_OK) return rc;
        if (host.empty()) FW_CUDA(cudaMemsetAsync(p, 0, bytes, c->stream));
        else FW_CUDA(cudaMemcpyAsync(p, host.data(), payload, cudaMemcpyHostToDevice, c->stream));
    }
    sc->h2d_bytes += payload;
    *dev = reinterpret_cast<const T*>(p);
    return FW_OK;
}

// Each family of render-context buffers has one function that frees it; destroy_ctx and the ensure_* that grow a family
// both call it, so a buffer added to a family is freed on both paths.
template <class T>
static void dev_free(T*& p) {
    if (p) { cudaFree(p); p = nullptr; }
}
// The path-state streams and the walk buffers sized with them.
static void free_path_state(RenderCtx* c) {
    PathState& ps = c->ps;
    for (int i = 0; i < 2; ++i) { dev_free(ps.xo[i]); dev_free(ps.xd[i]); }
    for (HitQueue& q : ps.hq) { dev_free(q.o); dev_free(q.d); dev_free(q.w); }
    dev_free(ps.atten); dev_free(ps.radiance); dev_free(ps.counters); dev_free(ps.poison);
    dev_free(c->walk.tkey); dev_free(c->walk.entries);
    c->walk = WalkAuxHost{};
    c->walk_key_cap = c->walk_ent_total = 0;
    c->ps_cap = 0;
}
static void free_sums(RenderCtx* c) {
    dev_free(c->d_sum); dev_free(c->d_rgb);
    c->d_sum_pix = 0;
}
static void free_adaptive(RenderCtx* c) {
    AdaptiveState& a = c->adapt;
    dev_free(a.m1); dev_free(a.m2); dev_free(a.count); dev_free(a.err); dev_free(a.list[0]); dev_free(a.list[1]); dev_free(a.keep);
    dev_free(a.block_base);
    c->adapt_pix = 0;
}
static void free_denoise(RenderCtx* c) {
    dev_free(c->aov.nz); dev_free(c->aov.alb); dev_free(c->aov.obj); dev_free(c->dn_cv[0]); dev_free(c->dn_cv[1]); dev_free(c->dn_planar);
    dev_free(c->dn_var); dev_free(c->dn_color);
    c->dn_pix = 0;
}
static void destroy_ctx(RenderCtx* c) {
    if (!c) return;
    cudaSetDevice(c->device);
    free_path_state(c);
    if (c->arena) cudaFree(c->arena);
    for (void* p : c->arena_retired) cudaFree(p);
    free_sums(c);
    free_adaptive(c);
    free_denoise(c);
    if (c->h_rays) cudaFreeHost(c->h_rays);
    if (c->h_stage) cudaFreeHost(c->h_stage);
    if (c->d_rays) cudaFree(c->d_rays);
    for (auto e : c->ev_pool) cudaEventDestroy(e);
    if (c->ev_begin) cudaEventDestroy(c->ev_begin);
    if (c->ev_end) cudaEventDestroy(c->ev_end);
    if (c->stream) cudaStreamDestroy(c->stream);
    delete c;
}

static int acquire_ctx(int device, RenderCtx** out) {
    {
        std::lock_guard<std::mutex> lk(g_ctx_mutex);
        for (RenderCtx* c : g_ctx_cache)
            if (c->device == device && !c->in_use) {
                c->in_use = true;
                *out = c;
                return FW_OK;
            }
    }
    RenderCtx* c = new RenderCtx();
    c->device = device;
    c->in_use = true;
    cudaError_t e = cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking);
    if (e == cudaSuccess) e = cudaEventCreate(&c->ev_begin);
    if (e == cudaSuccess) e = cudaEventCreate(&c->ev_end);
    if (e == cudaSuccess) e = cudaMallocHost(&c->h_rays, sizeof(unsigned long long));
    if (e == cudaSuccess) e = cudaMalloc(&c->d_rays, sizeof(unsigned long long));
    if (e != cudaSuccess) {
        destroy_ctx(c);
        return set_error(FW_ERR_CUDA, std::string("render context: ") + cudaGetErrorString(e));
    }
    {
        std::lock_guard<std::mutex> lk(g_ctx_mutex);
        g_ctx_cache.push_back(c);
    }
    *out = c;
    return FW_OK;
}

static void release_device(fw_scene* sc) {
    if (!sc) return;
    cudaSetDevice(sc->device);
    if (sc->ctx) {
        cudaStreamSynchronize(sc->ctx->stream);
        RenderCtx* c = sc->ctx;
        for (void* p : c->arena_retired) cudaFree(p);
        c->arena_retired.clear();
        c->arena_used = 0;                       // the next scene overwrites the tables
        tex_release(sc->tex_used, sc->device);
        std::lock_guard<std::mutex> lk(g_ctx_mutex);
        c->in_use = false;  // back to the cache
        sc->ctx = nullptr;
    }
    sc->committed = false;
}

// Nothing may propagate through the C ABI: entry points that allocate run their body through this.
template <class F>
static int guarded(F&& body) {
    try {
        return body();
    } catch (const std::bad_alloc&) {
        return set_error(FW_ERR_SCENE, "out of host memory");
    } catch (const std::exception& e) {
        return set_error(FW_ERR_SCENE, std::string("internal error: ") + e.what());
    } catch (...) {
        return set_error(FW_ERR_SCENE, "internal error");
    }
}

namespace {
struct DevBuf {  // tiny RAII helper for probe staging buffers
    void* p = nullptr;
    ~DevBuf() { if (p) cudaFree(p); }
    int alloc(size_t bytes) {
        FW_CUDA(cudaMalloc(&p, std::max<size_t>(bytes, 16)));
        return FW_OK;
    }
    int put(const void* src, size_t bytes) {
        int rc = alloc(bytes);
        if (rc != FW_OK) return rc;
        if (src && bytes) FW_CUDA(cudaMemcpy(p, src, bytes, cudaMemcpyHostToDevice));
        return FW_OK;
    }
    int get(void* dst, size_t bytes) {
        if (dst && bytes) FW_CUDA(cudaMemcpy(dst, p, bytes, cudaMemcpyDeviceToHost));
        return FW_OK;
    }
    template <class T> T* as() { return reinterpret_cast<T*>(p); }
};
// The seven per-ray outputs of the first-hit probes (FirstHitOut) and their copy back to the caller.
struct FirstHitBufs {
    DevBuf buf[7];   // obj, prim, material, t, point, normal, uv
    static constexpr size_t kBytes[7] = {4, 4, 4, 4, 12, 12, 8};   // per ray
    int alloc(uint32_t n) {
        for (int i = 0; i < 7; ++i)
            if (int rc = buf[i].alloc(n * kBytes[i]); rc != FW_OK) return rc;
        return FW_OK;
    }
    FirstHitOut out(unsigned long long* counters) {
        return FirstHitOut{buf[0].as<int>(), buf[1].as<int>(), buf[2].as<int>(), buf[3].as<float>(), buf[4].as<float>(), buf[5].as<float>(),
                           buf[6].as<float>(), counters};
    }
    int get(uint32_t n, int32_t* obj, int32_t* prim, int32_t* material, float* t, float* point, float* normal, float* uv) {
        void* dst[7] = {obj, prim, material, t, point, normal, uv};
        for (int i = 0; i < 7; ++i)
            if (int rc = buf[i].get(dst[i], n * kBytes[i]); rc != FW_OK) return rc;
        return FW_OK;
    }
};
}  // namespace

extern "C" {

const char* fw_last_error(void) { return g_last_error.c_str(); }
const char* fw_version(void) { return "firework_b200 0.1 (sm_100a)"; }
int fw_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) return 0;
    return n;
}

int fw_scene_from_yaml(const char* text, size_t len, fw_scene** out) {
    return guarded([&]() -> int {
        if (!text || !out) return set_error(FW_ERR_ARG, "null argument");
        auto sc = new fw_scene();
        std::string err;
        if (!load_scene_yaml(text, len, sc->desc, err)) {
            delete sc;
            return set_error(FW_ERR_PARSE, err);
        }
        *out = sc;
        return FW_OK;
});
}
int fw_scene_from_file(const char* path, fw_scene** out) {
    return guarded([&]() -> int {
        if (!path || !out) return set_error(FW_ERR_ARG, "null argument");
        std::ifstream f(path, std::ios::binary);
        if (!f) return set_error(FW_ERR_PARSE, std::string("cannot open ") + path);
        std::stringstream ss;
        ss << f.rdbuf();
        std::string text = ss.str();
        return fw_scene_from_yaml(text.data(), text.size(), out);
});
}
void fw_scene_destroy(fw_scene* sc) {
    if (!sc) return;
    for (fw_scene* r : sc->replicas) fw_scene_destroy(r);
    sc->replicas.clear();
    release_device(sc);   // synchronises the scene's stream: no upload from the staging buffers is still in flight
    if (!sc->asset_src)
        for (HdrStaging* h : sc->hdr_staging) staging_release(h);
    for (TexEntry* e : sc->asset_held) tex_unref(e);
    delete sc;
}

int fw_scene_num_assets(const fw_scene* sc) { return sc ? (int)sc->desc.assets.size() : 0; }
const char* fw_scene_asset_path(const fw_scene* sc, int i) {
    if (!sc || i < 0 || i >= (int)sc->desc.assets.size()) return nullptr;
    return sc->desc.assets[i].path.c_str();
}
int fw_scene_asset_kind(const fw_scene* sc, int i) {
    if (!sc || i < 0 || i >= (int)sc->desc.assets.size()) return set_error(FW_ERR_ARG, "asset index out of range");
    return sc->desc.assets[i].kind;
}
int fw_scene_set_image(fw_scene* sc, int i, uint32_t w, uint32_t h, const uint8_t* rgba) {
    return guarded([&]() -> int {
        if (!sc || !rgba || i < 0 || i >= (int)sc->desc.assets.size() || w == 0 || h == 0)
            return set_error(FW_ERR_ARG, "fw_scene_set_image: bad argument");
        AssetDesc& a = sc->desc.assets[i];
        if (a.kind != 0) return set_error(FW_ERR_ARG, "asset is not an image");
        if (sc->committed) return set_error(FW_ERR_STATE, "scene already committed");
        a.w = w; a.h = h;
        sc->asset_key.resize(sc->desc.assets.size());
        sc->asset_held.resize(sc->desc.assets.size(), nullptr);
        if (sc->asset_held[i]) { tex_unref(sc->asset_held[i]); sc->asset_held[i] = nullptr; }
        sc->asset_key[i] = tex_store_enabled() ? hash_texels(rgba, (size_t)w * h * 4, w, h, 0) : AssetKey();
        sc->asset_held[i] = tex_find_any(sc->asset_key[i], w, h, false);
        if (sc->asset_held[i]) { a.rgba.clear(); }   // resident already: no host copy (host_texels() reads it back if ever needed)
        else a.rgba.assign(rgba, rgba + (size_t)w * h * 4);
        a.provided = true;
        return FW_OK;
});
}
int fw_scene_set_hdr(fw_scene* sc, int i, uint32_t w, uint32_t h, const float* rgb) {
    return guarded([&]() -> int {
        if (!sc || !rgb || i < 0 || i >= (int)sc->desc.assets.size() || w == 0 || h == 0)
            return set_error(FW_ERR_ARG, "fw_scene_set_hdr: bad argument");
        AssetDesc& a = sc->desc.assets[i];
        if (a.kind != 1) return set_error(FW_ERR_ARG, "asset is not an HDR map");
        if (sc->committed) return set_error(FW_ERR_STATE, "scene already committed");
        a.w = w; a.h = h;
        const size_t texels = (size_t)w * h;
        sc->hdr_staging.resize(sc->desc.assets.size(), nullptr);
        if (sc->hdr_staging[i]) { staging_release(sc->hdr_staging[i]); sc->hdr_staging[i] = nullptr; }
        sc->asset_key.resize(sc->desc.assets.size());
        sc->asset_held.resize(sc->desc.assets.size(), nullptr);
        if (sc->asset_held[i]) { tex_unref(sc->asset_held[i]); sc->asset_held[i] = nullptr; }
        sc->asset_key[i] = tex_store_enabled() ? hash_texels(rgb, texels * 3 * sizeof(float), w, h, 1) : AssetKey();
        sc->asset_held[i] = tex_find_any(sc->asset_key[i], w, h, true);
        a.rgb.clear();
        if (!sc->asset_held[i]) {
            HdrStaging* st = staging_acquire(texels * 4);
            if (st) {
                expand_rgb_to_rgba(rgb, st->p, texels);
                sc->hdr_staging[i] = st;
            } else {
                a.rgb.assign(rgb, rgb + texels * 3);
            }
        }
        a.provided = true;
        return FW_OK;
});
}

// Host texels of asset i of `src` (RGBA8 in a.rgba, or RGBA fp32 in pinned staging): present unless set_* found the content
// resident and skipped the copy — then they are read back from that array (a commit onto another device, a replica).
static int host_texels(fw_scene* src, size_t i, const void** out) {
    AssetDesc& a = src->desc.assets[i];
    const size_t texels = (size_t)a.w * a.h;
    if (a.kind == 0) {
        if (a.rgba.size() == texels * 4) { *out = a.rgba.data(); return FW_OK; }
    } else {
        if (i < src->hdr_staging.size() && src->hdr_staging[i]) { *out = src->hdr_staging[i]->p; return FW_OK; }
    }
    TexEntry* e = i < src->asset_held.size() ? src->asset_held[i] : nullptr;
    if (e) {
        int cur = 0;
        cudaGetDevice(&cur);
        cudaSetDevice(e->device);
        cudaError_t err = cudaEventSynchronize(e->ready);
        const size_t row = (size_t)a.w * (a.kind == 0 ? 4 : 16);
        if (a.kind == 0) {
            a.rgba.resize(texels * 4);
            if (err == cudaSuccess) err = cudaMemcpy2DFromArray(a.rgba.data(), row, e->arr, 0, 0, row, a.h, cudaMemcpyDeviceToHost);
            *out = a.rgba.data();
        } else {
            src->hdr_staging.resize(src->desc.assets.size(), nullptr);
            HdrStaging* st = staging_acquire(texels * 4);
            if (!st) { cudaSetDevice(cur); return set_error(FW_ERR_CUDA, "no pinned memory for the texel read-back"); }
            src->hdr_staging[i] = st;
            if (err == cudaSuccess) err = cudaMemcpy2DFromArray(st->p, row, e->arr, 0, 0, row, a.h, cudaMemcpyDeviceToHost);
            *out = st->p;
        }
        cudaSetDevice(cur);
        if (err != cudaSuccess) return set_error(FW_ERR_CUDA, std::string("texel read-back: ") + cudaGetErrorString(err));
        return FW_OK;
    }
    if (a.kind == 1 && a.rgb.size() == texels * 3) {   // no pinned memory at set time: expand now
        src->hdr_staging.resize(src->desc.assets.size(), nullptr);
        HdrStaging* st = new HdrStaging();   // plain host memory, owned like a pooled buffer that is never reused
        st->p = static_cast<float*>(malloc(texels * 4 * sizeof(float)));
        if (!st->p) { delete st; return set_error(FW_ERR_SCENE, "out of host memory"); }
        st->floats = texels * 4; st->in_use = true; st->plain = true;
        expand_rgb_to_rgba(a.rgb.data(), st->p, texels);
        src->hdr_staging[i] = st;
        *out = st->p;
        return FW_OK;
    }
    return set_error(FW_ERR_ASSET, "asset `" + a.path + "` has no texels");
}

// Texture object for asset i of `src` on sc's device: shared when the content is resident there, else uploaded into an idle
// array of the same geometry or a new one.
static int make_texture(fw_scene* sc, fw_scene* src, size_t i, cudaTextureObject_t* out) {
    RenderCtx* c = sc->ctx;
    const AssetDesc& a = src->desc.assets[i];
    const bool is_float = a.kind == 1;
    const uint32_t w = a.w, h = a.h;
    const AssetKey key = i < src->asset_key.size() ? src->asset_key[i] : AssetKey();
    TexEntry* e = nullptr;
    if (key.hashed) {
        std::lock_guard<std::mutex> lk(g_tex_mutex);
        for (TexEntry* t : g_tex)
            if (t->device == sc->device && t->hashed && t->hash[0] == key.hash[0] && t->hash[1] == key.hash[1] && t->w == w && t->h == h &&
                t->is_float == is_float) { e = t; ++e->refs; ++g_tex_hits; break; }
    }
    if (e) {
        sc->tex_used.push_back(e);
        FW_CUDA(cudaStreamWaitEvent(c->stream, e->ready, 0));   // the fill may still be in flight on another scene's stream
        *out = e->tex;
        return FW_OK;
    }
    const void* texels = nullptr;
    int rc = host_texels(src, i, &texels);
    if (rc != FW_OK) return rc;
    const size_t row = (size_t)w * (is_float ? 16 : 4);
    {
        std::lock_guard<std::mutex> lk(g_tex_mutex);
        for (TexEntry* t : g_tex)
            if (t->device == sc->device && t->refs == 0 && t->w == w && t->h == h && t->is_float == is_float) {   // same geometry: refill
                e = t; ++e->refs; e->hashed = false;   // not addressable until the new content is in flight
                break;
            }
        ++g_tex_fills;
    }
    if (!e) {
        e = new TexEntry();
        e->device = sc->device; e->w = w; e->h = h; e->is_float = is_float; e->refs = 1;
        cudaChannelFormatDesc fmt = is_float ? cudaCreateChannelDesc<float4>() : cudaCreateChannelDesc<uchar4>();
        cudaError_t err = cudaMallocArray(&e->arr, &fmt, w, h);
        cudaResourceDesc rd;
        memset(&rd, 0, sizeof(rd));
        rd.resType = cudaResourceTypeArray;
        rd.res.array.array = e->arr;
        cudaTextureDesc td;
        memset(&td, 0, sizeof(td));
        td.addressMode[0] = td.addressMode[1] = cudaAddressModeClamp;
        td.filterMode = cudaFilterModePoint;  // nearest texel: texture.rs:296-309, hdri_test.rs:72-81
        td.readMode = cudaReadModeElementType;
        td.normalizedCoords = 0;
        if (err == cudaSuccess) err = cudaCreateTextureObject(&e->tex, &rd, &td, nullptr);
        if (err == cudaSuccess) err = cudaEventCreateWithFlags(&e->ready, cudaEventDisableTiming);
        if (err != cudaSuccess) {
            tex_destroy(e);
            return set_error(FW_ERR_CUDA, std::string("texture upload: ") + cudaGetErrorString(err));
        }
        std::lock_guard<std::mutex> lk(g_tex_mutex);
        g_tex.push_back(e);
    }
    sc->tex_used.push_back(e);
    FW_CUDA(cudaMemcpy2DToArrayAsync(e->arr, 0, 0, texels, row, row, h, cudaMemcpyHostToDevice, c->stream));
    FW_CUDA(cudaEventRecord(e->ready, c->stream));
    {
        std::lock_guard<std::mutex> lk(g_tex_mutex);
        e->hash[0] = key.hash[0]; e->hash[1] = key.hash[1];
        e->hashed = key.hashed;
    }
    sc->h2d_bytes += row * h;
    *out = e->tex;
    return FW_OK;
}

int fw_scene_build_host(fw_scene* sc) {
    return guarded([&]() -> int {
        if (!sc) return set_error(FW_ERR_ARG, "null scene");
        if (sc->built) return FW_OK;
        std::string err;
        if (!flatten_scene(sc->desc, sc->flat, err)) return set_error(FW_ERR_SCENE, err);
        sc->built = true;
        return FW_OK;
});
}

static int commit_uploads(fw_scene* sc);
int fw_scene_commit(fw_scene* sc, int device) {
    return guarded([&]() -> int {
        if (!sc) return set_error(FW_ERR_ARG, "null scene");
        if (sc->committed) return set_error(FW_ERR_STATE, "scene already committed");
        const fw_scene* src = sc->asset_src ? sc->asset_src : sc;
        for (const AssetDesc& a : src->desc.assets)
            if (!a.provided) return set_error(FW_ERR_ASSET, "asset `" + a.path + "` was not provided (fw_scene_set_image / fw_scene_set_hdr)");
        int brc = fw_scene_build_host(sc);
        if (brc != FW_OK) return brc;
        int ndev = 0;
        FW_CUDA(cudaGetDeviceCount(&ndev));
        if (device < 0 || device >= ndev) return set_error(FW_ERR_CUDA, "no such CUDA device " + std::to_string(device));
        sc->device = device;
        FW_CUDA(cudaSetDevice(device));
        {
            // device facts are queried once per device (cudaGetDeviceProperties costs milliseconds)
            static std::mutex info_mutex;
            static int cached_sm[64];
            static bool cached[64] = {false};
            std::lock_guard<std::mutex> lk(info_mutex);
            if (device < 64 && cached[device]) {
                sc->sm_count = cached_sm[device];
            } else {
                int smc = 0;
                FW_CUDA(cudaDeviceGetAttribute(&smc, cudaDevAttrMultiProcessorCount, device));
                sc->sm_count = smc;
                if (device < 64) { cached_sm[device] = sc->sm_count; cached[device] = true; }
            }
        }
        {
            int crc = acquire_ctx(device, &sc->ctx);
            if (crc != FW_OK) return crc;
        }
        int urc = commit_uploads(sc);
        if (urc != FW_OK) release_device(sc);   // hand the context back: a retry acquires it again
        return urc;
});
}
static int commit_uploads(fw_scene* sc) {
    // texels are read (and, after a set-time cache hit, lazily materialised) through the scene the replica was cloned from
    fw_scene* src = sc->asset_src ? const_cast<fw_scene*>(sc->asset_src) : sc;
    DeviceScene& D = sc->dscene;
    const HostFlat& F = sc->flat;
    int rc;
    sc->ctx->stage_off = sc->ctx->stage_len = 0;   // the context was synchronised when its previous scene let go of it
#define UP(field) if ((rc = upload(sc, F.field, &D.field)) != FW_OK) return rc
    UP(nodes); UP(top_leaves); UP(top_items); UP(leaf_posr); UP(leaf_meta); UP(obj_posr); UP(obj_meta); UP(obj_rot); UP(obj_irot); UP(shapes); UP(meshes);
    UP(tri_verts); UP(tri_perm); UP(tri_normals); UP(tri_uvs); UP(mats); UP(texs);
#undef UP
    std::vector<ImageRec> images(std::max<size_t>(sc->desc.assets.size(), 1));
    memset(images.data(), 0, images.size() * sizeof(ImageRec));
    memset(&D.env, 0, sizeof(D.env));
    D.env.kind = sc->desc.env_kind;
    for (int k = 0; k < 3; ++k) { D.env.a[k] = sc->desc.env_a[k]; D.env.b[k] = sc->desc.env_b[k]; }
    for (size_t i = 0; i < src->desc.assets.size(); ++i) {
        const AssetDesc& a = src->desc.assets[i];
        // host texels (a.rgba / the pinned staging copy) stay with the scene until fw_scene_destroy: the upload is
        // asynchronous, and fw_render_multi replicates the scene onto other devices from them
        cudaTextureObject_t t;
        if ((rc = make_texture(sc, src, i, &t)) != FW_OK) return rc;
        if (a.kind == 0) {
            images[i].tex = t; images[i].w = a.w; images[i].h = a.h;
        } else if ((int)i == sc->desc.env_asset) {
            D.env.tex = t; D.env.w = a.w; D.env.h = a.h;
        }
    }
    if ((rc = upload(sc, images, &D.images)) != FW_OK) return rc;
    if ((rc = stage_flush(sc->ctx)) != FW_OK) return rc;
    D.n_objects = (int)sc->desc.objects.size();
    D.n_nodes = (int)(F.nodes.size() / 8);
    D.n_tris = (int)(F.tri_verts.size() / 3);
    D.n_top_leaves = (int)(F.top_leaves.size() / 2);
    {
        int rc_bits = F.top_root_code;
        float rcf;
        memcpy(&rcf, &rc_bits, 4);
        D.top_lo = make_float4(F.top_root_box.mn.x, F.top_root_box.mn.y, F.top_root_box.mn.z, rcf);
        D.top_hi = make_float4(F.top_root_box.mx.x, F.top_root_box.mx.y, F.top_root_box.mx.z, 0.0f);
    }
    D.top_root_is_valid = 1;
    D.has_medium = F.has_medium ? 1 : 0;
    D.has_unbounded = F.has_unbounded ? 1 : 0;
    D.nan_bvh_obj = F.nan_bvh_obj; D.nan_bvh_prim = F.nan_bvh_prim;
    D.nan_lin_obj = F.nan_lin_obj; D.nan_lin_prim = F.nan_lin_prim;
    for (int k = 0; k < FW_MAX_WALK_MESHES; ++k) {
        D.mesh_rank[k] = F.mesh_rank[k];
        D.mesh_root[k] = D.mesh_tri0[k] = 0;
        if (F.walk_ok && k < F.n_top_meshes) {
            const ShapeRec& sh = F.shapes[F.obj_meta[F.top_items[F.mesh_rank[k]]].z];
            D.mesh_root[k] = F.meshes[sh.i0].root_code;
            D.mesh_tri0[k] = F.meshes[sh.i0].tri_first;
        }
    }
    for (const MatRec& m : F.mats) sc->mat_present[m.kind] = true;
    {
        // render.rs:31 with a black ColorEnv: an escaping path returns attenuation-chain * 0.  That is exactly 0
        // (radiance is pre-zeroed by raygen; adding +-0 never changes a sum that started at +0) as long as no
        // attenuation can be NaN / inf: all texture values are scene constants or u8 texels (procedural noise is
        // excluded because a NaN hit point would make it NaN), of magnitude <= 1e3 so ten factors cannot overflow.
        bool ok = sc->desc.env_kind == ENV_COLOR && sc->desc.env_a[0] == 0.0f && sc->desc.env_a[1] == 0.0f && sc->desc.env_a[2] == 0.0f;
        auto small = [](float v) { return std::fabs(v) <= 1e3f; };   // false for NaN
        for (const TexRec& t : F.texs) {
            if (t.kind == TEX_PERLIN || t.kind == TEX_TURBULENCE || t.kind == TEX_MARBLE) ok = false;
            if (t.kind == TEX_CONSTANT && !(small(t.color[0]) && small(t.color[1]) && small(t.color[2]))) ok = false;
        }
        for (const MatRec& m : F.mats)
            if (m.kind == MAT_METAL && !(small(m.albedo[0]) && small(m.albedo[1]) && small(m.albedo[2]))) ok = false;
        sc->miss_is_zero = ok;
        sc->env_black = sc->desc.env_kind == ENV_COLOR && sc->desc.env_a[0] == 0.0f && sc->desc.env_a[1] == 0.0f && sc->desc.env_a[2] == 0.0f;
        if (const char* e = getenv("FW_BLACK_ENV_SKIP")) sc->env_black = sc->env_black && atoi(e) != 0;
    }
    sc->lin_prog_ok = F.lin_words.size() <= (size_t)FW_LIN_MAX_WORDS;
    if (const char* e = getenv("FW_LINEAR_PROGRAM")) sc->lin_prog_ok = sc->lin_prog_ok && atoi(e) != 0;
    memset(&sc->lin_prog, 0, sizeof(sc->lin_prog));
    if (sc->lin_prog_ok) memcpy(sc->lin_prog.w, F.lin_words.data(), F.lin_words.size() * sizeof(float4));
    sc->plan.has_mesh = F.has_mesh; sc->plan.has_top_mesh = F.has_top_mesh; sc->plan.has_medium_mesh = F.has_medium_mesh;
    sc->plan.lin_prog_ok = sc->lin_prog_ok; sc->plan.lin_generic = F.lin_generic; sc->plan.lin_rect_tests = F.lin_rect_tests;
    sc->plan.small_top = F.top_leaves.size() / 2 <= 16;   // few top-level leaves: scanned straight through (pass 1 of the mesh walk)
    sc->plan.walk = F.walk_ok && F.has_top_mesh;   // mesh walk kernels (sphere-only trees stay on the lock-step kernel)
    // uploads ran on the context's stream; renders may be issued on another one (fw_render_accumulate_device)
    FW_CUDA(cudaStreamSynchronize(sc->ctx->stream));
    sc->committed = true;
    return FW_OK;
}

uint64_t fw_scene_device_bytes(const fw_scene* sc) { return sc ? sc->h2d_bytes : 0; }
int fw_scene_num_objects(const fw_scene* sc) { return sc ? (int)sc->desc.objects.size() : 0; }
int fw_scene_num_nodes(const fw_scene* sc) { return sc && sc->built ? (int)(sc->flat.nodes.size() / 8) : 0; }
int fw_scene_top_leaf_order(const fw_scene* sc, int* out, int cap) {
    if (!sc || !sc->built) return set_error(FW_ERR_STATE, "scene not built (fw_scene_build_host / fw_scene_commit)");
    int n = (int)sc->flat.top_items.size();
    if (out) for (int i = 0; i < std::min(n, cap); ++i) out[i] = sc->flat.top_items[i];
    return n;
}
int fw_scene_object_aabb(const fw_scene* sc, int obj, float o[6]) {
    if (!sc || !sc->built) return set_error(FW_ERR_STATE, "scene not built (fw_scene_build_host / fw_scene_commit)");
    if (obj < 0 || obj >= (int)sc->flat.obj_aabb.size() || !o) return set_error(FW_ERR_ARG, "bad object index");
    const Box& b = sc->flat.obj_aabb[obj];
    o[0] = b.mn.x; o[1] = b.mn.y; o[2] = b.mn.z; o[3] = b.mx.x; o[4] = b.mx.y; o[5] = b.mx.z;
    return FW_OK;
}
int fw_scene_mesh_leaf_order(const fw_scene* sc, int obj, int* out, int cap) {
    if (!sc || !sc->built) return set_error(FW_ERR_STATE, "scene not built (fw_scene_build_host / fw_scene_commit)");
    if (obj < 0 || obj >= (int)sc->desc.objects.size()) return set_error(FW_ERR_ARG, "bad object index");
    const ShapeRec& s = sc->flat.shapes[sc->desc.objects[obj].shape];
    if (s.kind != SH_MESH) return set_error(FW_ERR_ARG, "object is not a TriangleMesh");
    const MeshRec& m = sc->flat.meshes[s.i0];
    if (out)
        for (int i = 0; i < std::min(m.tri_count, cap); ++i) {
            int t;
            memcpy(&t, &sc->flat.tri_verts[3 * (size_t)(m.tri_first + i)].w, 4);
            out[i] = t;
        }
    return m.tri_count;
}
int fw_scene_bvh_nodes(const fw_scene* sc, float* out, int cap_nodes, int* top_root_code) {
    if (!sc || !sc->built) return set_error(FW_ERR_STATE, "scene not built (fw_scene_build_host / fw_scene_commit)");
    int n = (int)(sc->flat.nodes.size() / 8);
    if (out) memcpy(out, sc->flat.nodes.data(), sizeof(float4) * 8 * (size_t)std::max(0, std::min(n, cap_nodes)));
    if (top_root_code) *top_root_code = sc->flat.top_root_code;
    return n;
}
int fw_scene_linear_program(const fw_scene* sc, float* out, int cap) {
    if (!sc || !sc->built) return set_error(FW_ERR_STATE, "scene not built (fw_scene_build_host / fw_scene_commit)");
    int n = (int)sc->flat.lin_words.size();
    if (out) memcpy(out, sc->flat.lin_words.data(), sizeof(float4) * (size_t)std::max(0, std::min(n, cap)));
    return n;
}
int fw_scene_walk_info(const fw_scene* sc, int out[6]) {
    if (!sc || !sc->built || !out) return set_error(FW_ERR_STATE, "scene not built (fw_scene_build_host / fw_scene_commit)");
    const HostFlat& F = sc->flat;
    out[0] = F.walk_ok ? 1 : 0; out[1] = F.n_top_meshes; out[2] = F.top_wide_depth; out[3] = F.mesh_wide_depth;
    out[4] = F.walk_prim_bits; out[5] = (int)(F.tri_verts.size() / 3);
    return FW_OK;
}
int fw_material_texture(const fw_scene* sc, int material) {
    if (!sc || material < 0 || material >= (int)sc->desc.mats.size()) return -1;
    return sc->desc.mats[material].tex;
}
int fw_camera(const fw_params* p, float out[24]) {
    if (!p || !out) return set_error(FW_ERR_ARG, "null argument");
    RenderParamsHost hp;
    memcpy(&hp, p, sizeof(hp));
    CameraRec c = make_camera(hp);
    memcpy(out, &c, sizeof(float) * 22);
    out[22] = out[23] = 0.0f;
    return FW_OK;
}
// Idle render contexts keep their path state (gigabytes each) for the next scene; when an allocation fails they are the first
// thing to give back.  Returns how many were destroyed; the caller's current device stays current.
static size_t destroy_idle_contexts() {
    std::lock_guard<std::mutex> lk(g_ctx_mutex);
    std::vector<RenderCtx*> keep, idle;
    for (RenderCtx* c : g_ctx_cache) (c->in_use ? keep : idle).push_back(c);
    g_ctx_cache.swap(keep);
    if (!idle.empty()) {
        int cur = 0;
        cudaGetDevice(&cur);
        for (RenderCtx* c : idle) destroy_ctx(c);   // each on its own device
        cudaSetDevice(cur);
    }
    return idle.size();
}
int fw_release_cached_memory(void) {
    destroy_idle_contexts();
    {
        std::lock_guard<std::mutex> lk2(g_staging_mutex);
        for (HdrStaging* h : g_staging)
            if (!h->in_use && h->p) { cudaFreeHost(h->p); h->p = nullptr; h->floats = 0; }
    }
    {
        std::lock_guard<std::mutex> lk3(g_tex_mutex);
        std::vector<TexEntry*> keep_tex;
        for (TexEntry* e : g_tex) {
            if (e->refs > 0) keep_tex.push_back(e);
            else tex_destroy(e);
        }
        g_tex.swap(keep_tex);
    }
    return FW_OK;
}
int fw_texture_store_stats(uint64_t out[4]) {
    if (!out) return set_error(FW_ERR_ARG, "null output");
    std::lock_guard<std::mutex> lk(g_tex_mutex);
    out[0] = g_tex_hits; out[1] = g_tex_fills; out[2] = g_tex.size(); out[3] = 0;
    for (TexEntry* e : g_tex) out[3] += (uint64_t)e->w * e->h * (e->is_float ? 16 : 4);
    return FW_OK;
}
int fw_set_profiling(fw_scene* sc, int enabled) {
    if (!sc) return set_error(FW_ERR_ARG, "null scene");
    sc->profiling = enabled != 0;
    return FW_OK;
}
int fw_set_batch_paths(fw_scene* sc, uint64_t paths) {
    if (!sc) return set_error(FW_ERR_ARG, "null scene");
    sc->batch_paths = (size_t)paths;
    return FW_OK;
}

}  // extern "C"

// ----------------------------------------------------------------------------------------------------------
// wavefront orchestration
// ----------------------------------------------------------------------------------------------------------
// Segment geometry of a batch of `n` paths (wavefront.cuh "segmented queues"): enough segments to give every SM
// several blocks, few enough that a segment still holds whole tiles.
#ifndef FW_DEFAULT_BATCH_PATHS
#define FW_DEFAULT_BATCH_PATHS (1ull << 27)
#endif
static constexpr uint32_t FW_SEG_PER_SM_MAX = 32;   // measured: sm x 32 (segment-count sweep, profiles/r01_extend_variants.md)
static void segment_geometry(const fw_scene* sc, size_t n, uint32_t* nseg, uint32_t* seg_cap) {
    size_t tiles = (n + FW_TILE - 1) / FW_TILE;
    size_t want = std::max<size_t>((size_t)sc->sm_count, std::min<size_t>((size_t)sc->sm_count * FW_SEG_PER_SM_MAX, tiles / 8));
    *nseg = (uint32_t)want;
    *seg_cap = (uint32_t)(((tiles + want - 1) / want) * FW_TILE);
}

// Path-state streams for batches of up to `cap` paths.  Only the shade queues of materials present in the scene
// (and the mesh queue / barycentric streams when it has TriangleMesh objects) are allocated; a cached context
// grows on demand when a later scene needs more.
static int ensure_path_state(fw_scene* sc, size_t cap) {
    RenderCtx* ctx = sc->ctx;
    const size_t nseg_max = (size_t)sc->sm_count * FW_SEG_PER_SM_MAX;
    PathState& ps = ctx->ps;
    if (ctx->ps_cap < cap || ctx->ps_nseg_max < nseg_max) free_path_state(ctx);
    cap = std::max(cap, ctx->ps_cap);   // streams added later for another scene get the context's full size
    // queue regions: nseg * seg_cap <= n + nseg * FW_TILE slots for any batch of n <= cap paths
    const size_t qcap = cap + (nseg_max + 1) * FW_TILE;
    auto need = [&](float4*& p, size_t n) -> int {
        if (p) return FW_OK;
        FW_CUDA(cudaMalloc(&p, n * sizeof(float4)));
        return FW_OK;
    };
    int rc;
#define NEED(ptr, n) if ((rc = need(ptr, n)) != FW_OK) return rc
    for (int i = 0; i < 2; ++i) { NEED(ps.xo[i], qcap); NEED(ps.xd[i], qcap); }
    NEED(ps.atten, cap * FW_MAX_DEPTH);
    NEED(ps.radiance, cap);
    for (int k = 0; k < 8; ++k) {   // ps.hq[]
        bool used = k == MAT_MISS || (k < MAT_NUM_QUEUES && sc->mat_present[k]) ||
                    (k == FW_Q_MESH && sc->flat.has_top_mesh);   // rays that enter a mesh (two-pass extend / mesh walk)
        if (!used) continue;
        NEED(ps.hq[k].d, qcap);
        if (k == MAT_MISS) continue;
        NEED(ps.hq[k].o, qcap);
        NEED(ps.hq[k].w, qcap);
    }
#undef NEED
    if (sc->plan.walk) {
        // walk kernels (only scenes with top-level meshes get them): one 64-bit key per queue slot, and an entry queue with
        // room for every (ray, mesh) combination of a segment (n_top_meshes <= 8 is part of walk_ok)
        const size_t ent_per_seg_max = (size_t)sc->flat.n_top_meshes;
        const size_t ent_total = qcap * ent_per_seg_max;
        if (ctx->walk_key_cap < qcap) {
            dev_free(ctx->walk.tkey);
            ctx->walk_key_cap = 0;
            FW_CUDA(cudaMalloc(&ctx->walk.tkey, qcap * sizeof(unsigned long long)));
            ctx->walk_key_cap = qcap;
        }
        if (ctx->walk_ent_total < ent_total) {
            dev_free(ctx->walk.entries);
            ctx->walk_ent_total = 0;
            FW_CUDA(cudaMalloc(&ctx->walk.entries, ent_total * sizeof(uint4)));
            ctx->walk_ent_total = ent_total;
        }
    }
    ctx->walk.prim_bits = sc->flat.walk_prim_bits;
    if (!ps.poison) FW_CUDA(cudaMalloc(&ps.poison, 256));
    if (!ps.counters) FW_CUDA(cudaMalloc(&ps.counters, sizeof(uint32_t) * (FW_MAX_DEPTH + 2) * FW_NUM_QUEUES * nseg_max));
    ps.cap = (uint32_t)cap;
    ctx->ps_cap = cap;
    ctx->ps_nseg_max = nseg_max;
    return FW_OK;
}

// One render call of `p` on `sc`: what its batches share, and the totals that finish_call turns into fw_stats.  The camera and
// seed are built here alone, for every render entry point and fw_primary_rays.  A trace call (fw_trace_rays) sets `rays`
// instead: its params only carry the ray count as the width (height 1), the seed and use_bvh, and it has no camera.
struct CallFrame {
    fw_scene* sc;
    const fw_params* p;
    const RaySource* rays;
    CameraRec cam;
    uint2 seed;
    cudaStream_t st;
    size_t cap = 0;        // paths per batch (begin_call)
    uint64_t launches = 0, extend_launches = 0;
    std::vector<std::pair<cudaEvent_t, cudaEvent_t>> extend_events;   // fw_set_profiling: one pair per extend of run_batch
    size_t ev_next = 0;    // next free event of the context's pool
    CallFrame(fw_scene* s, const fw_params* q, cudaStream_t stream, const RaySource* r = nullptr) : sc(s), p(q), rays(r), st(stream) {
        memset(&cam, 0, sizeof(cam));
        if (!rays) {
            RenderParamsHost hp;
            memcpy(&hp, q, sizeof(hp));
            cam = make_camera(hp);
        }
        seed = make_uint2((uint32_t)q->seed, (uint32_t)(q->seed >> 32));
    }
};

static int get_event(fw_scene* sc, size_t& next, cudaEvent_t* ev) {
    if (next >= sc->ctx->ev_pool.size()) {
        cudaEvent_t e;
        FW_CUDA(cudaEventCreate(&e));
        sc->ctx->ev_pool.push_back(e);
    }
    *ev = sc->ctx->ev_pool[next++];
    return FW_OK;
}

unsigned fw::grid_for(size_t n, unsigned threads, unsigned max_blocks) {
    size_t g = (n + threads - 1) / threads;
    return (unsigned)std::max<size_t>(1, std::min<size_t>(g, max_blocks));
}

// FW_DEBUG_SYNC=1: synchronise after every kernel stage and name the one that faulted (debugging aid; slow).
static int sync_stage(cudaStream_t st, const char* what, uint32_t bounce) {
    static const bool debug_sync = getenv("FW_DEBUG_SYNC") != nullptr;
    if (!debug_sync) return FW_OK;
    cudaError_t e = cudaStreamSynchronize(st);
    if (e == cudaSuccess) e = cudaGetLastError();
    if (e != cudaSuccess)
        return set_error(FW_ERR_CUDA, std::string(what) + " (bounce " + std::to_string(bounce) + "): " + cudaGetErrorString(e));
    return FW_OK;
}
#define FW_STAGE(what, bounce) do { int rc__ = sync_stage(st, what, bounce); if (rc__ != FW_OK) return rc__; } while (0)

// The extend of one bounce, chosen from the scene alone: the collect / test mesh walk where the plan allows it, else the
// lock-step or linear-scan kernels of launch_extend.  Renders and fw_first_hit_wavefront both come here, so the probe runs
// exactly the kernels a render runs.  Adds the number of kernels launched to `launches`.
static int extend_bounce(fw_scene* sc, bool use_bvh, const Batch& b, uint2 seed, uint32_t bounce, cudaStream_t st, uint64_t& launches) {
    const PathState& ps = sc->ctx->ps;
    if (!(use_bvh && sc->plan.walk)) {
        launches += launch_extend(sc->plan, use_bvh, sc->lin_prog, sc->dscene, ps, b, seed, bounce, st);
        return FW_OK;
    }
    WalkAuxHost ax = sc->ctx->walk;
    ax.ent_cap = ps.seg_cap * (uint32_t)std::max(1, sc->flat.n_top_meshes);
    static const char* const part_name[3] = {"extend pass 1 (entries)", "mesh walk", "mesh classify"};
    for (int part = 0; part < 3; ++part) {
        launch_extend_walk_part(part, sc->plan, sc->dscene, ps, b, seed, bounce, ax, st);
        launches++;
        FW_STAGE(part_name[part], bounce);
    }
    return FW_OK;
}

// Segment geometry of a batch of `paths` paths, its queue counters and the poison word zeroed.
static int begin_batch(fw_scene* sc, size_t paths, cudaStream_t st) {
    PathState& ps = sc->ctx->ps;
    segment_geometry(sc, paths, &ps.nseg, &ps.seg_cap);
    FW_CUDA(cudaMemsetAsync(ps.counters, 0, sizeof(uint32_t) * (FW_MAX_DEPTH + 2) * FW_NUM_QUEUES * (size_t)ps.nseg, st));
    FW_CUDA(cudaMemsetAsync(ps.poison, 0, sizeof(uint32_t), st));
    return FW_OK;
}

// One batch: raygen (from the camera, or from the call's rays), up to FW_MAX_DEPTH+1 extend/shade rounds, accumulate into d_sum
// (and, for an adaptive or denoised render, into the moments and counts of `adapt`).
static int run_batch(CallFrame& f, const Batch& b, float* d_sum, const AdaptiveState* adapt) {
    fw_scene* sc = f.sc;
    const cudaStream_t st = f.st;
    PathState& ps = sc->ctx->ps;
    const DeviceScene& S = sc->dscene;
    int rc = begin_batch(sc, (size_t)b.npix * b.ns, st);
    if (rc != FW_OK) return rc;
    unsigned sm = (unsigned)sc->sm_count;
    if (f.rays) launch_raygen_rays(*f.rays, b, ps, st);
    else launch_raygen(f.cam, b, f.seed, ps, st);
    f.launches++;
    FW_STAGE("raygen", 0);
    for (uint32_t bounce = 0; bounce <= (uint32_t)FW_MAX_DEPTH; ++bounce) {
        cudaEvent_t e0 = nullptr, e1 = nullptr;
        if (sc->profiling) {
            if ((rc = get_event(sc, f.ev_next, &e0)) != FW_OK || (rc = get_event(sc, f.ev_next, &e1)) != FW_OK) return rc;
            FW_CUDA(cudaEventRecord(e0, st));
        }
        if ((rc = extend_bounce(sc, f.p->use_bvh != 0, b, f.seed, bounce, st, f.launches)) != FW_OK) return rc;
        if (sc->profiling) {
            FW_CUDA(cudaEventRecord(e1, st));
            f.extend_events.emplace_back(e0, e1);
        }
        f.extend_launches++;
        FW_STAGE("extend", bounce);
        if (!sc->miss_is_zero) {
            launch_miss(S, ps, bounce, sc->env_black, st);
            f.launches++;
            FW_STAGE("miss", bounce);
        }
        if (sc->mat_present[MAT_EMISSIVE]) {
            launch_shade_emissive(S, ps, bounce, st);
            f.launches++;
            FW_STAGE("shade emissive", bounce);
        }
        if (bounce < (uint32_t)FW_MAX_DEPTH) {
            for (int mat : {MAT_LAMBERTIAN, MAT_METAL, MAT_DIELECTRIC, MAT_ISOTROPIC})
                if (sc->mat_present[mat]) {
                    launch_shade_scatter(mat, S, ps, b, f.seed, bounce, st);
                    f.launches++;
                    FW_STAGE(mat == MAT_LAMBERTIAN ? "shade lambertian" : mat == MAT_METAL ? "shade metal" : mat == MAT_DIELECTRIC ? "shade dielectric" : "shade isotropic", bounce);
                }
        }
    }
    if (adapt) launch_accumulate_adaptive(d_sum, *adapt, ps, b, grid_for(b.npix, 256, sm * 8), st);
    else launch_accumulate(d_sum, ps, b, grid_for(b.npix, 256, sm * 8), st);
    f.launches++;
    launch_tally(ps, sc->ctx->d_rays, st);
    f.launches++;
    FW_STAGE("accumulate / tally", 0);
#undef FW_STAGE
    FW_CUDA(cudaGetLastError());
    return FW_OK;
}

// Paths in flight per batch for a render of `paths` paths in all, and path state for batches of that size (FW_BATCH_PATHS /
// fw_set_batch_paths, shrunk to what the device can give).  Results do not depend on the batch split, only the speed does.
static int prepare_batches(fw_scene* sc, size_t paths, size_t* cap_out) {
    // Paths in flight per batch.  Larger batches keep the deep, thinly populated bounces big enough to fill the
    // GPU and amortise the ~8 launches per bounce (measured: +6 % cornell, +18 % random_spheres, +34 % teapot
    // from 4 Mi to 32 Mi paths; part2_all at 4K another +6 % / +9 % at 64 Mi / 128 Mi); up to ~500 B of state per path
    // (five material queues) -> 66 GB at 128 Mi paths, laid out for the 180 GB of HBM3e of a B200.
    size_t cap = sc->batch_paths ? sc->batch_paths : ((size_t)FW_DEFAULT_BATCH_PATHS);
    if (const char* e = getenv("FW_BATCH_PATHS")) cap = std::max<size_t>(1024, strtoull(e, nullptr, 10));
    cap = std::min<size_t>(cap, paths);
    cap = std::max<size_t>(cap, 32);
    int rc;
    if (cap > sc->ctx->ps_cap) {
        // The context has to grow: keep the batch inside what the device can give (other scenes of this process hold
        // contexts of their own).
        size_t queues = 1;   // + mesh queue
        for (int k = 0; k < MAT_NUM_QUEUES; ++k) queues += (k != MAT_MISS && sc->mat_present[k]) ? 1 : 0;
        const size_t per_path = 64 + 16 * FW_MAX_DEPTH + 16 + 16 + 48 * queues + (sc->plan.walk ? 8 + 16 * (size_t)sc->flat.n_top_meshes : 0);
        size_t free_b = 0, total_b = 0;
        FW_CUDA(cudaMemGetInfo(&free_b, &total_b));
        double budget = 0.8 * ((double)free_b + (double)sc->ctx->ps_cap * per_path);
        // idle contexts of earlier scenes hold path state nobody is using
        if ((double)cap * per_path > budget && destroy_idle_contexts() > 0) {
            FW_CUDA(cudaMemGetInfo(&free_b, &total_b));
            budget = 0.8 * ((double)free_b + (double)sc->ctx->ps_cap * per_path);
        }
        while (cap > ((size_t)1 << 22) && (double)cap * per_path > budget) cap >>= 1;
    }
    for (bool freed_idle = false;;) {   // ... and if the allocation still fails: idle contexts give their memory back, then halve
        rc = ensure_path_state(sc, cap);
        if (rc == FW_OK || cudaPeekAtLastError() != cudaErrorMemoryAllocation) break;
        cudaGetLastError();
        free_path_state(sc->ctx);
        if (!freed_idle) {
            freed_idle = true;
            if (destroy_idle_contexts() > 0) continue;   // same size again
        }
        if (cap <= ((size_t)1 << 20)) break;
        cap >>= 1;
    }
    if (rc != FW_OK) return rc;
    *cap_out = std::min<size_t>(cap, sc->ctx->ps_cap);
    return FW_OK;
}

// ceil(2^32 / n), 0xffffffff for n <= 1: the magic number of div_magic / batch_path.
static uint32_t div_magic_number(uint32_t n) { return n <= 1 ? 0xffffffffu : (uint32_t)((((uint64_t)1 << 32) + n - 1) / n); }
// Samples [s0, s0 + ns) of pixels pix0 .. pix0 + npix - 1 of a width x height image, or of those entries of the pixel list `pixels`.
static Batch make_batch(uint32_t pix0, uint32_t npix, uint32_t s0, uint32_t ns, uint32_t width, uint32_t height, const uint32_t* pixels) {
    Batch b;
    b.pix0 = pix0; b.npix = npix; b.s0 = s0; b.ns = ns;
    b.width = width; b.height = height;
    b.npix_magic = div_magic_number(npix);
    b.width_magic = div_magic_number(width);
    b.pixels = pixels;
    return b;
}

// Opens the device work of a call of `paths` paths in all: the batch cap and path state (prepare_batches), the ray tally
// zeroed and ev_begin recorded.  finish_call closes it.
static int begin_call(CallFrame& f, size_t paths) {
    const int rc = prepare_batches(f.sc, paths, &f.cap);
    if (rc != FW_OK) return rc;
    FW_CUDA(cudaMemsetAsync(f.sc->ctx->d_rays, 0, sizeof(unsigned long long), f.st));
    FW_CUDA(cudaEventRecord(f.sc->ctx->ev_begin, f.st));
    return FW_OK;
}

// Samples [s_begin, s_begin + s_count) of `npix` pixels — the image's pixels 0 .. npix-1, or the first npix entries of a pixel
// list — in batches of at most f.cap paths: pixel tiles outer, sample chunks inner, so every pixel's samples are accumulated
// in sample order.  body(batch, first) runs each batch; `first`: the batch starts at sample s_begin.
template <class Body>
static int for_each_batch(const CallFrame& f, size_t npix, const uint32_t* pixels, uint32_t s_begin, uint32_t s_count, Body&& body) {
    const size_t tile = std::min(npix, f.cap);
    for (size_t pix0 = 0; pix0 < npix; pix0 += tile) {
        const size_t np = std::min(tile, npix - pix0);
        const uint32_t chunk = (uint32_t)std::max<size_t>(1, f.cap / np);
        for (uint32_t s = 0; s < s_count; s += chunk) {
            const Batch b = make_batch((uint32_t)pix0, (uint32_t)np, s_begin + s, std::min(chunk, s_count - s), f.p->width, f.p->height, pixels);
            const int rc = body(b, s == 0);
            if (rc != FW_OK) return rc;
        }
    }
    return FW_OK;
}

// run_batch over every batch of those samples.
static int run_tiles(CallFrame& f, size_t npix, const uint32_t* pixels, uint32_t s_begin, uint32_t s_count, float* d_sum,
                     const AdaptiveState* adapt) {
    return for_each_batch(f, npix, pixels, s_begin, s_count, [&](const Batch& b, bool) { return run_batch(f, b, d_sum, adapt); });
}

// The AOV pass (DESIGN.md §12) over samples [s_begin, s_begin + s_count) of every pixel, with the render's batching: raygen and
// the bounce-0 extend of each batch, its records collected and added in sample order.  Leaves the means in ctx->aov (and,
// when `planar` is set, the planar albedo / normal / depth there).
static int aov_pass(CallFrame& f, uint32_t s_begin, uint32_t s_count, float* planar) {
    fw_scene* sc = f.sc;
    RenderCtx* c = sc->ctx;
    PathState& ps = c->ps;
    const cudaStream_t st = f.st;
    const size_t npix = (size_t)f.p->width * f.p->height;
    const unsigned grid = grid_for(npix, 256, sc->sm_count * 8);
    FW_CUDA(cudaMemsetAsync(c->aov.nz, 0, npix * sizeof(float4), st));
    FW_CUDA(cudaMemsetAsync(c->aov.alb, 0, npix * sizeof(float4), st));
    const int rc = for_each_batch(f, npix, nullptr, s_begin, s_count, [&](const Batch& b, bool first) {
        int rc = begin_batch(sc, (size_t)b.npix * b.ns, st);
        if (rc != FW_OK) return rc;
        launch_raygen(f.cam, b, f.seed, ps, st);
        if ((rc = extend_bounce(sc, f.p->use_bvh != 0, b, f.seed, 0, st, f.launches)) != FW_OK) return rc;
        f.extend_launches++;
        launch_aov_collect(sc->dscene, ps, st);
        launch_aov_accumulate(c->aov, ps, b, first, grid_for(b.npix, 256, sc->sm_count * 8), st);
        launch_tally(ps, c->d_rays, st);
        f.launches += 4;
        return sync_stage(st, "AOV pass", 0);
    });
    if (rc != FW_OK) return rc;
    launch_aov_finalize(c->aov, (uint32_t)npix, (float)s_count, planar, grid, st);
    f.launches++;
    FW_CUDA(cudaGetLastError());
    return FW_OK;
}

// The a-trous iterations over ctx->dn_cv[0] with the guides in ctx->aov; returns the index of the buffer holding the result.
static int denoise_iterations(const fw_denoise* dn, uint32_t width, uint32_t height, float4* cv[2], const AovState& g, cudaStream_t st,
                              uint64_t* launches) {
    const DenoiseSigmas sg{dn->sigma_luminance, dn->sigma_depth, dn->sigma_albedo};
    int cur = 0;
    for (uint32_t it = 0; it < dn->iterations; ++it, cur ^= 1) launch_atrous(cv[cur], g.nz, g.alb, width, height, it, sg, cv[cur ^ 1], st);
    if (launches) *launches += dn->iterations;
    return cur;
}

static bool denoise_settings_ok(const fw_denoise* dn) {
    auto pos = [](float v) { return std::isfinite(v) && v > 0.0f; };
    if (dn->iterations < 1 || dn->iterations > 10) return set_error(FW_ERR_ARG, "iterations must be in 1..10"), false;
    if (dn->aov_samples < 1) return set_error(FW_ERR_ARG, "aov_samples must be >= 1"), false;
    if (!pos(dn->sigma_luminance) || !pos(dn->sigma_depth) || !pos(dn->sigma_albedo))
        return set_error(FW_ERR_ARG, "sigma_luminance, sigma_depth and sigma_albedo must be finite and > 0"), false;
    return true;
}

// Closes the device work of a call opened by begin_call: ray tally, event times -> stats.  Synchronises the call's stream.
static int finish_call(CallFrame& f, uint64_t samples, fw_stats* stats) {
    RenderCtx* c = f.sc->ctx;
    FW_CUDA(cudaEventRecord(c->ev_end, f.st));
    FW_CUDA(cudaMemcpyAsync(c->h_rays, c->d_rays, sizeof(unsigned long long), cudaMemcpyDeviceToHost, f.st));
    FW_CUDA(cudaStreamSynchronize(f.st));
    if (stats) {
        memset(stats, 0, sizeof(*stats));
        stats->samples = samples;
        stats->rays = *c->h_rays;
        stats->launches = f.launches;
        stats->extend_launches = f.extend_launches;
        float ms = 0;
        FW_CUDA(cudaEventElapsedTime(&ms, c->ev_begin, c->ev_end));
        stats->ms_device = ms;
        double me = 0;
        for (auto& pr : f.extend_events) {
            float m = 0;
            FW_CUDA(cudaEventElapsedTime(&m, pr.first, pr.second));
            me += m;
        }
        stats->ms_extend = me;
    }
    return FW_OK;
}

// Width, height and samples non-zero and fewer than 2^31 pixels: the image checks of every render entry point.
static int check_image(const fw_params* p) {
    if (!p || p->width == 0 || p->height == 0 || p->samples == 0) return set_error(FW_ERR_ARG, "width, height and samples must be non-zero");
    if ((uint64_t)p->width * p->height > 0x7fffffffull) return set_error(FW_ERR_ARG, "image too large");
    return FW_OK;
}

// d_sum and the luminance moments and sample counts of `npix` pixels zeroed: the start of an adaptive or denoised render.
static int zero_moments(RenderCtx* c, size_t npix, cudaStream_t st) {
    FW_CUDA(cudaMemsetAsync(c->d_sum, 0, npix * 3 * sizeof(float), st));
    FW_CUDA(cudaMemsetAsync(c->adapt.m1, 0, npix * sizeof(double), st));
    FW_CUDA(cudaMemsetAsync(c->adapt.m2, 0, npix * sizeof(double), st));
    FW_CUDA(cudaMemsetAsync(c->adapt.count, 0, npix * sizeof(uint32_t), st));
    return FW_OK;
}

int fw::render_into(fw_scene* sc, const fw_params* p, float* d_sum, cudaStream_t st, fw_stats* stats) {
    if (!sc->committed) return set_error(FW_ERR_STATE, "fw_scene_commit must be called before rendering");
    int rc = check_image(p);
    if (rc != FW_OK) return rc;
    FW_CUDA(cudaSetDevice(sc->device));
    const size_t npix = (size_t)p->width * p->height;
    CallFrame f(sc, p, st);
    if ((rc = begin_call(f, npix * std::max<uint32_t>(p->sample_count, 1))) != FW_OK ||
        (rc = run_tiles(f, npix, nullptr, p->sample_begin, p->sample_count, d_sum, nullptr)) != FW_OK)
        return rc;
    return finish_call(f, (uint64_t)npix * p->sample_count, stats);
}

int fw::ensure_sum_buffers(fw_scene* sc, size_t npix) {
    RenderCtx* c = sc->ctx;
    if (c->d_sum_pix >= npix) return FW_OK;
    free_sums(c);
    FW_CUDA(cudaMalloc(&c->d_sum, npix * 3 * sizeof(float)));
    FW_CUDA(cudaMalloc(&c->d_rgb, npix * 3));
    c->d_sum_pix = npix;
    return FW_OK;
}
int fw::ensure_adaptive_buffers(fw_scene* sc, size_t npix) {
    RenderCtx* c = sc->ctx;
    if (c->adapt_pix >= npix) return FW_OK;
    AdaptiveState& a = c->adapt;
    free_adaptive(c);
    FW_CUDA(cudaMalloc(&a.m1, npix * sizeof(double)));
    FW_CUDA(cudaMalloc(&a.m2, npix * sizeof(double)));
    FW_CUDA(cudaMalloc(&a.count, npix * sizeof(uint32_t)));
    FW_CUDA(cudaMalloc(&a.err, npix * sizeof(float)));
    FW_CUDA(cudaMalloc(&a.list[0], npix * sizeof(uint32_t)));
    FW_CUDA(cudaMalloc(&a.list[1], npix * sizeof(uint32_t)));
    FW_CUDA(cudaMalloc(&a.keep, npix));
    FW_CUDA(cudaMalloc(&a.block_base, ((size_t)adaptive_blocks((uint32_t)npix) + 1) * sizeof(uint32_t)));
    c->adapt_pix = npix;
    return FW_OK;
}
int fw::ensure_denoise_buffers(fw_scene* sc, size_t npix) {
    RenderCtx* c = sc->ctx;
    if (c->dn_pix >= npix) return FW_OK;
    free_denoise(c);
    FW_CUDA(cudaMalloc(&c->aov.nz, npix * sizeof(float4)));
    FW_CUDA(cudaMalloc(&c->aov.alb, npix * sizeof(float4)));
    FW_CUDA(cudaMalloc(&c->aov.obj, npix * sizeof(int)));
    FW_CUDA(cudaMalloc(&c->dn_cv[0], npix * sizeof(float4)));
    FW_CUDA(cudaMalloc(&c->dn_cv[1], npix * sizeof(float4)));
    FW_CUDA(cudaMalloc(&c->dn_planar, npix * 7 * sizeof(float)));
    FW_CUDA(cudaMalloc(&c->dn_var, npix * sizeof(float)));
    FW_CUDA(cudaMalloc(&c->dn_color, npix * 3 * sizeof(float)));
    c->dn_pix = npix;
    return FW_OK;
}

extern "C" {

// render.rs:184-189 + util.rs:14-23 for a host sum buffer (checkpoint resume, any caller that accumulated sums itself)
int fw_resolve_host(int device, const float* sum, uint32_t npix, uint32_t samples, float gamma, uint8_t* rgb_out) {
    if (!sum || !rgb_out || npix == 0 || samples == 0) return set_error(FW_ERR_ARG, "bad argument");
    int ndev = 0;
    FW_CUDA(cudaGetDeviceCount(&ndev));
    if (device < 0 || device >= ndev) return set_error(FW_ERR_CUDA, "no such CUDA device " + std::to_string(device));
    FW_CUDA(cudaSetDevice(device));
    DevBuf s, o;
    int rc;
    if ((rc = s.put(sum, (size_t)npix * 12)) != FW_OK || (rc = o.alloc((size_t)npix * 3)) != FW_OK) return rc;
    launch_resolve(s.as<float>(), npix, (float)samples, gamma, o.as<unsigned char>(), grid_for(npix, 256, 148 * 8), nullptr);
    FW_CUDA(cudaGetLastError());
    FW_CUDA(cudaDeviceSynchronize());
    return o.get(rgb_out, (size_t)npix * 3);
}

int fw_render_accumulate_device(fw_scene* sc, const fw_params* p, float* d_sum, void* cuda_stream, fw_stats* stats) {
    if (!sc || !d_sum) return set_error(FW_ERR_ARG, "null argument");
    if (!sc->committed || !sc->ctx) return set_error(FW_ERR_STATE, "fw_scene_commit must be called before rendering");
    cudaStream_t st = cuda_stream ? (cudaStream_t)cuda_stream : sc->ctx->stream;
    return render_into(sc, p, d_sum, st, stats);
}

int fw_resolve_device(fw_scene* sc, const float* d_sum, uint32_t npix, uint32_t samples, float gamma, uint8_t* d_rgb,
                      void* cuda_stream) {
    if (!sc || !d_sum || !d_rgb || samples == 0) return set_error(FW_ERR_ARG, "bad argument");
    if (!sc->committed) return set_error(FW_ERR_STATE, "scene not committed");
    FW_CUDA(cudaSetDevice(sc->device));
    cudaStream_t st = cuda_stream ? (cudaStream_t)cuda_stream : sc->ctx->stream;
    launch_resolve(d_sum, npix, (float)samples, gamma, d_rgb, grid_for(npix, 256, sc->sm_count * 8), st);
    FW_CUDA(cudaGetLastError());
    return FW_OK;
}

int fw_render(fw_scene* sc, const fw_params* p, uint8_t* rgb_out, float* sum_out, fw_stats* stats) {
    return guarded([&]() -> int {
        if (!sc || !p) return set_error(FW_ERR_ARG, "null argument");
        if (!sc->committed) return set_error(FW_ERR_STATE, "fw_scene_commit must be called before rendering");
        FW_CUDA(cudaSetDevice(sc->device));
        size_t npix = (size_t)p->width * p->height;
        if (npix == 0) return set_error(FW_ERR_ARG, "empty image");
        int brc = ensure_sum_buffers(sc, npix);
        if (brc != FW_OK) return brc;
        FW_CUDA(cudaMemsetAsync(sc->ctx->d_sum, 0, npix * 3 * sizeof(float), sc->ctx->stream));
        int rc = render_into(sc, p, sc->ctx->d_sum, sc->ctx->stream, stats);
        if (rc != FW_OK) return rc;
        if (rgb_out) {
            launch_resolve(sc->ctx->d_sum, (uint32_t)npix, (float)p->samples, p->gamma, sc->ctx->d_rgb, grid_for(npix, 256, sc->sm_count * 8), sc->ctx->stream);
            FW_CUDA(cudaGetLastError());
            if (stats) stats->launches++;
            FW_CUDA(cudaMemcpyAsync(rgb_out, sc->ctx->d_rgb, npix * 3, cudaMemcpyDeviceToHost, sc->ctx->stream));
        }
        if (sum_out) FW_CUDA(cudaMemcpyAsync(sum_out, sc->ctx->d_sum, npix * 3 * sizeof(float), cudaMemcpyDeviceToHost, sc->ctx->stream));
        FW_CUDA(cudaStreamSynchronize(sc->ctx->stream));
        return FW_OK;
});
}

// Adaptive sampling (DESIGN.md §11).  Round 0 renders samples [0, n0) of every pixel; after round r the pixels whose relative
// error is not yet <= threshold render [n_r, min(2 n_r, cap)) in round r + 1.  Each round is the ordinary batch loop over the
// active pixel list, so a pixel with k samples holds the sums of fw_render at samples = k.
int fw_render_adaptive(fw_scene* sc, const fw_params* p, const fw_adaptive* ad, uint8_t* rgb_out, float* sum_out, uint32_t* count_out,
                       float* error_out, fw_stats* stats, fw_adaptive_result* result) {
    return guarded([&]() -> int {
        // every argument check comes before the first CUDA call
        if (!sc || !p || !ad) return set_error(FW_ERR_ARG, "null argument");
        int rc = check_image(p);
        if (rc != FW_OK) return rc;
        if (p->sample_begin != 0 || p->sample_count != p->samples)
            return set_error(FW_ERR_ARG, "an adaptive render owns the sample range: sample_begin must be 0 and sample_count == samples (the cap)");
        if (ad->min_samples == 0) return set_error(FW_ERR_ARG, "min_samples must be >= 1");
        if (!(ad->threshold >= 0.0f) || !std::isfinite(ad->threshold)) return set_error(FW_ERR_ARG, "threshold must be finite and >= 0");
        if (!(ad->floor > 0.0f) || !std::isfinite(ad->floor)) return set_error(FW_ERR_ARG, "floor must be finite and > 0");
        if (!sc->committed || !sc->ctx) return set_error(FW_ERR_STATE, "fw_scene_commit must be called before rendering");
        FW_CUDA(cudaSetDevice(sc->device));
        const size_t npix = (size_t)p->width * p->height;
        RenderCtx* c = sc->ctx;
        const AdaptiveState& A = c->adapt;
        CallFrame f(sc, p, c->stream);
        const cudaStream_t st = f.st;
        if ((rc = ensure_sum_buffers(sc, npix)) != FW_OK || (rc = ensure_adaptive_buffers(sc, npix)) != FW_OK ||
            (rc = zero_moments(c, npix, st)) != FW_OK || (rc = begin_call(f, npix * p->samples)) != FW_OK)
            return rc;
        const unsigned grid = grid_for(npix, 256, sc->sm_count * 8);
        const double threshold = ad->threshold, floor = ad->floor;
        launch_adaptive_init(A.list[0], (uint32_t)npix, grid, st);
        f.launches++;
        fw_adaptive_result res;
        memset(&res, 0, sizeof(res));
        uint32_t active = (uint32_t)npix, n_prev = 0, n = std::min(ad->min_samples, p->samples);
        int cur = 0;
        for (;;) {
            if ((rc = run_tiles(f, active, A.list[cur], n_prev, n - n_prev, c->d_sum, &A)) != FW_OK) return rc;
            if (res.rounds < 32) res.active[res.rounds] = active;
            res.rounds++;
            res.samples += (uint64_t)active * (n - n_prev);
            if (n == p->samples) break;   // the cap: nothing left to decide
            f.launches += launch_converge_compact(A, A.list[cur], active, threshold, floor, A.list[cur ^ 1], st);
            FW_CUDA(cudaGetLastError());
            FW_CUDA(cudaMemcpyAsync(&active, A.block_base + adaptive_blocks(active), sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
            FW_CUDA(cudaStreamSynchronize(st));
            cur ^= 1;
            if (active == 0) break;
            n_prev = n;
            n = n > p->samples / 2 ? p->samples : 2 * n;
        }
        launch_resolve_adaptive(c->d_sum, A, (uint32_t)npix, p->gamma, floor, c->d_rgb, grid, st);
        FW_CUDA(cudaGetLastError());
        f.launches++;
        if ((rc = finish_call(f, res.samples, stats)) != FW_OK) return rc;
        if (rgb_out) FW_CUDA(cudaMemcpyAsync(rgb_out, c->d_rgb, npix * 3, cudaMemcpyDeviceToHost, st));
        if (sum_out) FW_CUDA(cudaMemcpyAsync(sum_out, c->d_sum, npix * 3 * sizeof(float), cudaMemcpyDeviceToHost, st));
        if (count_out) FW_CUDA(cudaMemcpyAsync(count_out, A.count, npix * sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
        if (error_out) FW_CUDA(cudaMemcpyAsync(error_out, A.err, npix * sizeof(float), cudaMemcpyDeviceToHost, st));
        FW_CUDA(cudaStreamSynchronize(st));
        if (result) *result = res;
        return FW_OK;
});
}

// ---- denoised renders (DESIGN.md §12) --------------------------------------------------------------------
static int copy_aov_out(RenderCtx* c, size_t npix, const fw_aov* aov, cudaStream_t st) {
    if (!aov) return FW_OK;
    if (aov->albedo) FW_CUDA(cudaMemcpyAsync(aov->albedo, c->dn_planar, npix * 3 * sizeof(float), cudaMemcpyDeviceToHost, st));
    if (aov->normal) FW_CUDA(cudaMemcpyAsync(aov->normal, c->dn_planar + 3 * npix, npix * 3 * sizeof(float), cudaMemcpyDeviceToHost, st));
    if (aov->depth) FW_CUDA(cudaMemcpyAsync(aov->depth, c->dn_planar + 6 * npix, npix * sizeof(float), cudaMemcpyDeviceToHost, st));
    if (aov->object) FW_CUDA(cudaMemcpyAsync(aov->object, c->aov.obj, npix * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
    return FW_OK;
}

int fw_render_aov(fw_scene* sc, const fw_params* p, const fw_aov* aov, fw_stats* stats) {
    return guarded([&]() -> int {
        // every argument check comes before the first CUDA call
        if (!sc || !p || !aov) return set_error(FW_ERR_ARG, "null argument");
        int rc = check_image(p);
        if (rc != FW_OK) return rc;
        if (p->sample_count == 0) return set_error(FW_ERR_ARG, "sample_count must be >= 1");
        if (!sc->committed || !sc->ctx) return set_error(FW_ERR_STATE, "fw_scene_commit must be called before rendering");
        FW_CUDA(cudaSetDevice(sc->device));
        const size_t npix = (size_t)p->width * p->height;
        RenderCtx* c = sc->ctx;
        CallFrame f(sc, p, c->stream);
        if ((rc = ensure_denoise_buffers(sc, npix)) != FW_OK || (rc = begin_call(f, npix * p->sample_count)) != FW_OK ||
            (rc = aov_pass(f, p->sample_begin, p->sample_count, c->dn_planar)) != FW_OK)
            return rc;
        if ((rc = finish_call(f, (uint64_t)npix * p->sample_count, stats)) != FW_OK || (rc = copy_aov_out(c, npix, aov, f.st)) != FW_OK)
            return rc;
        FW_CUDA(cudaStreamSynchronize(f.st));
        return FW_OK;
});
}

int fw_denoise_host(int device, uint32_t width, uint32_t height, const float* color, const float* variance, const float* albedo,
                    const float* normal, const float* depth, const fw_denoise* dn, float* color_out, float* variance_out) {
    return guarded([&]() -> int {
        if (!color || !variance || !albedo || !normal || !depth || !dn || !color_out) return set_error(FW_ERR_ARG, "null argument");
        if (width == 0 || height == 0) return set_error(FW_ERR_ARG, "width and height must be non-zero");
        if ((uint64_t)width * height > 0x7fffffffull) return set_error(FW_ERR_ARG, "image too large");
        if (!denoise_settings_ok(dn)) return FW_ERR_ARG;
        int ndev = 0;
        FW_CUDA(cudaGetDeviceCount(&ndev));
        if (device < 0 || device >= ndev) return set_error(FW_ERR_CUDA, "no such CUDA device " + std::to_string(device));
        FW_CUDA(cudaSetDevice(device));
        const size_t npix = (size_t)width * height;
        DevBuf dc, dv, da, dnrm, dd, cv0, cv1, nz, alb, oc, ov;
        int rc;
        if ((rc = dc.put(color, npix * 12)) != FW_OK || (rc = dv.put(variance, npix * 4)) != FW_OK || (rc = da.put(albedo, npix * 12)) != FW_OK ||
            (rc = dnrm.put(normal, npix * 12)) != FW_OK || (rc = dd.put(depth, npix * 4)) != FW_OK || (rc = cv0.alloc(npix * 16)) != FW_OK ||
            (rc = cv1.alloc(npix * 16)) != FW_OK || (rc = nz.alloc(npix * 16)) != FW_OK || (rc = alb.alloc(npix * 16)) != FW_OK ||
            (rc = oc.alloc(npix * 12)) != FW_OK || (rc = ov.alloc(npix * 4)) != FW_OK)
            return rc;
        const unsigned grid = grid_for(npix, 256, 148 * 8);
        launch_denoise_pack(dc.as<float>(), dv.as<float>(), da.as<float>(), dnrm.as<float>(), dd.as<float>(), (uint32_t)npix, cv0.as<float4>(),
                            nz.as<float4>(), alb.as<float4>(), grid, nullptr);
        float4* cv[2] = {cv0.as<float4>(), cv1.as<float4>()};
        AovState g;
        g.nz = nz.as<float4>(); g.alb = alb.as<float4>();
        const int cur = denoise_iterations(dn, width, height, cv, g, nullptr, nullptr);
        launch_denoise_unpack(cv[cur], (uint32_t)npix, oc.as<float>(), ov.as<float>(), grid, nullptr);
        FW_CUDA(cudaGetLastError());
        FW_CUDA(cudaDeviceSynchronize());
        if ((rc = oc.get(color_out, npix * 12)) != FW_OK) return rc;
        if (variance_out) return ov.get(variance_out, npix * 4);
        return FW_OK;
});
}

int fw_render_denoised(fw_scene* sc, const fw_params* p, const fw_denoise* dn, uint8_t* rgb_out, float* sum_out, float* denoised_out,
                       float* variance_out, const fw_aov* aov, fw_stats* stats) {
    return guarded([&]() -> int {
        // every argument check comes before the first CUDA call
        if (!sc || !p || !dn) return set_error(FW_ERR_ARG, "null argument");
        int rc = check_image(p);
        if (rc != FW_OK) return rc;
        if (p->sample_begin != 0 || p->sample_count != p->samples || p->samples < 2)
            return set_error(FW_ERR_ARG, "a denoised render owns the sample range: sample_begin must be 0, sample_count == samples and samples >= 2");
        if (!denoise_settings_ok(dn)) return FW_ERR_ARG;
        if (!sc->committed || !sc->ctx) return set_error(FW_ERR_STATE, "fw_scene_commit must be called before rendering");
        FW_CUDA(cudaSetDevice(sc->device));
        const size_t npix = (size_t)p->width * p->height;
        RenderCtx* c = sc->ctx;
        CallFrame f(sc, p, c->stream);
        const cudaStream_t st = f.st;
        if ((rc = ensure_sum_buffers(sc, npix)) != FW_OK || (rc = ensure_adaptive_buffers(sc, npix)) != FW_OK ||
            (rc = ensure_denoise_buffers(sc, npix)) != FW_OK || (rc = zero_moments(c, npix, st)) != FW_OK ||
            (rc = begin_call(f, npix * p->samples)) != FW_OK)
            return rc;
        if ((rc = run_tiles(f, npix, nullptr, 0, p->samples, c->d_sum, &c->adapt)) != FW_OK ||
            (rc = aov_pass(f, 0, std::min(dn->aov_samples, p->samples), c->dn_planar)) != FW_OK)
            return rc;
        const unsigned grid = grid_for(npix, 256, sc->sm_count * 8);
        launch_denoise_input(c->d_sum, c->adapt, (uint32_t)npix, p->samples, c->dn_cv[0], c->dn_var, grid, st);
        f.launches++;
        const int cur = denoise_iterations(dn, p->width, p->height, c->dn_cv, c->aov, st, &f.launches);
        launch_denoise_unpack(c->dn_cv[cur], (uint32_t)npix, c->dn_color, nullptr, grid, st);
        launch_resolve(c->dn_color, (uint32_t)npix, 1.0f, p->gamma, c->d_rgb, grid, st);
        f.launches += 2;
        FW_CUDA(cudaGetLastError());
        if ((rc = finish_call(f, (uint64_t)npix * p->samples, stats)) != FW_OK) return rc;
        if (rgb_out) FW_CUDA(cudaMemcpyAsync(rgb_out, c->d_rgb, npix * 3, cudaMemcpyDeviceToHost, st));
        if (sum_out) FW_CUDA(cudaMemcpyAsync(sum_out, c->d_sum, npix * 3 * sizeof(float), cudaMemcpyDeviceToHost, st));
        if (denoised_out) FW_CUDA(cudaMemcpyAsync(denoised_out, c->dn_color, npix * 3 * sizeof(float), cudaMemcpyDeviceToHost, st));
        if (variance_out) FW_CUDA(cudaMemcpyAsync(variance_out, c->dn_var, npix * sizeof(float), cudaMemcpyDeviceToHost, st));
        if ((rc = copy_aov_out(c, npix, aov, st)) != FW_OK) return rc;
        FW_CUDA(cudaStreamSynchronize(st));
        return FW_OK;
});
}

// ---- caller-supplied rays (DESIGN.md §13) ----------------------------------------------------------------
// The argument checks of both trace entry points; none of them makes a CUDA call.
static int check_trace(const fw_scene* sc, uint64_t n, const float* origins, const float* dirs, uint32_t sample_begin,
                       uint32_t sample_count, const float* sum) {
    if (!sc || !origins || !dirs || !sum) return set_error(FW_ERR_ARG, "null argument");
    if (n == 0 || n > 0x7fffffffull) return set_error(FW_ERR_ARG, "the number of rays must be in 1 .. 2^31 - 1");
    if (sample_count == 0) return set_error(FW_ERR_ARG, "sample_count must be >= 1");
    if ((uint64_t)sample_begin + sample_count > 0x100000000ull) return set_error(FW_ERR_ARG, "sample_begin + sample_count must be <= 2^32");
    if (!sc->committed || !sc->ctx) return set_error(FW_ERR_STATE, "fw_scene_commit must be called before tracing");
    return FW_OK;
}

// Adds samples [rs.sample_begin, rs.sample_begin + sample_count) of every ray of `rs`, ray i keyed as pixel d_keys[i] (or i when
// d_keys is null), into d_sum[3i .. 3i+2] on `st`: the render's batch loop with the rays as a one-row image of rs.n pixels.
static int trace_into(fw_scene* sc, const RaySource& rs, const uint32_t* d_keys, uint32_t sample_count, uint64_t seed, int use_bvh,
                      float* d_sum, cudaStream_t st, fw_stats* stats) {
    fw_params p;
    memset(&p, 0, sizeof(p));
    p.width = rs.n; p.height = 1;
    p.samples = p.sample_count = sample_count; p.sample_begin = rs.sample_begin;
    p.use_bvh = use_bvh != 0;
    p.seed = seed;
    CallFrame f(sc, &p, st, &rs);
    int rc;
    if ((rc = begin_call(f, (size_t)rs.n * sample_count)) != FW_OK ||
        (rc = run_tiles(f, rs.n, d_keys, rs.sample_begin, sample_count, d_sum, nullptr)) != FW_OK)
        return rc;
    return finish_call(f, (uint64_t)rs.n * sample_count, stats);
}

int fw_trace_rays(fw_scene* sc, uint64_t n, const float* origins, const float* dirs, const uint32_t* keys, int per_sample,
                  uint32_t sample_begin, uint32_t sample_count, uint64_t seed, int use_bvh, float* sum_out, fw_stats* stats) {
    return guarded([&]() -> int {
        int rc = check_trace(sc, n, origins, dirs, sample_begin, sample_count, sum_out);
        if (rc != FW_OK) return rc;
        FW_CUDA(cudaSetDevice(sc->device));
        RenderCtx* c = sc->ctx;
        const cudaStream_t st = c->stream;
        const size_t ray_bytes = (size_t)n * (per_sample ? sample_count : 1) * 12;
        DevBuf dO, dD, dK;
        if ((rc = dO.alloc(ray_bytes)) != FW_OK || (rc = dD.alloc(ray_bytes)) != FW_OK || (keys && (rc = dK.alloc(n * 4)) != FW_OK) ||
            (rc = ensure_sum_buffers(sc, n)) != FW_OK)
            return rc;
        FW_CUDA(cudaMemcpyAsync(dO.p, origins, ray_bytes, cudaMemcpyHostToDevice, st));
        FW_CUDA(cudaMemcpyAsync(dD.p, dirs, ray_bytes, cudaMemcpyHostToDevice, st));
        if (keys) FW_CUDA(cudaMemcpyAsync(dK.p, keys, n * 4, cudaMemcpyHostToDevice, st));
        FW_CUDA(cudaMemsetAsync(c->d_sum, 0, n * 3 * sizeof(float), st));
        const RaySource rs{dO.as<float>(), dD.as<float>(), (uint32_t)n, sample_begin, per_sample != 0};
        if ((rc = trace_into(sc, rs, keys ? dK.as<uint32_t>() : nullptr, sample_count, seed, use_bvh, c->d_sum, st, stats)) != FW_OK) return rc;
        FW_CUDA(cudaMemcpyAsync(sum_out, c->d_sum, n * 3 * sizeof(float), cudaMemcpyDeviceToHost, st));
        FW_CUDA(cudaStreamSynchronize(st));
        return FW_OK;
});
}

int fw_trace_rays_device(fw_scene* sc, uint64_t n, const float* d_origins, const float* d_dirs, const uint32_t* d_keys, int per_sample,
                         uint32_t sample_begin, uint32_t sample_count, uint64_t seed, int use_bvh, float* d_sum, void* cuda_stream,
                         fw_stats* stats) {
    return guarded([&]() -> int {
        int rc = check_trace(sc, n, d_origins, d_dirs, sample_begin, sample_count, d_sum);
        if (rc != FW_OK) return rc;
        FW_CUDA(cudaSetDevice(sc->device));
        const RaySource rs{d_origins, d_dirs, (uint32_t)n, sample_begin, per_sample != 0};
        return trace_into(sc, rs, d_keys, sample_count, seed, use_bvh, d_sum, cuda_stream ? (cudaStream_t)cuda_stream : sc->ctx->stream, stats);
});
}

// ---- probes ---------------------------------------------------------------------------------------------
#define TRY(x) do { int rc__ = (x); if (rc__ != FW_OK) return rc__; } while (0)

int fw_primary_rays(fw_scene* sc, const fw_params* p, uint32_t sample, uint32_t pix_begin, uint32_t n, float* origins,
                    float* dirs) {
    if (!sc || !p || !origins || !dirs) return set_error(FW_ERR_ARG, "null argument");
    if (!sc->committed) return set_error(FW_ERR_STATE, "scene not committed");
    FW_CUDA(cudaSetDevice(sc->device));
    const CallFrame f(sc, p, sc->ctx->stream);   // the rays of a render call of `p`
    DevBuf o, d;
    TRY(o.alloc((size_t)n * 12)); TRY(d.alloc((size_t)n * 12));
    launch_primary_rays_probe(f.cam, p->width, p->height, sample, f.seed, pix_begin, n, o.as<float>(), d.as<float>(), grid_for(n, 256, 4096),
                              f.st);
    FW_CUDA(cudaGetLastError());
    FW_CUDA(cudaStreamSynchronize(sc->ctx->stream));
    TRY(o.get(origins, (size_t)n * 12)); TRY(d.get(dirs, (size_t)n * 12));
    return FW_OK;
}

int fw_first_hit(fw_scene* sc, int use_bvh, uint64_t seed, uint32_t n, const float* origins, const float* dirs,
                 const uint32_t* pixel, const uint32_t* sample, const uint32_t* bounce, int32_t* obj, int32_t* prim,
                 int32_t* material, float* t, float* point, float* normal, float* uv, uint64_t counters[2]) {
    if (!sc || !origins || !dirs || !obj || !prim || !material || !t || !point || !normal || !uv)
        return set_error(FW_ERR_ARG, "null argument");
    if (!sc->committed) return set_error(FW_ERR_STATE, "scene not committed");
    FW_CUDA(cudaSetDevice(sc->device));
    DevBuf dO, dD, dP, dS, dB, oC;
    FirstHitBufs hit;
    TRY(dO.put(origins, (size_t)n * 12)); TRY(dD.put(dirs, (size_t)n * 12));
    if (pixel) TRY(dP.put(pixel, (size_t)n * 4));
    if (sample) TRY(dS.put(sample, (size_t)n * 4));
    if (bounce) TRY(dB.put(bounce, (size_t)n * 4));
    TRY(hit.alloc(n)); TRY(oC.alloc(16));
    FW_CUDA(cudaMemset(oC.p, 0, 16));
    uint2 sd = make_uint2((uint32_t)seed, (uint32_t)(seed >> 32));
    unsigned g = grid_for(n, 128, 8192);
    int mode = use_bvh ? 1 : (sc->lin_prog_ok ? (sc->flat.lin_generic ? 2 : 3) : 0);
    launch_first_hit_probe(mode, sc->lin_prog, sc->dscene, sd, n, dO.as<float>(), dD.as<float>(), pixel ? dP.as<uint32_t>() : nullptr,
                           sample ? dS.as<uint32_t>() : nullptr, bounce ? dB.as<uint32_t>() : nullptr, hit.out(oC.as<unsigned long long>()), g,
                           sc->ctx->stream);
    FW_CUDA(cudaGetLastError());
    FW_CUDA(cudaStreamSynchronize(sc->ctx->stream));
    TRY(hit.get(n, obj, prim, material, t, point, normal, uv));
    if (counters) TRY(oC.get(counters, 16));
    return FW_OK;
}

// The same query through the kernels a render launches (queues, segments, the scene's extend plan, finalize_hit).
int fw_first_hit_wavefront(fw_scene* sc, int use_bvh, uint64_t seed, uint32_t n, const float* origins, const float* dirs,
                           uint32_t sample, uint32_t bounce, int32_t* obj, int32_t* prim, int32_t* material, float* t, float* point,
                           float* normal, float* uv) {
    if (!sc || !origins || !dirs || !obj || !prim || !material || !t || !point || !normal || !uv)
        return set_error(FW_ERR_ARG, "null argument");
    if (!sc->committed) return set_error(FW_ERR_STATE, "scene not committed");
    if (n == 0 || bounce > (uint32_t)FW_MAX_DEPTH) return set_error(FW_ERR_ARG, "need n > 0 and bounce <= 10");
    FW_CUDA(cudaSetDevice(sc->device));
    int rc = ensure_path_state(sc, std::max<size_t>(n, 32));
    if (rc != FW_OK) return rc;
    DevBuf dO, dD;
    FirstHitBufs hit;
    TRY(dO.put(origins, (size_t)n * 12)); TRY(dD.put(dirs, (size_t)n * 12));
    TRY(hit.alloc(n));
    cudaStream_t st = sc->ctx->stream;
    const PathState& ps = sc->ctx->ps;
    TRY(begin_batch(sc, n, st));
    const Batch b = make_batch(0, n, sample, 1, n, 1, nullptr);   // ray i = path i = "pixel" i of a one-sample batch: RNG key (pixel i, sample, bounce)
    const uint2 sd = make_uint2((uint32_t)seed, (uint32_t)(seed >> 32));
    launch_probe_fill(ps, n, dO.as<float>(), dD.as<float>(), bounce, st);
    uint64_t launches = 0;
    TRY(extend_bounce(sc, use_bvh != 0, b, sd, bounce, st, launches));
    launch_probe_collect(sc->dscene, ps, bounce, hit.out(nullptr), st);
    FW_CUDA(cudaGetLastError());
    FW_CUDA(cudaStreamSynchronize(st));
    return hit.get(n, obj, prim, material, t, point, normal, uv);
}

// fw_scatter_step (uniforms != nullptr) and fw_scatter_step_keyed (pixel / sample / bounce keys) share everything else.
static int scatter_probe(fw_scene* sc, uint32_t n, const int32_t* material, const float* ray_o, const float* ray_d,
                         const float* hit_t, const float* hit_point, const float* hit_normal, const float* hit_uv,
                         const float* uniforms, uint32_t nu, uint64_t seed, const uint32_t* pixel, const uint32_t* sample,
                         const uint32_t* bounce, float* emit, int32_t* scattered, float* atten, float* out_o, float* out_d,
                         int32_t* consumed) {
    if (!sc || !material || !ray_o || !ray_d || !hit_t || !hit_point || !hit_normal || !hit_uv || !emit || !scattered ||
        !atten || !out_o || !out_d || !consumed || (!uniforms && (!pixel || !sample || !bounce)))
        return set_error(FW_ERR_ARG, "null argument");
    if (!sc->committed) return set_error(FW_ERR_STATE, "scene not committed");
    for (uint32_t i = 0; i < n; ++i)
        if (material[i] < 0 || material[i] >= (int)sc->desc.mats.size()) return set_error(FW_ERR_ARG, "material index out of range");
    FW_CUDA(cudaSetDevice(sc->device));
    DevBuf m, ro, rd, ht, hp, hn, hu, un, kp, ks, kb, e, s, a, oo, od, c;
    TRY(m.put(material, (size_t)n * 4)); TRY(ro.put(ray_o, (size_t)n * 12)); TRY(rd.put(ray_d, (size_t)n * 12));
    TRY(ht.put(hit_t, (size_t)n * 4)); TRY(hp.put(hit_point, (size_t)n * 12)); TRY(hn.put(hit_normal, (size_t)n * 12));
    TRY(hu.put(hit_uv, (size_t)n * 8));
    if (uniforms) {
        TRY(un.put(uniforms, (size_t)n * nu * 4));
    } else {
        TRY(kp.put(pixel, (size_t)n * 4)); TRY(ks.put(sample, (size_t)n * 4)); TRY(kb.put(bounce, (size_t)n * 4));
    }
    TRY(e.alloc((size_t)n * 12)); TRY(s.alloc((size_t)n * 4)); TRY(a.alloc((size_t)n * 12)); TRY(oo.alloc((size_t)n * 12));
    TRY(od.alloc((size_t)n * 12)); TRY(c.alloc((size_t)n * 4));
    ScatterProbeIO io{m.as<int>(), ro.as<float>(), rd.as<float>(), ht.as<float>(), hp.as<float>(), hn.as<float>(),
                      hu.as<float>(), uniforms ? un.as<float>() : nullptr, nu,
                      make_uint2((uint32_t)seed, (uint32_t)(seed >> 32)), kp.as<uint32_t>(), ks.as<uint32_t>(), kb.as<uint32_t>(),
                      e.as<float>(), s.as<int>(), a.as<float>(), oo.as<float>(), od.as<float>(), c.as<int>()};
    launch_scatter_step_probe(sc->dscene, n, io, grid_for(n, 128, 4096), sc->ctx->stream);
    FW_CUDA(cudaGetLastError());
    FW_CUDA(cudaStreamSynchronize(sc->ctx->stream));
    TRY(e.get(emit, (size_t)n * 12)); TRY(s.get(scattered, (size_t)n * 4)); TRY(a.get(atten, (size_t)n * 12));
    TRY(oo.get(out_o, (size_t)n * 12)); TRY(od.get(out_d, (size_t)n * 12)); TRY(c.get(consumed, (size_t)n * 4));
    return FW_OK;
}
int fw_scatter_step(fw_scene* sc, uint32_t n, const int32_t* material, const float* ray_o, const float* ray_d,
                    const float* hit_t, const float* hit_point, const float* hit_normal, const float* hit_uv,
                    const float* uniforms, uint32_t nu, float* emit, int32_t* scattered, float* atten, float* out_o,
                    float* out_d, int32_t* consumed) {
    if (!uniforms) return set_error(FW_ERR_ARG, "null argument");
    return scatter_probe(sc, n, material, ray_o, ray_d, hit_t, hit_point, hit_normal, hit_uv, uniforms, nu, 0, nullptr, nullptr,
                         nullptr, emit, scattered, atten, out_o, out_d, consumed);
}
int fw_scatter_step_keyed(fw_scene* sc, uint64_t seed, uint32_t n, const int32_t* material, const float* ray_o,
                          const float* ray_d, const float* hit_t, const float* hit_point, const float* hit_normal,
                          const float* hit_uv, const uint32_t* pixel, const uint32_t* sample, const uint32_t* bounce,
                          float* emit, int32_t* scattered, float* atten, float* out_o, float* out_d, int32_t* consumed) {
    return scatter_probe(sc, n, material, ray_o, ray_d, hit_t, hit_point, hit_normal, hit_uv, nullptr, 0, seed, pixel, sample,
                         bounce, emit, scattered, atten, out_o, out_d, consumed);
}

int fw_env_sample(fw_scene* sc, uint32_t n, const float* dirs, float* out) {
    if (!sc || !dirs || !out) return set_error(FW_ERR_ARG, "null argument");
    if (!sc->committed) return set_error(FW_ERR_STATE, "scene not committed");
    FW_CUDA(cudaSetDevice(sc->device));
    DevBuf d, o;
    TRY(d.put(dirs, (size_t)n * 12)); TRY(o.alloc((size_t)n * 12));
    launch_env_sample_probe(sc->dscene, n, d.as<float>(), o.as<float>(), grid_for(n, 256, 4096), sc->ctx->stream);
    FW_CUDA(cudaGetLastError());
    FW_CUDA(cudaStreamSynchronize(sc->ctx->stream));
    return o.get(out, (size_t)n * 12);
}
int fw_texture_sample(fw_scene* sc, int texture, uint32_t n, const float* uv, const float* point, float* out) {
    if (!sc || !uv || !point || !out) return set_error(FW_ERR_ARG, "null argument");
    if (!sc->committed) return set_error(FW_ERR_STATE, "scene not committed");
    if (texture < 0 || texture >= (int)sc->desc.texs.size()) return set_error(FW_ERR_ARG, "texture index out of range");
    FW_CUDA(cudaSetDevice(sc->device));
    DevBuf u, p, o;
    TRY(u.put(uv, (size_t)n * 8)); TRY(p.put(point, (size_t)n * 12)); TRY(o.alloc((size_t)n * 12));
    launch_texture_sample_probe(sc->dscene, texture, n, u.as<float>(), p.as<float>(), o.as<float>(), grid_for(n, 256, 4096), sc->ctx->stream);
    FW_CUDA(cudaGetLastError());
    FW_CUDA(cudaStreamSynchronize(sc->ctx->stream));
    return o.get(out, (size_t)n * 12);
}

int fw_selftest_shared_division(int device, uint64_t n_pairs, uint64_t seed, uint64_t violations[2]) {
    if (!violations) return set_error(FW_ERR_ARG, "null argument");
    int ndev = 0;
    FW_CUDA(cudaGetDeviceCount(&ndev));
    if (device < 0 || device >= ndev) return set_error(FW_ERR_CUDA, "no such CUDA device " + std::to_string(device));
    FW_CUDA(cudaSetDevice(device));
    DevBuf v;
    TRY(v.alloc(16));
    FW_CUDA(cudaMemset(v.p, 0, 16));
    launch_shared_division_probe(n_pairs, make_uint2((uint32_t)seed, (uint32_t)(seed >> 32)), v.as<unsigned long long>());
    FW_CUDA(cudaGetLastError());
    FW_CUDA(cudaDeviceSynchronize());
    return v.get(violations, 16);
}

// ---- roofline denominators ------------------------------------------------------------------------------
}  // extern "C"

extern "C" int fw_measure_peaks(int device, double* fp32_tflops, double* l2_gbs, int* sm_count, int* sm_clock_khz) {
    FW_CUDA(cudaSetDevice(device));
    cudaDeviceProp prop;
    FW_CUDA(cudaGetDeviceProperties(&prop, device));
    if (sm_count) *sm_count = prop.multiProcessorCount;
    int khz = 0;
    cudaDeviceGetAttribute(&khz, cudaDevAttrClockRate, device);
    if (sm_clock_khz) *sm_clock_khz = khz;
    cudaEvent_t e0, e1;
    FW_CUDA(cudaEventCreate(&e0));
    FW_CUDA(cudaEventCreate(&e1));
    float* out = nullptr;
    FW_CUDA(cudaMalloc(&out, 64));
    int blocks = prop.multiProcessorCount * 8, threads = 256, iters = 1 << 16;
    double best = 0;
    for (int rep = 0; rep < 4; ++rep) {
        FW_CUDA(cudaEventRecord(e0));
        launch_fp32_peak(out, iters, blocks, threads);
        FW_CUDA(cudaEventRecord(e1));
        FW_CUDA(cudaEventSynchronize(e1));
        float ms = 0;
        FW_CUDA(cudaEventElapsedTime(&ms, e0, e1));
        double flops = 2.0 * 8.0 * (double)iters * blocks * threads;
        if (rep > 0) best = std::max(best, flops / (ms * 1e-3) / 1e12);
    }
    if (fp32_tflops) *fp32_tflops = best;
    size_t bytes = (size_t)48 << 20;  // 48 MiB: resident in the 126 MB L2
    float4* buf = nullptr;
    FW_CUDA(cudaMalloc(&buf, bytes));
    FW_CUDA(cudaMemset(buf, 0, bytes));
    double bestbw = 0;
    int reps = 20;
    for (int rep = 0; rep < 4; ++rep) {
        FW_CUDA(cudaEventRecord(e0));
        launch_l2_read(buf, bytes / 16, reps, out, prop.multiProcessorCount * 8, 512);
        FW_CUDA(cudaEventRecord(e1));
        FW_CUDA(cudaEventSynchronize(e1));
        float ms = 0;
        FW_CUDA(cudaEventElapsedTime(&ms, e0, e1));
        if (rep > 0) bestbw = std::max(bestbw, (double)bytes * reps / (ms * 1e-3) / 1e9);
    }
    if (l2_gbs) *l2_gbs = bestbw;
    cudaFree(buf);
    cudaFree(out);
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    return FW_OK;
}
