// Internals shared by api.cu and multi_gpu.cu: the scene handle, the cached per-device render context, error plumbing.
#pragma once
#include <cuda_runtime.h>

#include <mutex>
#include <string>
#include <vector>

#include "../../include/firework_b200.h"
#include "launch.h"
#include "scene_host.h"

namespace fw {
int set_error(int code, const std::string& msg);   // records the thread's fw_last_error() text, returns `code`
}
using namespace fw;   // internal header: the structs below are global (fw_scene is the C ABI's opaque handle)
#define FW_CUDA(call)                                                                                         \
    do {                                                                                                      \
        cudaError_t e__ = (call);                                                                             \
        if (e__ != cudaSuccess)                                                                               \
            return fw::set_error(FW_ERR_CUDA, std::string(#call) + ": " + cudaGetErrorString(e__) + " (" __FILE__ \
                                              ":" + std::to_string(__LINE__) + ")");                          \
    } while (0)

// Pinned staging for equirect HDR maps (see api.cu).
struct HdrStaging {
    float* p = nullptr;
    size_t floats = 0;
    bool in_use = false;
    bool plain = false;   // malloc'ed fallback (no pinned memory): freed on release instead of pooled
};

// Render-time device state (path-state streams, sum / image buffers, stream, events).  It is independent of the
// scene, ~1.2 GB at the default batch size, and expensive to allocate, so contexts are cached per device and
// handed from one fw_scene to the next (fw_release_cached_memory frees them).
struct RenderCtx {
    int device = 0;
    bool in_use = false;
    PathState ps{};
    size_t ps_cap = 0;
    size_t ps_nseg_max = 0;
    WalkAuxHost walk{};          // key / entry buffers of the walk kernels (sized with the path state)
    size_t walk_key_cap = 0, walk_ent_total = 0;
    cudaStream_t stream = nullptr;
    float* d_sum = nullptr;
    unsigned char* d_rgb = nullptr;
    size_t d_sum_pix = 0;
    AdaptiveState adapt{};       // fw_render_adaptive: moments, counts, active lists (~33 B per pixel), sized on first use
    size_t adapt_pix = 0;
    // fw_render_aov / fw_render_denoised (~124 B per pixel), sized on first use: the AOV sums / guides, the filter's ping-pong
    // (colour, variance), the planar AOV, variance and denoised-colour outputs
    AovState aov{};
    float4* dn_cv[2] = {nullptr, nullptr};
    float* dn_planar = nullptr;    // albedo [3 npix], normal [3 npix], depth [npix]
    float* dn_var = nullptr;       // [npix]
    float* dn_color = nullptr;     // [3 npix]
    size_t dn_pix = 0;
    unsigned long long* d_rays = nullptr;   // device-side ray tally of the current render call
    unsigned long long* h_rays = nullptr;   // pinned
    std::vector<cudaEvent_t> ev_pool;
    cudaEvent_t ev_begin = nullptr, ev_end = nullptr;
    // Scene tables live in one device arena that the next scene on this context simply overwrites: committing and
    // releasing a scene costs no cudaMalloc / cudaFree (each cudaFree is a device-wide synchronisation; 17 of them
    // per scene made fw_scene_destroy take 200-500 ms inside a process that also runs torch).
    char* arena = nullptr;
    size_t arena_cap = 0, arena_used = 0;
    std::vector<void*> arena_retired;   // outgrown slabs, freed when the scene that may still use them is released
    // pinned staging for the small scene tables (api.cu upload): one H2D copy per contiguous arena range
    char* h_stage = nullptr;
    bool stage_failed = false;
    size_t stage_off = 0, stage_begin = 0, stage_len = 0;
    char* stage_dst = nullptr;
};

// Device-resident texture, process-wide and content-addressed (api.cu "texture store"): texels handed to
// fw_scene_set_image / fw_scene_set_hdr are hashed, and a scene whose texels are already resident on its device shares
// the array (read-only) instead of copying and uploading them again.
struct TexEntry {
    int device = 0;
    cudaArray_t arr = nullptr;
    cudaTextureObject_t tex = 0;
    cudaEvent_t ready = nullptr;   // recorded on the filling stream after the upload
    uint32_t w = 0, h = 0;
    bool is_float = false;
    bool hashed = false;           // false: filled with the store disabled (never shared by content)
    uint64_t hash[2] = {0, 0};
    int refs = 0;                  // scenes holding it: matched at set time and / or committed with it
    uint64_t last_use = 0;
};
struct AssetKey {
    bool hashed = false;
    uint64_t hash[2] = {0, 0};
};

struct fw_scene {
    SceneDesc desc;
    HostFlat flat;
    uint64_t h2d_bytes = 0;  // bytes copied host->device by commit
    bool built = false;      // host-side BVH build + flattening done
    bool committed = false;  // uploaded to the device
    int device = 0;
    int sm_count = 148;
    ExtendPlan plan;         // which extend kernel serves this scene (filled at commit)
    DeviceScene dscene{};
    LinProgram lin_prog{};     // linear-scan program, passed to the kernels by value (kernel-parameter space)
    bool lin_prog_ok = false;  // the scene's program fits FW_LIN_MAX_WORDS (else: object-loop kernels)
    bool mat_present[MAT_NUM_QUEUES] = {false, false, false, false, false, false};
    std::vector<HdrStaging*> hdr_staging;   // per asset: pinned RGBA copy of an HDR map (set_hdr .. commit)
    std::vector<AssetKey> asset_key;        // per asset: content hash of the texels handed in
    std::vector<TexEntry*> asset_held;      // per asset: resident copy matched at set time (the host copy was skipped)
    std::vector<TexEntry*> tex_used;        // entries the committed device scene reads (released with the device state)
    bool miss_is_zero = false;  // every escaping path contributes exactly 0: the miss kernel is not launched
    bool env_black = false;     // black ColorEnv: the miss kernel only has work in a batch some attenuation poisoned
    RenderCtx* ctx = nullptr;  // render-time state, borrowed from the per-device cache at commit
    size_t batch_paths = 0;    // 0 = default
    bool profiling = false;
    // fw_render_multi: committed copies of this scene on the other devices (created on first use, owned by this scene);
    // a replica reads its texels from the scene it was cloned from
    std::vector<fw_scene*> replicas;
    const fw_scene* asset_src = nullptr;
};

namespace fw {
// One sample range of `p` added into d_sum (device, width*height*3 fp32) on stream `st`; synchronises `st`.
int render_into(fw_scene* sc, const fw_params* p, float* d_sum, cudaStream_t st, fw_stats* stats);
int ensure_sum_buffers(fw_scene* sc, size_t npix);   // ctx->d_sum / d_rgb sized for npix pixels
int ensure_adaptive_buffers(fw_scene* sc, size_t npix);   // ctx->adapt sized for npix pixels
int ensure_denoise_buffers(fw_scene* sc, size_t npix);    // ctx->aov / dn_* sized for npix pixels
unsigned grid_for(size_t n, unsigned threads, unsigned max_blocks);
}  // namespace fw
