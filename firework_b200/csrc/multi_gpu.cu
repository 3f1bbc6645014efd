// fw_render_multi: one render call over several GPUs of one box, inside one process (SURVEY.md §8b / §8e).
//
// The sample range of the call is split into contiguous slices, one per device (the RNG is keyed by the global sample
// index, so the union of the slices is the single-GPU render).  The scene is replicated (it is KiB..MiB plus textures),
// one host thread drives each device through the ordinary single-GPU path into that device's fp32 sum buffer, and the
// buffers are then combined on the first device in one of two ways:
//   FW_REDUCE_NCCL : ncclReduce(sum, fp32) over NVLink / NVSwitch to device 0, then the resolve kernel there
//                    (BASELINE.json north_star: "summed with a single NCCL reduce, which is the only collective");
//   FW_REDUCE_PEER : one kernel on device 0 reads every peer's buffer directly through NVLink peer mappings, adds them in
//                    rank order and resolves in the same pass (sum + mean + gamma + quantise fused; no staging copy, and
//                    the summation order is fixed, so the image is bit-reproducible for a given device count).
// NCCL is bound at run time (dlopen of libnccl.so.2), so the library itself carries no link-time dependency on it; the
// reference has no multi-device path at all (src/render.rs:127 is a rayon loop).
#include <dlfcn.h>

#include <algorithm>
#include <cstdlib>
#include <cstring>
#include <map>
#include <thread>

#include "api_internal.h"

using namespace fw;

namespace {

// ---- the slice of NCCL's C API used here (stable ABI since NCCL 2.0; nccl.h is not required to build) ----
typedef struct ncclComm* ncclComm_t;
typedef int ncclResult_t;
constexpr int kNcclFloat = 7, kNcclSum = 0;
struct NcclApi {
    void* handle = nullptr;
    ncclResult_t (*CommInitAll)(ncclComm_t*, int, const int*) = nullptr;
    ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
    ncclResult_t (*Reduce)(const void*, void*, size_t, int, int, int, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*GroupStart)() = nullptr;
    ncclResult_t (*GroupEnd)() = nullptr;
    const char* (*GetErrorString)(ncclResult_t) = nullptr;
    std::string error;
};
std::mutex g_nccl_mutex;
NcclApi g_nccl;
std::map<std::vector<int>, std::vector<ncclComm_t>> g_comms;   // communicators per device list, created once

bool load_nccl() {
    if (g_nccl.handle) return true;
    // FW_NCCL_LIB names the library to use.  A host that also loads another NCCL user later (PyTorch bundles its own, newer
    // libnccl.so.2) must point this at THAT copy: the dynamic loader keeps one library per SONAME, so whichever is loaded
    // first serves both (firework_b200/_native.py sets it when the nvidia-nccl wheel is installed).
    const char* names[] = {getenv("FW_NCCL_LIB"), "libnccl.so.2", "libnccl.so"};
    for (const char* n : names) {
        if (!n || !*n) continue;
        g_nccl.handle = dlopen(n, RTLD_NOW | RTLD_LOCAL);
        if (g_nccl.handle) break;
    }
    if (!g_nccl.handle) {
        g_nccl.error = std::string("cannot load libnccl.so.2: ") + dlerror();
        return false;
    }
    bool ok = true;
    auto sym = [&](const char* name) {
        void* p = dlsym(g_nccl.handle, name);
        if (!p) { ok = false; g_nccl.error = std::string("libnccl lacks ") + name; }
        return p;
    };
    g_nccl.CommInitAll = reinterpret_cast<decltype(g_nccl.CommInitAll)>(sym("ncclCommInitAll"));
    g_nccl.CommDestroy = reinterpret_cast<decltype(g_nccl.CommDestroy)>(sym("ncclCommDestroy"));
    g_nccl.Reduce = reinterpret_cast<decltype(g_nccl.Reduce)>(sym("ncclReduce"));
    g_nccl.GroupStart = reinterpret_cast<decltype(g_nccl.GroupStart)>(sym("ncclGroupStart"));
    g_nccl.GroupEnd = reinterpret_cast<decltype(g_nccl.GroupEnd)>(sym("ncclGroupEnd"));
    g_nccl.GetErrorString = reinterpret_cast<decltype(g_nccl.GetErrorString)>(sym("ncclGetErrorString"));
    if (!ok) { dlclose(g_nccl.handle); g_nccl.handle = nullptr; }
    return ok;
}

int nccl_comms(const std::vector<int>& devs, std::vector<ncclComm_t>** out) {
    std::lock_guard<std::mutex> lk(g_nccl_mutex);
    if (!load_nccl()) return set_error(FW_ERR_CUDA, g_nccl.error);
    auto it = g_comms.find(devs);
    if (it == g_comms.end()) {
        std::vector<ncclComm_t> comms(devs.size(), nullptr);
        ncclResult_t r = g_nccl.CommInitAll(comms.data(), (int)devs.size(), devs.data());
        if (r != 0) return set_error(FW_ERR_CUDA, std::string("ncclCommInitAll: ") + g_nccl.GetErrorString(r));
        it = g_comms.emplace(devs, std::move(comms)).first;
    }
    *out = &it->second;
    return FW_OK;
}

// Creates (once) and commits the copy of `sc` that lives on `device`.
int replica_on(fw_scene* sc, int device, fw_scene** out) {
    if (device == sc->device) { *out = sc; return FW_OK; }
    for (fw_scene* r : sc->replicas)
        if (r->device == device) { *out = r; return FW_OK; }
    fw_scene* r = new fw_scene();
    r->desc = sc->desc;
    for (AssetDesc& a : r->desc.assets) {   // texels stay with the original (commit reads them through asset_src)
        a.rgba.clear(); a.rgba.shrink_to_fit();
        a.rgb.clear(); a.rgb.shrink_to_fit();
    }
    r->flat = sc->flat;
    r->built = sc->built;
    r->asset_src = sc;
    r->batch_paths = sc->batch_paths;
    int rc = fw_scene_commit(r, device);
    if (rc != FW_OK) { fw_scene_destroy(r); return rc; }
    sc->replicas.push_back(r);
    *out = r;
    return FW_OK;
}

}  // namespace

extern "C" int fw_render_multi(fw_scene* sc, const fw_params* p, int n_gpus, const int* devices, int reduce_mode,
                               uint8_t* rgb_out, float* sum_out, fw_stats* stats, double* ms_reduce) {
    if (!sc || !p) return set_error(FW_ERR_ARG, "null argument");
    if (!sc->committed) return set_error(FW_ERR_STATE, "fw_scene_commit must be called before rendering");
    if (n_gpus < 1 || n_gpus > kMaxPeers) return set_error(FW_ERR_ARG, "n_gpus must be in [1, 16]");
    if (reduce_mode != FW_REDUCE_NCCL && reduce_mode != FW_REDUCE_PEER) return set_error(FW_ERR_ARG, "unknown reduce mode");
    int ndev = 0;
    FW_CUDA(cudaGetDeviceCount(&ndev));
    std::vector<int> devs(n_gpus);
    for (int i = 0; i < n_gpus; ++i) {
        devs[i] = devices ? devices[i] : (i == 0 ? sc->device : (i <= sc->device ? i - 1 : i));
        if (devs[i] < 0 || devs[i] >= ndev) return set_error(FW_ERR_CUDA, "no such CUDA device " + std::to_string(devs[i]));
        for (int j = 0; j < i; ++j)
            if (devs[j] == devs[i]) return set_error(FW_ERR_ARG, "device listed twice");
    }
    if (devs[0] != sc->device) return set_error(FW_ERR_ARG, "devices[0] must be the device the scene was committed on");
    const size_t npix = (size_t)p->width * p->height;
    if (npix == 0 || p->samples == 0) return set_error(FW_ERR_ARG, "width, height and samples must be non-zero");

    // replicas are created serially (cudaMalloc / texture creation), then every device renders from its own host thread
    std::vector<fw_scene*> sc_on(n_gpus, nullptr);
    for (int i = 0; i < n_gpus; ++i) {
        int rc = replica_on(sc, devs[i], &sc_on[i]);
        if (rc != FW_OK) return rc;
        sc_on[i]->profiling = sc->profiling;
        sc_on[i]->batch_paths = sc->batch_paths;
    }
    std::vector<int> rcs(n_gpus, FW_OK);
    std::vector<std::string> errs(n_gpus);
    std::vector<fw_stats> sts(n_gpus);
    auto work = [&](int i) {
        fw_scene* s = sc_on[i];
        int rc = FW_OK;
        do {
            if (cudaSetDevice(s->device) != cudaSuccess) { rc = set_error(FW_ERR_CUDA, "cudaSetDevice failed"); break; }
            if ((rc = ensure_sum_buffers(s, npix)) != FW_OK) break;
            if (cudaMemsetAsync(s->ctx->d_sum, 0, npix * 3 * sizeof(float), s->ctx->stream) != cudaSuccess) {
                rc = set_error(FW_ERR_CUDA, "cudaMemsetAsync failed");
                break;
            }
            // slice i of the call's sample range: contiguous, disjoint, covering; sizes differ by at most one
            fw_params q = *p;
            const uint64_t c = p->sample_count;
            const uint32_t b0 = (uint32_t)((uint64_t)i * c / n_gpus), b1 = (uint32_t)((uint64_t)(i + 1) * c / n_gpus);
            q.sample_begin = p->sample_begin + b0;
            q.sample_count = b1 - b0;
            memset(&sts[i], 0, sizeof(fw_stats));
            if (q.sample_count == 0) {
                if (cudaStreamSynchronize(s->ctx->stream) != cudaSuccess) rc = set_error(FW_ERR_CUDA, "cudaStreamSynchronize failed");
                break;
            }
            rc = render_into(s, &q, s->ctx->d_sum, s->ctx->stream, &sts[i]);
        } while (false);
        rcs[i] = rc;
        if (rc != FW_OK) errs[i] = fw_last_error();
    };
    {
        std::vector<std::thread> th;
        for (int i = 1; i < n_gpus; ++i) th.emplace_back(work, i);
        work(0);
        for (auto& t : th) t.join();
    }
    for (int i = 0; i < n_gpus; ++i)
        if (rcs[i] != FW_OK) return set_error(rcs[i], "device " + std::to_string(devs[i]) + ": " + errs[i]);

    // ---- combine on devs[0] --------------------------------------------------------------------------------------
    FW_CUDA(cudaSetDevice(sc->device));
    RenderCtx* c0 = sc->ctx;
    cudaEvent_t e0, e1;
    FW_CUDA(cudaEventCreate(&e0));
    FW_CUDA(cudaEventCreate(&e1));
    FW_CUDA(cudaEventRecord(e0, c0->stream));
    const uint32_t n_values = (uint32_t)(npix * 3);
    bool resolved = false;
    if (n_gpus > 1 && reduce_mode == FW_REDUCE_PEER) {
        PeerSums src;
        src.n = n_gpus;
        for (int i = 0; i < n_gpus; ++i) src.p[i] = sc_on[i]->ctx->d_sum;
        for (int i = 1; i < n_gpus; ++i) {
            int can = 0;
            FW_CUDA(cudaDeviceCanAccessPeer(&can, sc->device, devs[i]));
            if (!can) return set_error(FW_ERR_CUDA, "device " + std::to_string(sc->device) + " cannot map the memory of device " + std::to_string(devs[i]));
            cudaError_t e = cudaDeviceEnablePeerAccess(devs[i], 0);
            if (e == cudaErrorPeerAccessAlreadyEnabled) cudaGetLastError();
            else if (e != cudaSuccess) return set_error(FW_ERR_CUDA, std::string("cudaDeviceEnablePeerAccess: ") + cudaGetErrorString(e));
        }
        launch_peer_reduce_resolve(src, c0->d_sum, n_values, (float)p->samples, p->gamma, rgb_out ? c0->d_rgb : nullptr,
                                   grid_for(n_values, 256, sc->sm_count * 8), c0->stream);
        FW_CUDA(cudaGetLastError());
        resolved = true;
    } else if (n_gpus > 1) {
        std::vector<ncclComm_t>* comms = nullptr;
        int rc = nccl_comms(devs, &comms);
        if (rc != FW_OK) return rc;
        ncclResult_t r = g_nccl.GroupStart();
        for (int i = 0; i < n_gpus && r == 0; ++i) {
            float* buf = sc_on[i]->ctx->d_sum;
            r = g_nccl.Reduce(buf, buf, n_values, kNcclFloat, kNcclSum, 0, (*comms)[i], sc_on[i]->ctx->stream);
        }
        ncclResult_t r2 = g_nccl.GroupEnd();
        if (r == 0) r = r2;
        if (r != 0) return set_error(FW_ERR_CUDA, std::string("ncclReduce: ") + g_nccl.GetErrorString(r));
    }
    if (rgb_out && !resolved) {
        launch_resolve(c0->d_sum, (uint32_t)npix, (float)p->samples, p->gamma, c0->d_rgb, grid_for(npix, 256, sc->sm_count * 8), c0->stream);
        FW_CUDA(cudaGetLastError());
    }
    FW_CUDA(cudaEventRecord(e1, c0->stream));
    if (rgb_out) FW_CUDA(cudaMemcpyAsync(rgb_out, c0->d_rgb, npix * 3, cudaMemcpyDeviceToHost, c0->stream));
    if (sum_out) FW_CUDA(cudaMemcpyAsync(sum_out, c0->d_sum, npix * 3 * sizeof(float), cudaMemcpyDeviceToHost, c0->stream));
    FW_CUDA(cudaStreamSynchronize(c0->stream));
    for (int i = 1; i < n_gpus; ++i) {   // the peers' part of the reduce has completed too before their buffers are reused
        FW_CUDA(cudaSetDevice(devs[i]));
        FW_CUDA(cudaStreamSynchronize(sc_on[i]->ctx->stream));
    }
    FW_CUDA(cudaSetDevice(sc->device));
    float ms = 0.0f;
    FW_CUDA(cudaEventElapsedTime(&ms, e0, e1));
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    if (ms_reduce) *ms_reduce = ms;
    if (stats) {
        memset(stats, 0, sizeof(*stats));
        for (int i = 0; i < n_gpus; ++i) {
            stats->samples += sts[i].samples;
            stats->rays += sts[i].rays;
            stats->launches += sts[i].launches;
            stats->extend_launches += sts[i].extend_launches;
            stats->ms_device = std::max(stats->ms_device, sts[i].ms_device);   // devices run concurrently
            stats->ms_extend = std::max(stats->ms_extend, sts[i].ms_extend);
        }
        stats->launches += 1;
        stats->ms_device += ms;
    }
    return FW_OK;
}
