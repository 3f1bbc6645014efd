/* firework_b200.h — C ABI of the B200-native replacement for firework's rendering hot path.
 *
 * The reference (ritobanrc/firework, Rust) has no FFI layer; the seam this library sits behind is the call
 *
 *     Renderer::render(&self, scene: Scene) -> Vec<Color>            (reference src/render.rs:109)
 *
 * reached from src/main.rs:42 and every file under examples/.  `Scene` holds only trait objects
 * (src/scene.rs:20-24), so the type-erased form any host can hand over is the serde document
 * `serde_yaml::to_string(&scene)` (src/scene.rs:18, src/serde_compat.rs) — that text is what
 * fw_scene_from_yaml takes.  INTEGRATION.md shows the Rust binding (`extern "C"` + build.rs) a
 * maintainer would add to call this from `Renderer::render`; include/firework.hpp is a C++ mirror of the crate's public
 * builder API on top of this header (examples/ restates seven of the crate's examples with it).
 *
 * Conventions: plain pointers and sizes; the caller owns every buffer it passes; the library owns
 * fw_scene until fw_scene_destroy; every call returns 0 on success or a negative fw_status, and
 * fw_last_error() (thread-local) describes the failure; nothing throws or aborts across the boundary.
 * Calls on one fw_scene must not overlap; different scenes may be used from different threads.
 * There is no CPU fallback: without a CUDA device every compute entry point fails with FW_ERR_CUDA.
 */
#ifndef FIREWORK_B200_H
#define FIREWORK_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct fw_scene fw_scene;

typedef enum fw_status {
    FW_OK = 0,
    FW_ERR_PARSE = -1,    /* malformed YAML or unknown type tag                      */
    FW_ERR_SCENE = -2,    /* semantically invalid scene (no objects, bad indices...) */
    FW_ERR_ASSET = -3,    /* an ImageTexture / HdrEnvironment asset was not provided */
    FW_ERR_CUDA = -4,     /* CUDA runtime failure (incl. no device)                  */
    FW_ERR_ARG = -5,      /* bad argument                                            */
    FW_ERR_STATE = -6     /* call order violated (e.g. render before commit)         */
} fw_status;

/* Renderer + CameraSettings of the reference (src/render.rs:57-77, src/camera.rs:18-24), as one POD.
 * `samples` is the spp the image is normalised by (render.rs:184); the call renders the sample indices
 * [sample_begin, sample_begin + sample_count), which is how the sample range is sharded across GPUs.
 * `seed` keys the counter-based RNG that replaces tiny_rng::LcRng::new(idx) (render.rs:172). */
typedef struct fw_params {
    uint32_t width, height;
    uint32_t samples;
    uint32_t sample_begin, sample_count;
    uint32_t use_bvh;                  /* Renderer::use_bvh (render.rs:117-121, 128-132) */
    float gamma;                       /* Renderer::gamma   (render.rs:185-187)          */
    float cam_pos[3], look_at[3];
    float vfov, aperture, focus_dist;  /* camera.rs:74-107                                */
    uint64_t seed;
} fw_params;

typedef struct fw_stats {
    uint64_t samples;        /* width*height*sample_count                                   */
    uint64_t rays;           /* top-level closest-hit queries (calls of color(), render.rs:19) */
    uint64_t launches;       /* kernels launched by this call                               */
    double ms_device;        /* CUDA-event time of the device work of this call              */
    double ms_extend;        /* CUDA-event time spent in the extend kernels (0 unless profiling enabled) */
    uint64_t extend_launches;
} fw_stats;

/* ---- scene lifecycle ----------------------------------------------------------------------------------
 * replaces: serde_yaml::from_reader::<Scene> (src/main.rs:25-26) + SceneInternal::from(scene)
 *           (src/render.rs:113, src/scene.rs:111-135, 279-292) + build_bvh (src/bvh.rs:79-113).      */
int fw_scene_from_yaml(const char* text, size_t len, fw_scene** out);
int fw_scene_from_file(const char* path, fw_scene** out);
void fw_scene_destroy(fw_scene* scene);

/* Assets named by the document (ImageTexture `value:` — src/texture.rs:251-278; HdrEnvironment —
 * examples/hdri_test.rs:22-67).  The host decodes them and hands over texels. kind: 0 = image, 1 = HDR. */
int fw_scene_num_assets(const fw_scene* scene);
const char* fw_scene_asset_path(const fw_scene* scene, int index);
int fw_scene_asset_kind(const fw_scene* scene, int index);
int fw_scene_set_image(fw_scene* scene, int index, uint32_t width, uint32_t height, const uint8_t* rgba8);
int fw_scene_set_hdr(fw_scene* scene, int index, uint32_t width, uint32_t height, const float* rgb32f);

/* fw_scene_build_host: builds the BVHs with the reference's split rule (src/bvh.rs:21-71) and flattens the
 * scene into pointer-free arrays — host only, no CUDA.  fw_scene_commit: the same, then uploads to `device`. */
int fw_scene_build_host(fw_scene* scene);
int fw_scene_commit(fw_scene* scene, int device);

/* Introspection (host data; valid after fw_scene_build_host or fw_scene_commit). */
int fw_scene_num_objects(const fw_scene* scene);
int fw_scene_num_nodes(const fw_scene* scene);
int fw_scene_top_leaf_order(const fw_scene* scene, int* out, int capacity);          /* object ids, DFS leaf order */
int fw_scene_object_aabb(const fw_scene* scene, int object, float out_min_max[6]);   /* scene.rs:167-212 */
int fw_scene_mesh_leaf_order(const fw_scene* scene, int object, int* out, int capacity); /* triangle ids */
uint64_t fw_scene_device_bytes(const fw_scene* scene);  /* host->device bytes copied by fw_scene_commit */
/* The flattened 4-wide BVH nodes of all trees (top-level tree first; 32 floats per node, layout in
 * firework_b200/csrc/fw_types.h) and the top-level root code.  Copies up to `capacity_nodes` nodes, returns the count. */
int fw_scene_bvh_nodes(const fw_scene* scene, float* out_nodes, int capacity_nodes, int* top_root_code);
/* The linear-scan program of the scene (SceneInternal::hit, src/scene.rs:137-149, compiled to 16-byte words;
 * encoding in firework_b200/csrc/fw_types.h LinItem).  Copies up to `capacity_words` words (4 floats each) and
 * returns the program's length in words. */
int fw_scene_linear_program(const fw_scene* scene, float* out_words, int capacity_words);
/* Facts that decide whether the mesh-walk kernels serve the scene (firework_b200/csrc/walk.cuh): out = {usable, top-level
 * TriangleMesh objects, depth of the 4-wide top-level tree, depth of the deepest 4-wide mesh tree, primitive bits of the
 * 64-bit hit key, triangle slots}. */
int fw_scene_walk_info(const fw_scene* scene, int out[6]);

/* ---- the hot path -------------------------------------------------------------------------------------
 * replaces: the per-pixel loop of Renderer::render (src/render.rs:123-196).
 * rgb_out : width*height*3 u8, row 0 = top of image (== Vec<Color>); may be NULL.
 * sum_out : width*height*3 fp32 un-normalised radiance sums of the rendered sample range; may be NULL.
 * Host buffers; the call is synchronous.                                                                */
int fw_render(fw_scene* scene, const fw_params* params, uint8_t* rgb_out, float* sum_out, fw_stats* stats);

/* ---- adaptive sampling (no reference counterpart) -------------------------------------------------------
 * Renders each pixel until its noise estimate meets a target, with params->samples as the cap per pixel.  The call owns
 * the sample range: sample_begin must be 0 and sample_count == samples (else FW_ERR_ARG).  Single GPU.
 * Schedule: round 0 renders samples [0, n0), n0 = min(min_samples, samples), of every pixel; a pixel that does not stop
 *   after round r renders [n_r, n_{r+1}), n_{r+1} = min(2 n_r, samples), in round r + 1.  The render ends when no pixel is
 *   active or n_r == samples.
 * Stop rule (fp64, in this order): per sample Y = (0.2126 r + 0.7152 g) + 0.0722 b of the fp32 radiance; per pixel in
 *   sample order A = sum Y, B = sum Y^2; after n samples mean = A / n, var = max(0, (B - A mean) / (n - 1)),
 *   err = sqrt(var / n) / max(|mean|, floor), both maxima propagating NaN.  A pixel stops when n >= 2 and err <= threshold;
 *   a NaN error (NaN radiance; n = 1) never stops a pixel.
 * Exactness: a pixel that received k samples has the fp32 sum, bit for bit, and the u8 value of fw_render at samples = k.
 * Outputs (each nullable, width*height entries, row 0 = top): rgb_out u8 x3 = quantise(sum / (float)count); sum_out fp32 x3
 *   un-normalised sums; count_out samples per pixel; error_out the final err of each pixel.  stats->samples = sum of the
 *   counts; rays / launches / ms_device cover the whole call.  result->active[r] = pixels rendered in round r (r < 32).
 * Argument errors (null scene / params / adaptive, min_samples == 0, threshold negative or not finite, floor not > 0 or not
 * finite, the sample range) are reported before any CUDA call; an uncommitted scene gives FW_ERR_STATE. */
typedef struct fw_adaptive {
    uint32_t min_samples;   /* samples every pixel gets in round 0 (>= 1)                                 */
    float threshold;        /* stop a pixel when its relative standard error <= threshold (>= 0, finite) */
    float floor;            /* luminance floor of the relative error's denominator (> 0, finite)         */
} fw_adaptive;
typedef struct fw_adaptive_result {
    uint32_t rounds;
    uint64_t samples;       /* sum of the per-pixel counts */
    uint32_t active[32];    /* pixels rendered in round r  */
} fw_adaptive_result;
int fw_render_adaptive(fw_scene* scene, const fw_params* params, const fw_adaptive* adaptive, uint8_t* rgb_out, float* sum_out,
                       uint32_t* count_out, float* error_out, fw_stats* stats, fw_adaptive_result* result);

/* ---- denoised renders (no reference counterpart) ----------------------------------------------------------
 * First-hit feature buffers (AOVs) and an edge-aware a-trous filter (the spatial filter of SVGF, Schied et al. 2017); the
 * definitions, the filter's exact operation order and the measured results are in DESIGN.md §12.  Single GPU.
 *
 * fw_render_aov traces the primary ray of every (pixel, sample) of the sample range [sample_begin, sample_begin + sample_count)
 * through the scene's own bounce-0 extend kernels and averages, per pixel and in sample order in fp32, what it hits:
 *   albedo : the attenuation the first vertex applies, bit for bit what fw_render's shade kernel writes at bounce 0 (Lambertian
 *            and isotropic: the texture at the hit; metal: its albedo; dielectric, emissive and a miss: (1, 1, 1));
 *   normal : the normalised shading normal of the hit, (0, 0, 0) on a miss; the mean is not renormalised;
 *   depth  : t * |d| along the (unnormalised) camera ray, 0 on a miss;
 *   object : the object hit by sample sample_begin, -1 on a miss.
 * The RNG is keyed by (pixel, sample, bounce): the AOV of sample s describes the first vertex of fw_render's path for sample s.
 * Each fw_aov pointer is nullable: albedo / normal width*height*3 fp32, depth width*height fp32, object width*height int32. */
typedef struct fw_aov {
    float* albedo;
    float* normal;
    float* depth;
    int32_t* object;
} fw_aov;
/* Filter settings; every field is checked: iterations 1..10 (step 2^i at iteration i), aov_samples >= 1 (the AOV samples of
 * fw_render_denoised), each sigma finite and > 0.  Defaults (DESIGN.md §12): 5, 4, 4.0, 0.1, 0.1. */
typedef struct fw_denoise {
    uint32_t iterations;
    uint32_t aov_samples;
    float sigma_luminance;   /* luminance edge-stopping scale, in standard deviations of the 3x3-filtered variance */
    float sigma_depth;       /* relative depth difference scale                                                    */
    float sigma_albedo;      /* albedo difference scale                                                            */
} fw_denoise;
int fw_render_aov(fw_scene* scene, const fw_params* params, const fw_aov* aov, fw_stats* stats);
/* The filter on host buffers (width*height pixels, row 0 = top), on `device`, needs no scene: color fp32 x3 (linear), variance
 * fp32 (of the mean luminance), albedo x3, normal x3, depth.  color_out x3 receives the filtered colour, variance_out (nullable)
 * the filtered variance.  Argument errors are reported before any CUDA call. */
int fw_denoise_host(int device, uint32_t width, uint32_t height, const float* color, const float* variance, const float* albedo,
                    const float* normal, const float* depth, const fw_denoise* settings, float* color_out, float* variance_out);
/* A render followed by the AOV pass and the filter.  The call owns the sample range: sample_begin must be 0, sample_count ==
 * samples and samples >= 2 (else FW_ERR_ARG).
 *   1. every pixel renders samples [0, samples) with the kernels fw_render launches: sum_out equals fw_render's sums bit for
 *      bit; per pixel the luminance moments A = sum Y, B = sum Y^2 (fp64, Y as in fw_render_adaptive) give the variance of the
 *      mean v = max(0, (B - A (A / n)) / (n - 1)) / n, computed in fp64 and stored as fp32 (variance_out);
 *   2. fw_render_aov over samples [0, min(aov_samples, samples));
 *   3. fw_denoise_host's filter on (sum / (float)samples, v, the AOVs) -> denoised_out (linear fp32 x3); rgb_out u8 x3 is its
 *      resolve at samples = 1 with params->gamma.
 * Outputs are nullable; stats covers the whole call.  Argument errors (null scene / params / settings, the settings' ranges, the
 * sample range) are reported before any CUDA call; fw_render_aov and fw_render_denoised give FW_ERR_STATE for an uncommitted
 * scene. */
int fw_render_denoised(fw_scene* scene, const fw_params* params, const fw_denoise* settings, uint8_t* rgb_out, float* sum_out,
                       float* denoised_out, float* variance_out, const fw_aov* aov, fw_stats* stats);

/* Device-resident variant for multi-GPU sharding: ADDS the sample range into d_sum (device pointer,
 * width*height*3 fp32, on the scene's device) on `cuda_stream` (a cudaStream_t, or NULL for the scene's own
 * stream) and returns once the work is enqueued and statistics are read back. */
int fw_render_accumulate_device(fw_scene* scene, const fw_params* params, float* d_sum, void* cuda_stream,
                                fw_stats* stats);
/* render.rs:184-189 + util.rs:14-23 on a device sum buffer: d_rgb = quantise((d_sum / samples)^(1/gamma)). */
int fw_resolve_device(fw_scene* scene, const float* d_sum, uint32_t npix, uint32_t samples, float gamma,
                      uint8_t* d_rgb, void* cuda_stream);

/* The same resolve for a HOST sum buffer (e.g. sums accumulated by the caller across checkpointed render calls);
 * runs on `device`, needs no scene. */
int fw_resolve_host(int device, const float* sum, uint32_t npix, uint32_t samples, float gamma, uint8_t* rgb_out);

/* ---- one render call over several GPUs of one box (single process) ------------------------------------------
 * replaces: the same loop (src/render.rs:123-196); the reference has no multi-device path.  The call's sample range
 * [sample_begin, sample_begin + sample_count) is split into n_gpus contiguous slices; device i renders every pixel for
 * slice i (own host thread, own stream, own replica of the scene, created on first use), the fp32 sum buffers are
 * combined on devices[0] and resolved there.  `devices` lists the CUDA devices to use (NULL: the scene's device first,
 * then the lowest-numbered others); devices[0] must be the device the scene was committed on.
 * reduce_mode FW_REDUCE_NCCL: one ncclReduce(sum, fp32, root 0) over NVLink (libnccl.so.2 is loaded on first use);
 *             FW_REDUCE_PEER: one kernel on devices[0] reads the peers' buffers through NVLink peer mappings, sums them
 *             in rank order and resolves in the same pass.
 * rgb_out / sum_out as fw_render (sum_out receives the TOTAL over all devices).  ms_reduce (nullable): CUDA-event time
 * of the combine + resolve step on devices[0].  stats: samples / rays / launches summed over devices, ms_device = the
 * slowest device + the combine step. */
enum { FW_REDUCE_NCCL = 0, FW_REDUCE_PEER = 1 };
int fw_render_multi(fw_scene* scene, const fw_params* params, int n_gpus, const int* devices, int reduce_mode,
                    uint8_t* rgb_out, float* sum_out, fw_stats* stats, double* ms_reduce);

/* ---- probe entry points for the parity gates (host buffers) -----------------------------------------------
 * fw_primary_rays : camera.rs:109-116 + render.rs:173-180 for sample index `sample`, pixels [pix_begin, +n).
 * fw_first_hit    : render.rs:19 `root.hit(r, 0.001, 2e9, rng)`; obj = -1 on miss. pixel/sample/bounce key
 *                   the ConstantMedium draw (may be NULL: pixel = i, sample = bounce = 0).
 *                   counters (nullable) receives {node tests, primitive tests}.
 * fw_scatter_step : render.rs:20-22 emit + scatter with EXPLICIT uniforms (nu per item, consumed in order).
 * fw_env_sample / fw_texture_sample : render.rs:31 / texture.rs lookups.                                 */
int fw_primary_rays(fw_scene* scene, const fw_params* params, uint32_t sample, uint32_t pix_begin, uint32_t n,
                    float* origins, float* dirs);
int fw_first_hit(fw_scene* scene, int use_bvh, uint64_t seed, uint32_t n, const float* origins, const float* dirs,
                 const uint32_t* pixel, const uint32_t* sample, const uint32_t* bounce, int32_t* obj, int32_t* prim,
                 int32_t* material, float* t, float* point, float* normal, float* uv, uint64_t counters[2]);
/* fw_first_hit answers from a probe kernel that calls the traversal routines directly; fw_first_hit_wavefront pushes the
 * same rays through the kernels a render launches — the segmented queues, the scene's own extend kernels (lock-step,
 * linear program or the mesh walk) and finalize_hit — so the first-hit gate covers the production path.  Ray i is keyed
 * as (pixel i, `sample`, `bounce`), bounce <= 10. */
int fw_first_hit_wavefront(fw_scene* scene, int use_bvh, uint64_t seed, uint32_t n, const float* origins, const float* dirs,
                           uint32_t sample, uint32_t bounce, int32_t* obj, int32_t* prim, int32_t* material, float* t,
                           float* point, float* normal, float* uv);
int fw_scatter_step(fw_scene* scene, uint32_t n, const int32_t* material, const float* ray_o, const float* ray_d,
                    const float* hit_t, const float* hit_point, const float* hit_normal, const float* hit_uv,
                    const float* uniforms, uint32_t nu, float* emit, int32_t* scattered, float* atten, float* out_o,
                    float* out_d, int32_t* consumed);
int fw_env_sample(fw_scene* scene, uint32_t n, const float* dirs, float* out);
int fw_texture_sample(fw_scene* scene, int texture, uint32_t n, const float* uv, const float* point, float* out);
int fw_material_texture(const fw_scene* scene, int material);  /* texture index of a material, or -1 */
int fw_camera(const fw_params* params, float out24[24]);        /* camera.rs:74-107 constants, host only */

/* ---- misc ----------------------------------------------------------------------------------------------- */
const char* fw_last_error(void);
const char* fw_version(void);
int fw_device_count(void);
/* ---- asset ingestion in front of the path (what the reference's examples do with third-party crates) --------
 * fw_obj_load  : Wavefront OBJ -> indexed triangle models, as tobj 1.0.0 `load_obj` (examples/suzanne.rs:15-51,
 *                examples/teapot.rs:17-64): one model per `o` / `g` group, fan triangulation, one vertex per distinct
 *                v/vt/vn triple in order of first use.  The arrays feed TriangleMesh::new (src/objects/mesh.rs:36-72).
 * fw_hdr_load  : Radiance RGBE .hdr -> fp32 RGB, row 0 = top, as image 0.23.9 `HdrDecoder::read_image_hdr`
 *                (examples/hdri_test.rs:45-67); the result feeds fw_scene_set_hdr.  Free with fw_hdr_free.
 * The native command-line driver built on these (csrc/cli_main.cpp -> firework_b200/bin/firework) is src/main.rs. */
typedef struct fw_obj fw_obj;
int fw_obj_load(const char* path, fw_obj** out);
int fw_obj_num_models(const fw_obj* obj);
const char* fw_obj_model_name(const fw_obj* obj, int model);
int fw_obj_model_sizes(const fw_obj* obj, int model, uint32_t sizes[4]);   /* floats: positions, normals, texcoords; indices */
int fw_obj_model_copy(const fw_obj* obj, int model, float* positions, float* normals, float* texcoords, uint32_t* indices);
void fw_obj_destroy(fw_obj* obj);
int fw_hdr_load(const char* path, uint32_t* width, uint32_t* height, float** rgb);
void fw_hdr_free(float* rgb);
/* fw_image_load: PNG (non-interlaced) or baseline JPEG -> RGBA8, row 0 = top, as `image::open(path)...to_rgba()` in
 *                ImageTexture::from_path / sample (src/texture.rs:285-292, 304); feeds fw_scene_set_image.  Free with
 *                fw_image_free.
 * fw_png_write : width*height*3 u8 (what fw_render returns) -> PNG file, as window.rs `save_image` (src/main.rs:55). */
int fw_image_load(const char* path, uint32_t* width, uint32_t* height, uint8_t** rgba);
void fw_image_free(uint8_t* rgba);
int fw_png_write(const char* path, uint32_t width, uint32_t height, const uint8_t* rgb);

/* Self-test of the shared-reciprocal division used by the linear-scan kernels (t = (k - o[a]) / d[a],
 * src/objects/rect.rs:49) against the hardware's IEEE division on n_pairs pseudo-random / adversarial operand pairs.
 * violations[0]: results that are not bit-identical where exactness is promised; violations[1]: tiny-numerator
 * results that would not be rejected by t_min = 0.001 (src/render.rs:19).  Both must be 0. */
int fw_selftest_shared_division(int device, uint64_t n_pairs, uint64_t seed, uint64_t violations[2]);

/* Microbenchmarks used by bench.py for the roofline denominators: dependent-free FP32 FMA rate (TFLOP/s) and
 * L2-resident streaming read bandwidth (GB/s) on `device`. */
int fw_measure_peaks(int device, double* fp32_tflops, double* l2_gbs, int* sm_count, int* sm_clock_khz);
/* Per-kernel CUDA-event profiling of extend launches (adds synchronisation; off by default). */
int fw_set_profiling(fw_scene* scene, int enabled);
/* Render-time device buffers (path-state streams, ~1.2 GB at the default batch size) are cached per device
 * across scenes; this frees every cached context that is not in use. */
int fw_release_cached_memory(void);
/* Texture store (no reference counterpart): texels handed to fw_scene_set_image / fw_scene_set_hdr are hashed, and a scene
 * whose texels are already resident on its device shares that array instead of copying and uploading them again
 * (FW_TEXTURE_CACHE=0 in the environment disables the lookup).  out = {commits served from a resident array, uploads,
 * arrays resident now, their bytes}. */
int fw_texture_store_stats(uint64_t out[4]);
/* Maximum number of paths in flight per batch (0 = default). */
int fw_set_batch_paths(fw_scene* scene, uint64_t paths);

#ifdef __cplusplus
}
#endif
#endif /* FIREWORK_B200_H */
