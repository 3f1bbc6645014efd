"""Thin host-side wrapper over the C ABI: scene handle, asset hand-over, render and probe calls.

Mirrors the call sequence of the reference's front ends (src/main.rs:22-47, examples/*.rs):
load/build a `Scene` -> `Renderer::render(scene)` -> pixels.
"""
from __future__ import annotations

import ctypes as C
from typing import Optional

import numpy as np

from . import _native as N
from .assets import load_asset

# Default luminance floor of the adaptive stop rule's denominator, max(|mean|, floor).  Below it the rule asks for an absolute
# standard error of threshold * floor instead of a relative one: at 0.01 (linear; u8 31 after gamma 2.2) and threshold 0.05
# that is 5e-4, under one u8 level after the gamma curve, so black and near-black pixels (shadows, an unlit background)
# stop instead of chasing a relative error their displayed value can not show.
ADAPTIVE_FLOOR = 0.01

# Settings of the edge-aware a-trous filter (fw_denoise, DESIGN.md §12): iterations (step 2^i at iteration i, 1..10), the AOV
# samples of a denoised render, and the luminance (SVGF's value), relative depth and albedo edge-stopping scales.
DENOISE_DEFAULTS = {"iterations": 5, "aov_samples": 4, "sigma_luminance": 4.0, "sigma_depth": 0.1, "sigma_albedo": 0.1}


def _denoise_settings(settings) -> N.FwDenoise:
    unknown = set(settings) - set(DENOISE_DEFAULTS)
    if unknown:
        raise TypeError(f"unknown denoise settings: {sorted(unknown)}")
    s = dict(DENOISE_DEFAULTS, **settings)
    return N.FwDenoise(int(s["iterations"]), int(s["aov_samples"]), float(s["sigma_luminance"]), float(s["sigma_depth"]),
                       float(s["sigma_albedo"]))


def _aov_arrays(h, w):
    aov = {"albedo": np.empty((h, w, 3), np.float32), "normal": np.empty((h, w, 3), np.float32),
           "depth": np.empty((h, w), np.float32), "object": np.empty((h, w), np.int32)}
    return aov, N.FwAov(*(N.ptr(aov[k]) for k in ("albedo", "normal", "depth", "object")))


def _ray_layout(origins, dirs, sample_count, keys):
    """(number of rays, per-sample layout?) of trace_rays' inputs: (N, 3) shared, (sample_count, N, 3) per sample."""
    shape = tuple(origins.shape)
    if tuple(dirs.shape) != shape:
        raise ValueError(f"origins {shape} and dirs {tuple(dirs.shape)} must have the same shape")
    if len(shape) == 2 and shape[1] == 3:
        n, per_sample = shape[0], False
    elif len(shape) == 3 and shape[2] == 3 and shape[0] == sample_count:
        n, per_sample = shape[1], True
    else:
        raise ValueError(f"rays must be (N, 3) or (sample_count={sample_count}, N, 3), got {shape}")
    if keys is not None and tuple(keys.shape) != (n,):
        raise ValueError(f"keys must be ({n},), got {tuple(keys.shape)}")
    return int(n), per_sample


class NativeScene:
    """A committed fw_scene on one GPU."""

    def __init__(self, yaml_text: str, device: int = 0, asset_dir: Optional[str] = None,
                 assets: Optional[dict] = None, commit: bool = True):
        L = N.lib()
        self._h = C.c_void_p()
        data = yaml_text.encode("utf-8")
        N.check(L.fw_scene_from_yaml(data, len(data), C.byref(self._h)))
        self.device = device
        self.h2d_asset_bytes = 0
        for i in range(L.fw_scene_num_assets(self._h)):
            path = L.fw_scene_asset_path(self._h, i).decode()
            kind = L.fw_scene_asset_kind(self._h, i)
            arr = load_asset(path, "hdr" if kind == 1 else "image", asset_dir, assets)
            if kind == 1:
                arr = np.ascontiguousarray(arr, np.float32)
                N.check(L.fw_scene_set_hdr(self._h, i, arr.shape[1], arr.shape[0], N.ptr(arr)))
            else:
                arr = np.ascontiguousarray(arr, np.uint8)
                N.check(L.fw_scene_set_image(self._h, i, arr.shape[1], arr.shape[0], N.ptr(arr)))
            self.h2d_asset_bytes += arr.nbytes
        self.yaml_bytes = len(data)
        if commit:
            self.commit()

    @staticmethod
    def from_scene(scene, device: int = 0) -> "NativeScene":
        return NativeScene(scene.to_yaml(), device, scene.asset_dir, scene.assets)

    def commit(self):
        N.check(N.lib().fw_scene_commit(self._h, self.device))

    def build_host(self):
        """BVH build + flattening only (no CUDA): enough for the structural introspection calls."""
        N.check(N.lib().fw_scene_build_host(self._h))

    def close(self):
        if self._h:
            N.lib().fw_scene_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ---- introspection ---------------------------------------------------------------------------------
    def num_objects(self):
        return N.lib().fw_scene_num_objects(self._h)

    def num_nodes(self):
        return N.lib().fw_scene_num_nodes(self._h)

    def device_bytes(self):
        return int(N.lib().fw_scene_device_bytes(self._h))

    def top_leaf_order(self):
        n = self.num_objects()
        out = np.zeros(n, np.int32)
        N.check(N.lib().fw_scene_top_leaf_order(self._h, N.ptr(out), n))
        return out

    def object_aabbs(self):
        n = self.num_objects()
        out = np.zeros((n, 6), np.float32)
        for i in range(n):
            N.check(N.lib().fw_scene_object_aabb(self._h, i, N.ptr(out[i])))
        return out

    def mesh_leaf_order(self, obj):
        n = N.check(N.lib().fw_scene_mesh_leaf_order(self._h, obj, None, 0))
        out = np.zeros(n, np.int32)
        N.check(N.lib().fw_scene_mesh_leaf_order(self._h, obj, N.ptr(out), n))
        return out

    def bvh_nodes(self):
        """(nodes (n, 8, 4) float32 — int fields are bit patterns —, top-level root code)."""
        root = C.c_int()
        n = N.check(N.lib().fw_scene_bvh_nodes(self._h, None, 0, C.byref(root)))
        out = np.zeros((max(n, 1), 8, 4), np.float32)
        N.check(N.lib().fw_scene_bvh_nodes(self._h, N.ptr(out), n, C.byref(root)))
        return out[:n], root.value

    def linear_program(self):
        """The scene's linear-scan program as an (n_words, 4) float32 array (fw_types.h LinItem encoding)."""
        n = N.check(N.lib().fw_scene_linear_program(self._h, None, 0))
        out = np.zeros((n, 4), np.float32)
        N.check(N.lib().fw_scene_linear_program(self._h, N.ptr(out), n))
        return out

    def walk_info(self):
        """{usable, top_meshes, top_wide_depth, mesh_wide_depth, prim_bits, triangles} (fw_scene_walk_info)."""
        out = np.zeros(6, np.int32)
        N.check(N.lib().fw_scene_walk_info(self._h, N.ptr(out)))
        return dict(zip(("usable", "top_meshes", "top_wide_depth", "mesh_wide_depth", "prim_bits", "triangles"), (int(v) for v in out)))

    def material_texture(self, material):
        return N.lib().fw_material_texture(self._h, material)

    def set_profiling(self, on: bool):
        N.check(N.lib().fw_set_profiling(self._h, 1 if on else 0))

    def set_batch_paths(self, paths: int):
        N.check(N.lib().fw_set_batch_paths(self._h, int(paths)))

    # ---- the hot path ----------------------------------------------------------------------------------
    def render(self, params: N.FwParams, want_rgb=True, want_sum=True):
        """fw_render with host buffers. Returns (rgb (H,W,3) u8 | None, sum (H,W,3) f32 | None, stats dict)."""
        h, w = params.height, params.width
        rgb = np.empty((h, w, 3), np.uint8) if want_rgb else None
        s = np.empty((h, w, 3), np.float32) if want_sum else None
        st = N.FwStats()
        N.check(N.lib().fw_render(self._h, C.byref(params), N.ptr(rgb) if want_rgb else None,
                                  N.ptr(s) if want_sum else None, C.byref(st)))
        return rgb, s, st.as_dict()

    def render_adaptive(self, params: N.FwParams, threshold: float, min_samples: int = 16, floor: float = ADAPTIVE_FLOOR,
                        want_rgb=True, want_sum=True):
        """fw_render_adaptive: every pixel renders until its relative standard error is <= `threshold`, with
        `params.samples` as the cap (params must cover the whole range: sample_begin 0, sample_count == samples).
        Returns (rgb (H,W,3) u8 | None, sum (H,W,3) f32 | None, counts (H,W) u32, err (H,W) f32, stats dict); stats adds
        `rounds` and `active` (pixels rendered in each round) to the fw_stats fields, and stats["samples"] is the sum of
        the counts."""
        h, w = params.height, params.width
        rgb = np.empty((h, w, 3), np.uint8) if want_rgb else None
        s = np.empty((h, w, 3), np.float32) if want_sum else None
        counts = np.empty((h, w), np.uint32)
        err = np.empty((h, w), np.float32)
        ad = N.FwAdaptive(int(min_samples), float(threshold), float(floor))
        st, res = N.FwStats(), N.FwAdaptiveResult()
        N.check(N.lib().fw_render_adaptive(self._h, C.byref(params), C.byref(ad), N.ptr(rgb) if want_rgb else None,
                                           N.ptr(s) if want_sum else None, N.ptr(counts), N.ptr(err), C.byref(st), C.byref(res)))
        d = st.as_dict()
        d["rounds"] = int(res.rounds)
        d["active"] = [int(res.active[r]) for r in range(min(res.rounds, 32))]
        return rgb, s, counts, err, d

    def render_aov(self, params: N.FwParams):
        """fw_render_aov: per-pixel means over the params' sample range of what the primary rays hit first.  Returns
        ({albedo (H,W,3), normal (H,W,3), depth (H,W) f32, object (H,W) i32 of the range's first sample}, stats dict)."""
        aov, fa = _aov_arrays(params.height, params.width)
        st = N.FwStats()
        N.check(N.lib().fw_render_aov(self._h, C.byref(params), C.byref(fa), C.byref(st)))
        return aov, st.as_dict()

    def render_denoised(self, params: N.FwParams, want_rgb=True, want_sum=True, **settings):
        """fw_render_denoised: a render of samples [0, params.samples) (params must cover that whole range, samples >= 2), the AOV
        pass over the first `aov_samples` of them and the a-trous filter; `settings` override DENOISE_DEFAULTS.  Returns
        (rgb (H,W,3) u8 of the denoised image | None, sum (H,W,3) f32 | None, denoised (H,W,3) f32 linear, variance (H,W) f32 of
        the mean luminance before filtering, aov dict as render_aov, stats dict)."""
        h, w = params.height, params.width
        rgb = np.empty((h, w, 3), np.uint8) if want_rgb else None
        s = np.empty((h, w, 3), np.float32) if want_sum else None
        den = np.empty((h, w, 3), np.float32)
        var = np.empty((h, w), np.float32)
        aov, fa = _aov_arrays(h, w)
        st = N.FwStats()
        N.check(N.lib().fw_render_denoised(self._h, C.byref(params), C.byref(_denoise_settings(settings)),
                                           N.ptr(rgb) if want_rgb else None, N.ptr(s) if want_sum else None, N.ptr(den), N.ptr(var),
                                           C.byref(fa), C.byref(st)))
        return rgb, s, den, var, aov, st.as_dict()

    def render_multi(self, params: N.FwParams, n_gpus: int, devices=None, reduce="nccl", want_rgb=True, want_sum=True):
        """fw_render_multi: the call's sample range split over `n_gpus` devices of this box (single process), sums
        combined on this scene's device by one NCCL reduce (`reduce="nccl"`) or by the fused peer-memory
        reduce + resolve kernel (`reduce="peer"`).  Returns (rgb | None, total sum | None, stats dict)."""
        h, w = params.height, params.width
        rgb = np.empty((h, w, 3), np.uint8) if want_rgb else None
        s = np.empty((h, w, 3), np.float32) if want_sum else None
        st = N.FwStats()
        ms = C.c_double()
        dev = None if devices is None else np.ascontiguousarray(devices, np.int32)
        N.check(N.lib().fw_render_multi(self._h, C.byref(params), int(n_gpus), None if dev is None else N.ptr(dev),
                                        {"nccl": 0, "peer": 1}[reduce], N.ptr(rgb) if want_rgb else None,
                                        N.ptr(s) if want_sum else None, C.byref(st), C.byref(ms)))
        d = st.as_dict()
        d["ms_reduce"] = ms.value
        return rgb, s, d

    def render_accumulate_device(self, params: N.FwParams, d_sum_ptr: int, stream_ptr: int = 0):
        """Adds the params' sample range into a device fp32 buffer (e.g. a torch tensor's data_ptr())."""
        st = N.FwStats()
        N.check(N.lib().fw_render_accumulate_device(self._h, C.byref(params), C.c_void_p(d_sum_ptr),
                                                    C.c_void_p(stream_ptr) if stream_ptr else None, C.byref(st)))
        return st.as_dict()

    def trace_rays(self, origins, dirs, sample_count=1, sample_begin=0, seed=0, use_bvh=False, keys=None):
        """fw_trace_rays (DESIGN.md §13): path-traces samples [sample_begin, sample_begin + sample_count) of caller-supplied rays.
        `origins` / `dirs` of shape (N, 3) are re-traced for every sample (shared layout); of shape (sample_count, N, 3) they give
        one ray per sample (per-sample layout).  Ray i is keyed as pixel keys[i] (uint32, default i).  numpy arrays: returns
        (sum (N, 3) f32, stats dict).  torch CUDA tensors on this scene's device: runs fw_trace_rays_device into a new torch
        buffer on a stream of its own and returns (sum tensor (N, 3) f32, stats dict)."""
        n, per_sample = _ray_layout(origins, dirs, sample_count, keys)
        if type(origins).__module__.startswith("torch"):
            import torch
            dev = torch.device("cuda", self.device)
            o = origins.to(dev, torch.float32).contiguous()
            d = dirs.to(dev, torch.float32).contiguous()
            k = None if keys is None else keys.to(dev, torch.int64).to(torch.int32).contiguous()   # uint32 bit patterns
            out = torch.zeros((n, 3), dtype=torch.float32, device=dev)
            # torch's default stream has handle 0, which the C ABI reads as the scene's own stream: use an explicit one
            stream = torch.cuda.Stream(device=dev)
            stream.wait_stream(torch.cuda.current_stream(dev))
            st = self.trace_rays_device(o.data_ptr(), d.data_ptr(), n, out.data_ptr(), stream.cuda_stream, per_sample, sample_count,
                                        sample_begin, seed, use_bvh, 0 if k is None else k.data_ptr())
            torch.cuda.current_stream(dev).wait_stream(stream)
            return out, st
        o = np.ascontiguousarray(origins, np.float32)
        d = np.ascontiguousarray(dirs, np.float32)
        k = None if keys is None else np.ascontiguousarray(keys, np.uint32)
        s = np.empty((n, 3), np.float32)
        st = N.FwStats()
        N.check(N.lib().fw_trace_rays(self._h, n, N.ptr(o), N.ptr(d), None if k is None else N.ptr(k), int(per_sample),
                                      int(sample_begin), int(sample_count), int(seed), 1 if use_bvh else 0, N.ptr(s), C.byref(st)))
        return s, st.as_dict()

    def trace_rays_device(self, d_origins_ptr: int, d_dirs_ptr: int, n: int, d_sum_ptr: int, stream_ptr: int, per_sample=False,
                          sample_count=1, sample_begin=0, seed=0, use_bvh=False, d_keys_ptr: int = 0):
        """fw_trace_rays_device: ADDS the per-ray sums into a device fp32 (n, 3) buffer (e.g. a torch tensor's data_ptr()) on
        `stream_ptr` (0: the scene's own stream)."""
        st = N.FwStats()
        N.check(N.lib().fw_trace_rays_device(self._h, int(n), C.c_void_p(d_origins_ptr), C.c_void_p(d_dirs_ptr),
                                             C.c_void_p(d_keys_ptr) if d_keys_ptr else None, 1 if per_sample else 0, int(sample_begin),
                                             int(sample_count), int(seed), 1 if use_bvh else 0, C.c_void_p(d_sum_ptr),
                                             C.c_void_p(stream_ptr) if stream_ptr else None, C.byref(st)))
        return st.as_dict()

    def resolve_device(self, d_sum_ptr: int, npix: int, samples: int, gamma: float, d_rgb_ptr: int, stream_ptr: int = 0):
        N.check(N.lib().fw_resolve_device(self._h, C.c_void_p(d_sum_ptr), npix, samples, C.c_float(gamma),
                                          C.c_void_p(d_rgb_ptr), C.c_void_p(stream_ptr) if stream_ptr else None))

    # ---- probes ----------------------------------------------------------------------------------------
    def primary_rays(self, params: N.FwParams, sample: int, pix_begin=0, n=None):
        if n is None:
            n = params.width * params.height - pix_begin
        o = np.zeros((n, 3), np.float32)
        d = np.zeros((n, 3), np.float32)
        N.check(N.lib().fw_primary_rays(self._h, C.byref(params), sample, pix_begin, n, N.ptr(o), N.ptr(d)))
        return o, d

    def first_hit(self, origins, dirs, use_bvh: bool, seed=0, pixel=None, sample=None, bounce=None):
        o = np.ascontiguousarray(origins, np.float32)
        d = np.ascontiguousarray(dirs, np.float32)
        n = len(o)
        keys = [None if k is None else np.ascontiguousarray(k, np.uint32) for k in (pixel, sample, bounce)]
        res = {"obj": np.zeros(n, np.int32), "prim": np.zeros(n, np.int32), "material": np.zeros(n, np.int32),
               "t": np.zeros(n, np.float32), "point": np.zeros((n, 3), np.float32),
               "normal": np.zeros((n, 3), np.float32), "uv": np.zeros((n, 2), np.float32)}
        cnt = np.zeros(2, np.uint64)
        N.check(N.lib().fw_first_hit(self._h, 1 if use_bvh else 0, seed, n, N.ptr(o), N.ptr(d),
                                     *[None if k is None else N.ptr(k) for k in keys],
                                     N.ptr(res["obj"]), N.ptr(res["prim"]), N.ptr(res["material"]), N.ptr(res["t"]),
                                     N.ptr(res["point"]), N.ptr(res["normal"]), N.ptr(res["uv"]), N.ptr(cnt)))
        res["node_tests"], res["prim_tests"] = int(cnt[0]), int(cnt[1])
        return res

    def first_hit_wavefront(self, origins, dirs, use_bvh: bool, seed=0, sample=0, bounce=0):
        """The first-hit query through the kernels a render launches (fw_first_hit_wavefront); ray i is keyed as pixel i."""
        o = np.ascontiguousarray(origins, np.float32)
        d = np.ascontiguousarray(dirs, np.float32)
        n = len(o)
        res = {"obj": np.zeros(n, np.int32), "prim": np.zeros(n, np.int32), "material": np.zeros(n, np.int32),
               "t": np.zeros(n, np.float32), "point": np.zeros((n, 3), np.float32),
               "normal": np.zeros((n, 3), np.float32), "uv": np.zeros((n, 2), np.float32)}
        N.check(N.lib().fw_first_hit_wavefront(self._h, 1 if use_bvh else 0, seed, n, N.ptr(o), N.ptr(d), int(sample), int(bounce),
                                               N.ptr(res["obj"]), N.ptr(res["prim"]), N.ptr(res["material"]), N.ptr(res["t"]),
                                               N.ptr(res["point"]), N.ptr(res["normal"]), N.ptr(res["uv"])))
        return res

    def scatter_step(self, material, ray_o, ray_d, hit_t, hit_point, hit_normal, hit_uv, uniforms):
        n = len(material)
        material = np.ascontiguousarray(material, np.int32)
        arrs = [np.ascontiguousarray(a, np.float32) for a in (ray_o, ray_d, hit_t, hit_point, hit_normal, hit_uv)]
        uniforms = np.ascontiguousarray(uniforms, np.float32)
        res = {"emit": np.zeros((n, 3), np.float32), "scattered": np.zeros(n, np.int32),
               "atten": np.zeros((n, 3), np.float32), "o": np.zeros((n, 3), np.float32),
               "d": np.zeros((n, 3), np.float32), "consumed": np.zeros(n, np.int32)}
        N.check(N.lib().fw_scatter_step(self._h, n, N.ptr(material), *[N.ptr(a) for a in arrs], N.ptr(uniforms),
                                        uniforms.shape[1], N.ptr(res["emit"]), N.ptr(res["scattered"]),
                                        N.ptr(res["atten"]), N.ptr(res["o"]), N.ptr(res["d"]), N.ptr(res["consumed"])))
        return res

    def scatter_step_keyed(self, material, ray_o, ray_d, hit_t, hit_point, hit_normal, hit_uv, seed, pixel, sample, bounce):
        """scatter_step drawing from the render's keyed Philox stream; "consumed" counts the uniforms drawn."""
        n = len(material)
        material = np.ascontiguousarray(material, np.int32)
        arrs = [np.ascontiguousarray(a, np.float32) for a in (ray_o, ray_d, hit_t, hit_point, hit_normal, hit_uv)]
        keys = [np.ascontiguousarray(np.broadcast_to(k, (n,)), np.uint32) for k in (pixel, sample, bounce)]
        res = {"emit": np.zeros((n, 3), np.float32), "scattered": np.zeros(n, np.int32),
               "atten": np.zeros((n, 3), np.float32), "o": np.zeros((n, 3), np.float32),
               "d": np.zeros((n, 3), np.float32), "consumed": np.zeros(n, np.int32)}
        N.check(N.lib().fw_scatter_step_keyed(self._h, C.c_uint64(seed), n, N.ptr(material), *[N.ptr(a) for a in arrs],
                                              *[N.ptr(k) for k in keys], N.ptr(res["emit"]), N.ptr(res["scattered"]),
                                              N.ptr(res["atten"]), N.ptr(res["o"]), N.ptr(res["d"]), N.ptr(res["consumed"])))
        return res

    def env_sample(self, dirs):
        d = np.ascontiguousarray(dirs, np.float32)
        out = np.zeros_like(d)
        N.check(N.lib().fw_env_sample(self._h, len(d), N.ptr(d), N.ptr(out)))
        return out

    def texture_sample(self, tex, uv, point):
        uv = np.ascontiguousarray(uv, np.float32)
        pt = np.ascontiguousarray(point, np.float32)
        out = np.zeros_like(pt)
        N.check(N.lib().fw_texture_sample(self._h, int(tex), len(pt), N.ptr(uv), N.ptr(pt), N.ptr(out)))
        return out


def camera_constants(params: N.FwParams) -> np.ndarray:
    out = np.zeros(24, np.float32)
    N.check(N.lib().fw_camera(C.byref(params), N.ptr(out)))
    return out


def measure_peaks(device=0):
    f, l, sm, khz = C.c_double(), C.c_double(), C.c_int(), C.c_int()
    N.check(N.lib().fw_measure_peaks(device, C.byref(f), C.byref(l), C.byref(sm), C.byref(khz)))
    return {"fp32_tflops": f.value, "l2_gbs": l.value, "sm_count": sm.value, "sm_clock_khz": khz.value}


def selftest_shared_division(n_pairs: int, seed: int = 1, device: int = 0):
    """fw_selftest_shared_division: (bit mismatches, tiny-numerator threshold violations); both must be 0."""
    v = np.zeros(2, np.uint64)
    N.check(N.lib().fw_selftest_shared_division(device, C.c_uint64(n_pairs), C.c_uint64(seed), N.ptr(v)))
    return int(v[0]), int(v[1])


def bvh_build(boxes, unbounded=None, device: int = 0) -> dict:
    """fw_bvh_build: one BVH over boxes (n, 6) = (min xyz, max xyz), as a scene build makes each tree; on the host when
    device = -1, else with the sorts and SAH splits on that CUDA device.  Returns items (leaf order), nodes (wide nodes,
    (count, 32) float32), root_box and info {nodes, root_code, wide_depth, max_depth}."""
    b = np.ascontiguousarray(boxes, np.float32).reshape(-1, 6)
    n = b.shape[0]
    u = None if unbounded is None else np.ascontiguousarray(unbounded, np.uint8).reshape(n)
    items = np.empty(max(n, 1), np.int32)
    root = np.empty(6, np.float32)
    info = np.zeros(4, np.int32)
    cap = 2 * n + 1   # the SAH tree has n_leaves - 1 <= n interior nodes; every wide node opens at least one of them
    nodes = np.empty((cap, 32), np.float32)
    N.check(N.lib().fw_bvh_build(int(device), n, N.ptr(b), None if u is None else N.ptr(u), N.ptr(items), N.ptr(nodes), cap,
                                 N.ptr(root), N.ptr(info)))
    return {"items": items[:n], "nodes": nodes[:info[0]].copy(), "root_box": root,
            "info": {"nodes": int(info[0]), "root_code": int(info[1]), "wide_depth": int(info[2]), "max_depth": int(info[3])}}


def texture_store_stats() -> dict:
    """fw_texture_store_stats: commits served from a resident array, uploads, arrays resident now and their bytes."""
    v = np.zeros(4, np.uint64)
    N.check(N.lib().fw_texture_store_stats(N.ptr(v)))
    return {"hits": int(v[0]), "uploads": int(v[1]), "arrays": int(v[2]), "bytes": int(v[3])}


def release_cached_memory():
    N.check(N.lib().fw_release_cached_memory())


def resolve_host(sums: np.ndarray, samples: int, gamma: float, device: int = 0) -> np.ndarray:
    """render.rs:184-189 for a host fp32 sum buffer (H, W, 3) -> u8 image, on the GPU (fw_resolve_host)."""
    s = np.ascontiguousarray(sums, np.float32)
    out = np.empty(s.shape, np.uint8)
    N.check(N.lib().fw_resolve_host(device, N.ptr(s), s.size // 3, int(samples), C.c_float(gamma), N.ptr(out)))
    return out


def denoise(color, variance, albedo, normal, depth, device: int = 0, **settings):
    """fw_denoise_host: the a-trous filter of DESIGN.md §12 on host arrays — color (H,W,3) linear, variance (H,W) of the mean
    luminance, albedo (H,W,3), normal (H,W,3), depth (H,W); `settings` override DENOISE_DEFAULTS (`aov_samples` is checked but
    unused).  Returns (filtered colour (H,W,3), filtered variance (H,W)), float32."""
    c = np.ascontiguousarray(color, np.float32)
    if c.ndim != 3 or c.shape[2] != 3:
        raise ValueError("color must be (height, width, 3)")
    h, w = c.shape[:2]
    v = np.ascontiguousarray(variance, np.float32)
    a = np.ascontiguousarray(albedo, np.float32)
    n = np.ascontiguousarray(normal, np.float32)
    z = np.ascontiguousarray(depth, np.float32)
    if v.shape != (h, w) or a.shape != c.shape or n.shape != c.shape or z.shape != (h, w):
        raise ValueError("variance and depth must be (height, width), albedo and normal (height, width, 3)")
    out_c = np.empty_like(c)
    out_v = np.empty((h, w), np.float32)
    N.check(N.lib().fw_denoise_host(int(device), w, h, N.ptr(c), N.ptr(v), N.ptr(a), N.ptr(n), N.ptr(z),
                                    C.byref(_denoise_settings(settings)), N.ptr(out_c), N.ptr(out_v)))
    return out_c, out_v


def render_scene(scene, renderer, device: int = 0):
    """`Renderer::render(scene)` on one GPU: YAML -> native scene -> fw_render. Returns (rgb, sum, stats)."""
    ns = NativeScene.from_scene(scene, device)
    try:
        return ns.render(renderer.params())
    finally:
        ns.close()
