"""Path tracing of caller-supplied rays (fw_trace_rays, fw_trace_rays_device; DESIGN.md §13): fw_render's own camera rays fed back in
give fw_render's sums bit for bit on every extend path; keys, the shared layout, misses, determinism, the device entry point and the
mirrors are checked exactly, arbitrary rays against the CPU oracle.  Argument checks and the Renderer's refusals need no device."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from conftest import ASSETS, CONFIGS, REPO, native_scene, oracle_scene, params_for, scene_text

F32 = np.float32
U32 = np.uint32


def bits(a):
    return np.ascontiguousarray(a, F32).view(U32)


def camera_rays(ns, p):
    """fw_primary_rays for every sample of p's range, in the per-sample layout (sample_count, npix, 3)."""
    rays = [ns.primary_rays(p, s) for s in range(p.sample_begin, p.sample_begin + p.sample_count)]
    return np.stack([o for o, _ in rays]), np.stack([d for _, d in rays])


# ---- the oracle's trace entry point (tests/trace_oracle.cpp: the unchanged oracle source plus orc_trace_rays) ------------------
@pytest.fixture(scope="module")
def trace_oracle_lib(tmp_path_factory):
    out = str(tmp_path_factory.mktemp("oracle") / "liboracle_trace.so")
    r = subprocess.run(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-fopenmp", "-ffp-contract=off", "-fno-fast-math", "-o", out,
                        os.path.join(REPO, "tests", "trace_oracle.cpp")], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    lib = C.CDLL(out)
    lib.orc_scene_new.restype = C.c_void_p
    lib.orc_trace_rays.argtypes = [C.c_void_p, C.c_uint32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_uint32, C.c_uint32,
                                   C.c_uint64, C.c_int, C.c_void_p]
    return lib


@pytest.fixture
def trace_oracle(trace_oracle_lib, monkeypatch):
    """oracle_scene(name) built in the library that has orc_trace_rays, and its trace call."""
    import oracle.oracle as O
    monkeypatch.setattr(O, "_lib", lambda fast=False: trace_oracle_lib)

    def make(name):
        orc = oracle_scene(name)

        def trace(origins, dirs, sample_count=1, sample_begin=0, seed=0, keys=None):
            o = np.ascontiguousarray(origins, F32)
            d = np.ascontiguousarray(dirs, F32)
            n = o.shape[-2]
            k = None if keys is None else np.ascontiguousarray(keys, U32)
            s = np.zeros((n, 3), F32)
            rc = trace_oracle_lib.orc_trace_rays(orc.h, n, o.ctypes.data, d.ctypes.data, None if k is None else k.ctypes.data,
                                                 1 if o.ndim == 3 else 0, sample_begin, sample_count, seed, 1 if orc.use_bvh else 0,
                                                 s.ctypes.data)
            assert rc == 0
            return s
        orc.trace_rays = trace
        return orc
    return make


def test_oracle_trace_of_camera_rays_is_orc_render(trace_oracle):
    """The oracle's trace entry point keys a path exactly as orc_render does (no device needed)."""
    for name in ("cornell_box", "volume"):
        orc = trace_oracle(name)
        p = params_for(name, 24, 16, 8, seed=3, sample_begin=2, sample_count=3)
        rays = [orc.primary_rays(p, s) for s in range(2, 5)]
        got = orc.trace_rays(np.stack([o for o, _ in rays]), np.stack([d for _, d in rays]), sample_count=3, sample_begin=2, seed=3)
        _, want, _ = orc.render(p, want_rgb=False)
        assert np.array_equal(bits(got), bits(want.reshape(-1, 3))), name


# ---- argument checks: no device needed -----------------------------------------------------------------------------------
def test_trace_arguments_are_checked_before_any_cuda_call():
    from firework_b200 import _native as N
    from firework_b200.engine import NativeScene
    L = N.lib()
    buf = np.zeros(64 * 3, F32)
    P = N.ptr(buf)
    ns = NativeScene(scene_text("cornell_box"), commit=False)
    try:
        h = ns._h
        # (scene, n, origins, dirs, keys, per_sample, sample_begin, sample_count, seed, use_bvh, sum)
        good = [h, 8, P, P, None, 0, 0, 4, 0, 0, P]

        def host(a):
            return L.fw_trace_rays(*a, None)

        def dev(a):
            return L.fw_trace_rays_device(*a, None, None)
        for call in (host, dev):
            for i in (0, 2, 3, 10):                                          # null scene, origins, dirs, sum
                a = list(good)
                a[i] = None
                assert call(a) == -5, (call.__name__, i)
            for field, value in ((1, 0), (1, 1 << 31), (1, 1 << 40), (7, 0), (6, 2), (6, 0xffffffff)):
                a = list(good)
                a[field] = value
                if field == 6:
                    a[7] = 0xffffffff                                        # sample_begin + sample_count > 2^32
                assert call(a) == -5, (call.__name__, field, value)
            assert call(good) == -6                                          # FW_ERR_STATE: not committed
            for field, value in ((1, (1 << 31) - 1), (6, 1)):                # the limits themselves are accepted
                a = list(good)
                a[field] = value
                if field == 6:
                    a[7] = 0xffffffff                                        # sample_begin + sample_count == 2^32
                assert call(a) == -6, (call.__name__, field, value)
        with pytest.raises(ValueError, match="same shape"):
            ns.trace_rays(np.zeros((4, 3), F32), np.zeros((5, 3), F32))
        with pytest.raises(ValueError, match="sample_count"):
            ns.trace_rays(np.zeros((3, 4, 3), F32), np.zeros((3, 4, 3), F32), sample_count=2)
        with pytest.raises(ValueError, match="keys"):
            ns.trace_rays(np.zeros((4, 3), F32), np.zeros((4, 3), F32), keys=np.arange(5, dtype=U32))
    finally:
        ns.close()


def test_renderer_refuses_trace_rays_on_several_gpus_with_adaptive_or_denoise():
    from firework_b200 import scenes
    o = np.zeros((4, 3), F32)
    d = np.ones((4, 3), F32)
    cfg = CONFIGS["cornell_box"]
    for r, what in ((cfg.renderer(samples=4).gpus(2), "one GPU"), (cfg.renderer(samples=4).adaptive(0.1), "adaptive"),
                    (cfg.renderer(samples=4).denoise(), "denoise")):
        with pytest.raises(ValueError, match=what):
            r.trace_rays(scenes.cornell_box(), o, d)


# ---- on the device --------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("name", ["cornell_box", "conics", "random_spheres", "suzanne", "teapot", "volume", "earth", "hdri_test",
                                  "part2_all"])
def test_camera_rays_reproduce_fw_render_bit_for_bit(name):
    w, h = (48, 27) if name == "part2_all" else (40, 30)
    ns = native_scene(name)
    try:
        for begin, count in ((0, 4), (5, 3)):
            p = params_for(name, w, h, 16, seed=3, sample_begin=begin, sample_count=count)
            o, d = camera_rays(ns, p)
            got, st = ns.trace_rays(o, d, sample_count=count, sample_begin=begin, seed=3, use_bvh=p.use_bvh != 0)
            _, want, wst = ns.render(p, want_rgb=False)
            assert np.array_equal(bits(got), bits(want.reshape(-1, 3))), (name, begin, count)
            assert st["samples"] == w * h * count and st["rays"] == wst["rays"]
    finally:
        ns.close()


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["volume", "random_spheres"])
def test_keys_select_the_pixels_of_a_render(name):
    w, h = 40, 30
    ns = native_scene(name)
    try:
        p = params_for(name, w, h, 8, seed=5, sample_count=3)
        o, d = camera_rays(ns, p)
        _, want, _ = ns.render(p, want_rgb=False)
        want = want.reshape(-1, 3)
        yy, xx = np.mgrid[7:19, 11:31]
        pix = (yy * w + xx).reshape(-1).astype(U32)                 # a crop rectangle
        crop, _ = ns.trace_rays(o[:, pix], d[:, pix], sample_count=3, seed=5, use_bvh=p.use_bvh != 0, keys=pix)
        assert np.array_equal(bits(crop), bits(want[pix]))
        perm = np.random.default_rng(1).permutation(len(pix))       # the same rays shuffled, with their keys
        shuf, _ = ns.trace_rays(o[:, pix[perm]], d[:, pix[perm]], sample_count=3, seed=5, use_bvh=p.use_bvh != 0, keys=pix[perm])
        assert np.array_equal(bits(shuf), bits(crop[perm]))
    finally:
        ns.close()


@pytest.mark.gpu
def test_shared_layout_is_the_sum_of_single_sample_calls():
    ns = native_scene("cornell_box")
    try:
        p = params_for("cornell_box", 16, 8, 1, seed=2)
        o, d = ns.primary_rays(p, 0)
        for n in (1, len(o)):
            k = 6
            got, st = ns.trace_rays(o[:n], d[:n], sample_count=k, seed=2)
            acc = np.zeros((n, 3), F32)
            for s in range(k):
                one, _ = ns.trace_rays(o[:n], d[:n], sample_count=1, sample_begin=s, seed=2)
                acc = acc + one
            assert np.array_equal(bits(got), bits(acc)), n
            assert st["samples"] == n * k
        assert np.any(got != 0)
    finally:
        ns.close()


def _arbitrary_rays(ns, n, seed):
    """Origins inside and outside the scene bounds (also inside objects: boxes, media), directions in all octants, axis-aligned
    directions and one NaN direction."""
    rng = np.random.default_rng(seed)
    boxes = ns.object_aabbs()
    boxes = boxes[np.all(np.isfinite(boxes), axis=1) & np.all(np.abs(boxes) < 1e3, axis=1)]
    lo, hi = boxes[:, :3].min(axis=0), boxes[:, 3:].max(axis=0)
    span = hi - lo
    o = lo + span * rng.uniform(-0.3, 1.3, (n, 3))
    inside = rng.integers(0, len(boxes), n // 3)                    # a third start inside some object's box
    b = boxes[inside]
    o[:n // 3] = b[:, :3] + (b[:, 3:] - b[:, :3]) * rng.uniform(0.05, 0.95, (n // 3, 3))
    d = rng.normal(size=(n, 3)) * rng.uniform(0.2, 5.0, (n, 1))
    axes = np.concatenate([np.eye(3), -np.eye(3)])
    d[-60:] = axes[np.arange(60) % 6] * rng.uniform(0.5, 2.0, (60, 1))
    d[-61] = (np.nan, 1.0, 0.0)
    return o.astype(F32), d.astype(F32)


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["cornell_box", "volume", "random_spheres", "suzanne", "conics"])
def test_arbitrary_rays_match_the_oracle(name, trace_oracle):
    ns = native_scene(name)
    orc = trace_oracle(name)
    try:
        o, d = _arbitrary_rays(ns, 3000, seed=len(name))
        keys = np.random.default_rng(4).permutation(1 << 20)[:len(o)].astype(U32)
        for kw in ({"sample_count": 4, "seed": 11}, {"sample_count": 2, "sample_begin": 7, "seed": 11, "keys": keys}):
            got, st = ns.trace_rays(o, d, use_bvh=CONFIGS[name].use_bvh, **kw)
            want = orc.trace_rays(o, d, **kw)
            assert np.array_equal(np.isfinite(got), np.isfinite(want)), kw.keys()
            close = np.all(np.abs(got - want) <= 1e-4 * np.maximum(np.abs(want), 1e-3), axis=1) | np.all(~np.isfinite(want), axis=1)
            assert close.mean() >= 0.995, f"{(~close).sum()} of {len(close)} rays differ"
    finally:
        ns.close()


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["hdri_test", "random_spheres", "cornell_box"])
def test_rays_that_miss_sum_the_environment(name):
    ns = native_scene(name)
    try:
        rng = np.random.default_rng(3)
        up = rng.normal(size=(500, 3)).astype(F32)
        up[:, 1] = np.abs(up[:, 1]) + F32(0.05)
        down = -up
        d = np.concatenate([up, down, [[0, 1, 0], [0, -1, 0], [0, 3, 0], [0, -0.5, 0]]]).astype(F32)
        o = np.full_like(d, F32(-7e3))                                # beside the scene (off every axis-aligned wall's plane) ...
        o[:, 1] = np.where(d[:, 1] > 0, F32(1e5), F32(-1e5))         # ... far above it looking up, far below it looking down
        hit = ns.first_hit(o, d, CONFIGS[name].use_bvh)
        assert np.all(hit["obj"] < 0)                                # every ray really misses
        env = ns.env_sample(d)
        k = 3
        got, _ = ns.trace_rays(o, d, sample_count=k, seed=1, use_bvh=CONFIGS[name].use_bvh)
        acc = np.zeros_like(env)
        for _ in range(k):
            acc = acc + env
        assert np.array_equal(bits(got), bits(acc))
        if name != "cornell_box":
            assert np.all(got > 0)
    finally:
        ns.close()


@pytest.mark.gpu
def test_trace_is_deterministic_and_independent_of_the_batch_geometry():
    ns = native_scene("random_spheres")
    try:
        o, d = _arbitrary_rays(ns, 2000, seed=9)
        ps_o = np.stack([o, o[::-1], o])
        ps_d = np.stack([d, d, d[::-1]])
        keys = np.arange(len(o), dtype=U32)[::-1].copy()
        calls = [dict(origins=o, dirs=d, sample_count=6, seed=4, use_bvh=True),
                 dict(origins=ps_o, dirs=ps_d, sample_count=3, sample_begin=2, seed=4, use_bvh=True, keys=keys)]
        ref = [ns.trace_rays(**c) for c in calls]
        again = [ns.trace_rays(**c) for c in calls]
        ns.set_batch_paths(300)                                      # ray tiles x one-sample chunks
        tiled = [ns.trace_rays(**c) for c in calls]
        ns.set_batch_paths(0)
        for (a, sa), (b, _), (c, _), call in zip(ref, again, tiled, calls):
            assert np.array_equal(a.view(np.uint8), b.view(np.uint8))
            assert np.array_equal(a.view(np.uint8), c.view(np.uint8))
            assert sa["samples"] == len(o) * call["sample_count"]
    finally:
        ns.close()


@pytest.mark.gpu
def test_device_entry_point_adds_into_a_torch_buffer():
    import torch
    ns = native_scene("cornell_box")
    try:
        p = params_for("cornell_box", 32, 24, 8, seed=6, sample_count=4)
        o, d = camera_rays(ns, p)
        keys = np.arange(o.shape[1], dtype=U32) * U32(7) + U32(3)
        want, _ = ns.trace_rays(o, d, sample_count=4, seed=6, keys=keys)
        to, td = torch.from_numpy(o).cuda(), torch.from_numpy(d).cuda()
        tk = torch.from_numpy(keys.astype(np.int64)).cuda()
        got, st = ns.trace_rays(to, td, sample_count=4, seed=6, keys=tk)
        assert got.is_cuda and np.array_equal(bits(got.cpu().numpy()), bits(want))
        assert st["samples"] == o.shape[1] * 4
        buf = torch.zeros((o.shape[1], 3), dtype=torch.float32, device="cuda")
        tk32 = tk.to(torch.int32)
        stream = torch.cuda.Stream()
        stream.wait_stream(torch.cuda.current_stream())
        for k in (1, 2):
            ns.trace_rays_device(to.data_ptr(), td.data_ptr(), o.shape[1], buf.data_ptr(), stream.cuda_stream, per_sample=True,
                                 sample_count=4, seed=6, d_keys_ptr=tk32.data_ptr())
            torch.cuda.current_stream().wait_stream(stream)
            assert np.array_equal(bits(buf.cpu().numpy()), bits(want * F32(k))), k
    finally:
        ns.close()


@pytest.mark.gpu
def test_cpp_mirror_traces_what_the_python_mirror_traces(tmp_path):
    from firework_b200.build import STATIC_LIB
    exe = str(tmp_path / "trace_rays_mirror")
    cuda_lib = os.path.join(os.environ.get("CUDA_HOME", "/usr/local/cuda"), "lib64")
    r = subprocess.run(["g++", "-O1", "-std=c++17", "-Wall", "-Werror", "-ffp-contract=off", "-o", exe,
                        os.path.join(REPO, "tests", "trace_rays_mirror.cpp"), STATIC_LIB, "-L" + cuda_lib, "-lcudart_static", "-lz", "-ldl",
                        "-lpthread", "-lrt"], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    for name in ("cornell_box", "volume"):
        cfg = CONFIGS[name]
        renderer = cfg.renderer(samples=4, seed=8)
        ns = native_scene(name)
        try:
            o, d = _arbitrary_rays(ns, 500, seed=2)
        finally:
            ns.close()
        for oo, dd in ((o, d), (np.stack([o] * 4), np.stack([d, d[::-1], d, d[::-1]]))):
            rays = str(tmp_path / "rays.f32")
            np.concatenate([oo.reshape(-1), dd.reshape(-1)]).astype(F32).tofile(rays)
            out = str(tmp_path / "means.f32")
            r = subprocess.run([exe, cfg.path(), ASSETS, "4", "8", "1" if cfg.use_bvh else "0", str(len(o)), rays, out],
                               capture_output=True, text=True)
            assert r.returncode == 0, r.stderr
            cpp = np.fromfile(out, F32).reshape(-1, 3)
            want = renderer.trace_rays(cfg.load(), oo, dd)
            assert want.shape == (len(o), 3)
            assert np.array_equal(bits(cpp), bits(want)), name
            assert np.array_equal(bits(renderer.last_stats["sum"] / F32(4)), bits(want))
