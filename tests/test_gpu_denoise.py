"""Denoised renders (fw_render_aov, fw_denoise_host, fw_render_denoised; DESIGN.md §12): the AOVs equal, bit for bit, a numpy build
from the first-hit probe of the same rays; the filter equals a numpy float32 replay of its definition; the denoised render is the
composition of fw_render's sums, the moments' variance, the AOV pass and the filter.  Argument checks and the drivers' refusals
need no device; everything else is marked gpu."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import CONFIGS, REPO, native_scene, params_for, scene_doc, scene_text

F32 = np.float32
MAT_KIND = {"LambertianMat": 0, "MetalMat": 1, "DielectricMat": 2, "EmissiveMat": 3, "IsotropicMat": 4}


# ---- numpy builds of the AOVs and the filter -----------------------------------------------------------------------------
def _mag(v):
    return np.sqrt((v[:, 0] * v[:, 0] + v[:, 1] * v[:, 1]) + v[:, 2] * v[:, 2])


def aov_reference(ns, name, p):
    """The AOVs of p's sample range from fw_primary_rays -> fw_first_hit_wavefront (ray i = pixel i) and fw_texture_sample."""
    mats = scene_doc(name)["materials"]
    npix = p.width * p.height
    acc_a, acc_n, acc_z = np.zeros((npix, 3), F32), np.zeros((npix, 3), F32), np.zeros(npix, F32)
    obj0 = None
    for s in range(p.sample_begin, p.sample_begin + p.sample_count):
        o, d = ns.primary_rays(p, s)
        r = ns.first_hit_wavefront(o, d, p.use_bvh != 0, seed=p.seed, sample=s, bounce=0)
        hit = r["obj"] >= 0
        albedo = np.ones((npix, 3), F32)                    # dielectric, emissive, miss
        for m in np.unique(r["material"][hit]):
            sel = hit & (r["material"] == m)
            kind = MAT_KIND[mats[m]["material"]]
            if kind in (0, 4):                               # Lambertian, isotropic: the texture at the hit
                albedo[sel] = ns.texture_sample(ns.material_texture(int(m)), r["uv"][sel], r["point"][sel])
            elif kind == 1:                                  # metal: its albedo
                a = mats[m]["albedo"]
                albedo[sel] = np.array([a["x"], a["y"], a["z"]], F32)
        normal = np.zeros((npix, 3), F32)
        nh = r["normal"][hit]
        normal[hit] = nh / _mag(nh)[:, None]
        depth = np.zeros(npix, F32)
        depth[hit] = r["t"][hit] * _mag(d[hit])
        if obj0 is None:
            obj0 = r["obj"].copy()
        acc_a, acc_n, acc_z = acc_a + albedo, acc_n + normal, acc_z + depth
    n = F32(p.sample_count)
    h, w = p.height, p.width
    return {"albedo": (acc_a / n).reshape(h, w, 3), "normal": (acc_n / n).reshape(h, w, 3), "depth": (acc_z / n).reshape(h, w),
            "object": obj0.reshape(h, w)}


K1 = np.array([1 / 16, 1 / 4, 3 / 8, 1 / 4, 1 / 16], F32)
G1 = np.array([1 / 4, 1 / 2, 1 / 4], F32)


def _lum(c):
    return (F32(0.2126) * c[..., 0] + F32(0.7152) * c[..., 1]) + F32(0.0722) * c[..., 2]


def _tap(a, oy, ox, fill):
    """a[y + oy, x + ox] for every (y, x), `fill` outside the image, and the in-image mask."""
    h, w = a.shape[:2]
    out = np.full_like(a, fill)
    inb = np.zeros((h, w), bool)
    ys, ye = max(0, -oy), min(h, h - oy)
    xs, xe = max(0, -ox), min(w, w - ox)
    if ys < ye and xs < xe:
        out[ys:ye, xs:xe] = a[ys + oy:ye + oy, xs + ox:xe + ox]
        inb[ys:ye, xs:xe] = True
    return out, inb


def atrous_reference(color, variance, albedo, normal, depth, iterations=5, sigma_luminance=4.0, sigma_depth=0.1, sigma_albedo=0.1):
    """numpy float32 replay of DESIGN.md §12 (tap order dy outer, dx inner; every sum in that order)."""
    sl, sz, sa = F32(sigma_luminance), F32(sigma_depth), F32(sigma_albedo)
    eps = F32(1e-6)
    c = np.concatenate([color.astype(F32), variance.astype(F32)[..., None]], axis=-1)
    nz = np.concatenate([normal.astype(F32), depth.astype(F32)[..., None]], axis=-1)
    alb = albedo.astype(F32)
    np_zero = np.all(nz[..., :3] == 0, axis=-1)
    with np.errstate(all="ignore"):
        for it in range(iterations):
            step = 1 << it
            finite = np.all(np.isfinite(c), axis=-1)
            gs, gw = np.zeros(c.shape[:2], F32), np.zeros(c.shape[:2], F32)
            for dy in (-1, 0, 1):
                for dx in (-1, 0, 1):
                    q, inb = _tap(c, dy, dx, 0)
                    ok = inb & _tap(finite, dy, dx, False)[0]
                    wg = G1[dx + 1] * G1[dy + 1]
                    gs = np.where(ok, gs + wg * q[..., 3], gs)
                    gw = np.where(ok, gw + wg, gw)
            den_l = sl * np.sqrt(gs / gw) + eps
            lp = _lum(c)
            sw = np.zeros(c.shape[:2], F32)
            s = np.zeros(c.shape, F32)
            for dy in range(-2, 3):
                for dx in range(-2, 3):
                    q, inb = _tap(c, step * dy, step * dx, 0)
                    ok = inb & _tap(finite, step * dy, step * dx, False)[0]
                    if dx == 0 and dy == 0:
                        wt = np.full(c.shape[:2], F32(9 / 64))
                    else:
                        nq, _ = _tap(nz, step * dy, step * dx, 0)
                        aq, _ = _tap(alb, step * dy, step * dx, 0)
                        wl = np.exp(-np.abs(lp - _lum(q)) / den_l)
                        wn = np.fmax((nz[..., 0] * nq[..., 0] + nz[..., 1] * nq[..., 1]) + nz[..., 2] * nq[..., 2], F32(0))
                        for _ in range(7):
                            wn = wn * wn
                        wn = np.where(np_zero & np.all(nq[..., :3] == 0, axis=-1), F32(1), wn)
                        wz = np.exp(-np.abs(nz[..., 3] - nq[..., 3]) / (sz * np.fmax(nz[..., 3], nq[..., 3]) + eps))
                        da = alb - aq
                        wa = np.exp(-((da[..., 0] * da[..., 0] + da[..., 1] * da[..., 1]) + da[..., 2] * da[..., 2]) / (sa * sa))
                        wt = K1[dx + 2] * K1[dy + 2]
                        wt = wt * wl
                        wt = wt * wn
                        wt = wt * wz
                        wt = wt * wa
                    sw = np.where(ok, sw + wt, sw)
                    s[..., :3] = np.where(ok[..., None], s[..., :3] + wt[..., None] * q[..., :3], s[..., :3])
                    s[..., 3] = np.where(ok, s[..., 3] + (wt * wt) * q[..., 3], s[..., 3])
            new = np.concatenate([s[..., :3] / sw[..., None], (s[..., 3] / (sw * sw))[..., None]], axis=-1)
            c = np.where(finite[..., None], new, c)
    return c[..., :3], c[..., 3]


def luminance(rad):
    r, g, b = (rad[..., k].astype(np.float64) for k in range(3))
    return (0.2126 * r + 0.7152 * g) + 0.0722 * b


def variance_of_mean(rad):
    """rad: (n, ...) fp32 per-sample radiance -> fp32 variance of the mean luminance from fp64 moments in sample order."""
    n = rad.shape[0]
    A = np.zeros(rad.shape[1:-1])
    B = np.zeros(rad.shape[1:-1])
    for k in range(n):
        y = luminance(rad[k])
        A = A + y
        B = B + y * y
    var = (B - A * (A / n)) / (n - 1.0)
    var = np.where(var < 0.0, 0.0, var)
    return (var / n).astype(F32)


def synthetic(h, w, seed=0):
    """An image with hard edges in every guide: normals by column band, depth by row band, albedo in blocks, misses in a corner."""
    rng = np.random.default_rng(seed)
    yy, xx = np.mgrid[0:h, 0:w]
    normal = np.zeros((h, w, 3), F32)
    normal[xx < w // 2] = (0, 0, 1)
    normal[xx >= w // 2] = (0.6, 0, 0.8)
    depth = np.where(yy < h // 2, F32(2.0), F32(7.5)).astype(F32)
    albedo = np.where(((yy // 5 + xx // 7) % 2 == 0)[..., None], F32(0.8), F32(0.2)).astype(F32) * np.array([1.0, 0.7, 0.4], F32)
    miss = (yy < h // 4) & (xx < w // 4)
    normal[miss] = 0
    depth[miss] = 0
    albedo[miss] = 1
    base = albedo * (F32(0.5) + F32(0.5) * (xx / max(w, 1)).astype(F32)[..., None])
    color = (base + rng.normal(0, 0.15, (h, w, 3)).astype(F32)).astype(F32)
    variance = rng.uniform(0, 0.02, (h, w)).astype(F32)
    variance[rng.random((h, w)) < 0.2] = 0                  # zero-variance pixels, as a few-sample render has
    return color, variance, albedo.astype(F32), normal, depth.astype(F32)


# ---- argument checks: no device needed ---------------------------------------------------------------------------------
def test_denoise_arguments_are_checked_before_any_cuda_call():
    from firework_b200 import _native as N
    from firework_b200.engine import NativeScene
    L = N.lib()
    good = N.FwDenoise(5, 4, 4.0, 0.1, 0.1)
    bad = [N.FwDenoise(0, 4, 4.0, 0.1, 0.1), N.FwDenoise(11, 4, 4.0, 0.1, 0.1), N.FwDenoise(5, 0, 4.0, 0.1, 0.1)]
    for k in range(3):
        for v in (float("nan"), float("inf"), 0.0, -1.0):
            sig = [4.0, 0.1, 0.1]
            sig[k] = v
            bad.append(N.FwDenoise(5, 4, *sig))
    buf = np.zeros(64 * 3, np.float32)
    P = N.ptr(buf)
    # fw_denoise_host: null pointers, empty image, every bad setting
    args = [0, 8, 8, P, P, P, P, P, C.byref(good), P, None]
    for i in (3, 4, 5, 6, 7, 8, 9):
        a = list(args)
        a[i] = None
        assert L.fw_denoise_host(*a) == -5, i
    for wh in ((0, 8), (8, 0)):
        assert L.fw_denoise_host(0, *wh, *args[3:]) == -5
    for s in bad:
        assert L.fw_denoise_host(0, 8, 8, P, P, P, P, P, C.byref(s), P, None) == -5, (s.iterations, s.aov_samples, s.sigma_luminance)
    ns = NativeScene(scene_text("cornell_box"), commit=False)
    try:
        p = params_for("cornell_box", 16, 16, 32)
        aov = N.FwAov()

        def den(pp, dn, scene=ns._h):
            return L.fw_render_denoised(scene, C.byref(pp) if pp is not None else None, C.byref(dn) if dn is not None else None,
                                        None, None, None, None, None, None)
        assert den(p, good, scene=None) == -5
        assert den(None, good) == -5
        assert den(p, None) == -5
        for s in bad:
            assert den(p, s) == -5
        for samples, begin, count in ((1, 0, 1), (32, 1, 31), (32, 0, 16), (32, 4, 32)):   # samples >= 2 and the whole range
            assert den(params_for("cornell_box", 16, 16, samples, sample_begin=begin, sample_count=count), good) == -5
        for field in ("width", "height", "samples"):
            q = params_for("cornell_box", 16, 16, 32)
            setattr(q, field, 0)
            assert den(q, good) == -5, field
            assert L.fw_render_aov(ns._h, C.byref(q), C.byref(aov), None) == -5, field
        assert den(p, good) == -6                                                       # FW_ERR_STATE: not committed
        assert den(params_for("cornell_box", 16, 16, 2), N.FwDenoise(10, 1, 1e-3, 1e-3, 1e-3)) == -6   # limits are accepted
        assert L.fw_render_aov(None, C.byref(p), C.byref(aov), None) == -5
        assert L.fw_render_aov(ns._h, None, C.byref(aov), None) == -5
        assert L.fw_render_aov(ns._h, C.byref(p), None, None) == -5
        assert L.fw_render_aov(ns._h, C.byref(params_for("cornell_box", 16, 16, 32, sample_count=0)), C.byref(aov), None) == -5
        assert L.fw_render_aov(ns._h, C.byref(p), C.byref(aov), None) == -6
    finally:
        ns.close()


def test_drivers_refuse_denoise_with_checkpoint_chunk_gpus_or_target_error(tmp_path):
    from firework_b200.build import CLI
    scene = CONFIGS["cornell_box"].path()
    base = [CLI, "--scene-file", scene, "-s", "8", "--denoise", "-o", str(tmp_path / "x.png")]
    for extra, what in ((["--checkpoint", str(tmp_path / "a.fwck")], "--checkpoint"), (["--chunk", "4"], "--chunk"),
                        (["--gpus", "2"], "--gpus"), (["--target-error", "0.1"], "--target-error")):
        r = subprocess.run(base + extra, capture_output=True, text=True)
        assert r.returncode != 0 and what in r.stderr, (extra, r.stderr)
    r = subprocess.run([CLI, "--scene-file", scene, "-s", "1", "--denoise", "-o", str(tmp_path / "x.png")], capture_output=True, text=True)
    assert r.returncode != 0 and "--samples >= 2" in r.stderr
    assert not os.path.exists(tmp_path / "x.png")
    for extra in (["--checkpoint", str(tmp_path / "b.fwck")], ["--chunk", "4"], ["--target-error", "0.1"]):
        r = subprocess.run([sys.executable, "-m", "firework_b200", "--scene-file", scene, "-s", "8", "--denoise"] + extra,
                           capture_output=True, text=True, cwd=REPO)
        assert r.returncode != 0 and "--denoise can not be combined" in r.stderr, r.stderr
    assert not os.path.exists(tmp_path / "b.fwck")


def test_renderer_refuses_denoise_on_several_gpus_or_with_adaptive():
    from firework_b200 import scenes
    r = CONFIGS["cornell_box"].renderer(width=8, height=8, samples=4, seed=0).denoise().gpus(2)
    with pytest.raises(ValueError, match="one GPU"):
        r.render(scenes.cornell_box())
    r = CONFIGS["cornell_box"].renderer(width=8, height=8, samples=4, seed=0).adaptive(0.1).denoise()
    with pytest.raises(ValueError, match="adaptive"):
        r.render(scenes.cornell_box())


# ---- on the device ----------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("name", ["cornell_box", "random_spheres", "suzanne", "earth", "volume", "hdri_test"])
def test_aovs_equal_a_numpy_build_from_the_first_hit_probe(name):
    w, h = 40, 30
    ns = native_scene(name)
    try:
        for begin, count in ((0, 1), (0, 4), (5, 4)):
            p = params_for(name, w, h, 16, seed=3, sample_begin=begin, sample_count=count)
            got, st = ns.render_aov(p)
            want = aov_reference(ns, name, p)
            assert st["samples"] == w * h * count
            for k in ("albedo", "normal", "depth", "object"):
                assert np.array_equal(got[k].view(np.uint32), want[k].view(np.uint32)), (name, begin, count, k)
        if name == "hdri_test":
            assert (got["object"] < 0).any()
    finally:
        ns.close()


@pytest.mark.gpu
@pytest.mark.parametrize("h,w,iterations", [(37, 53, 5), (37, 53, 1), (37, 53, 10), (1, 1, 5), (1, 70, 5), (70, 1, 5), (20, 300, 3)])
def test_filter_matches_a_numpy_replay(h, w, iterations):
    from firework_b200.engine import denoise
    color, variance, albedo, normal, depth = synthetic(h, w, seed=h * 1000 + w)
    settings = {"iterations": iterations, "sigma_luminance": 4.0, "sigma_depth": 0.1, "sigma_albedo": 0.1}
    got_c, got_v = denoise(color, variance, albedo, normal, depth, **settings)
    want_c, want_v = atrous_reference(color, variance, albedo, normal, depth, **settings)
    np.testing.assert_allclose(got_c, want_c, rtol=1e-4, atol=1e-6)
    np.testing.assert_allclose(got_v, want_v, rtol=1e-4, atol=1e-6)
    if h * w > 100:
        assert np.abs(got_c - color).max() > 1e-3                    # the filter did something


@pytest.mark.gpu
def test_filter_non_finite_taps_and_centres():
    from firework_b200.engine import denoise
    h, w = 33, 47
    color, variance, albedo, normal, depth = synthetic(h, w, seed=7)
    rng = np.random.default_rng(1)
    bad = rng.random((h, w)) < 0.05
    vals = np.array([np.nan, np.inf, -np.inf], F32)
    color[bad, rng.integers(0, 3, bad.sum())] = vals[rng.integers(0, 3, bad.sum())]
    badv = (rng.random((h, w)) < 0.03) & ~bad
    variance[badv] = vals[rng.integers(0, 3, badv.sum())]
    for settings in ({"iterations": 5}, {"iterations": 2, "sigma_luminance": 0.5, "sigma_depth": 2.0, "sigma_albedo": 3.0}):
        got_c, got_v = denoise(color, variance, albedo, normal, depth, **settings)
        want_c, want_v = atrous_reference(color, variance, albedo, normal, depth, **settings)
        np.testing.assert_allclose(got_c, want_c, rtol=1e-4, atol=1e-6)
        np.testing.assert_allclose(got_v, want_v, rtol=1e-4, atol=1e-6)
        centre = bad | badv                                         # non-finite centres pass through unchanged
        assert np.array_equal(got_c[centre], color[centre], equal_nan=True)
        assert np.array_equal(got_v[centre], variance[centre], equal_nan=True)
        assert np.all(np.isfinite(got_c[~centre])) and np.all(np.isfinite(got_v[~centre]))


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["cornell_box", "suzanne"])
def test_denoised_render_is_the_composition_of_its_parts(name):
    from firework_b200.engine import DENOISE_DEFAULTS, denoise, resolve_host
    w, h, n = 48, 36, 8
    ns = native_scene(name)
    try:
        p = params_for(name, w, h, n, seed=5)
        rgb, s, den, var, aov, st = ns.render_denoised(p)
        _, us, _ = ns.render(p)
        assert np.array_equal(s.view(np.uint32), us.view(np.uint32))
        rad = np.stack([ns.render(params_for(name, w, h, n, seed=5, sample_begin=k, sample_count=1), want_rgb=False)[1]
                        for k in range(n)])
        assert np.array_equal(var.view(np.uint32), variance_of_mean(rad).view(np.uint32))
        want_aov, _ = ns.render_aov(params_for(name, w, h, n, seed=5, sample_count=DENOISE_DEFAULTS["aov_samples"]))
        for k in want_aov:
            assert np.array_equal(aov[k].view(np.uint32), want_aov[k].view(np.uint32)), k
        want_den, _ = denoise(s / F32(n), var, aov["albedo"], aov["normal"], aov["depth"], **DENOISE_DEFAULTS)
        assert np.array_equal(den.view(np.uint32), want_den.view(np.uint32))
        assert np.array_equal(rgb, resolve_host(den, 1, p.gamma))
        assert st["samples"] == w * h * n
        # aov_samples above samples: the AOVs cover [0, samples)
        _, _, _, _, aov2, _ = ns.render_denoised(params_for(name, w, h, 2, seed=5), aov_samples=16, iterations=1)
        want2, _ = ns.render_aov(params_for(name, w, h, 2, seed=5))
        assert np.array_equal(aov2["depth"].view(np.uint32), want2["depth"].view(np.uint32))
    finally:
        ns.close()


@pytest.mark.gpu
@pytest.mark.parametrize("name,w,h", [("cornell_box", 128, 128), ("suzanne", 160, 90)])
def test_denoising_lowers_the_error_against_a_converged_render(name, w, h):
    ns = native_scene(name)
    try:
        _, ref_sum, _ = ns.render(params_for(name, w, h, 1024, seed=9), want_rgb=False)
        ref = ref_sum.astype(np.float64) / 1024
        _, s, den, _, _, _ = ns.render_denoised(params_for(name, w, h, 16, seed=1), want_rgb=False)
        noisy = np.sqrt(np.mean((s.astype(np.float64) / 16 - ref) ** 2))
        filtered = np.sqrt(np.mean((den.astype(np.float64) - ref) ** 2))
        assert filtered < noisy, (name, filtered, noisy)
    finally:
        ns.close()


@pytest.mark.gpu
def test_denoised_outputs_are_deterministic_and_independent_of_the_batch_geometry():
    ns = native_scene("random_spheres")
    try:
        p = params_for("random_spheres", 37, 29, 8, seed=2)
        ref = ns.render_denoised(p)
        again = ns.render_denoised(p)
        ns.set_batch_paths(300)                  # pixel tiles x one sample per batch, for the render and the AOV pass
        tiled = ns.render_denoised(p)
        ns.set_batch_paths(0)
        for got in (again, tiled):
            for a, b in zip(ref[:4], got[:4]):
                assert np.array_equal(a.view(np.uint8), b.view(np.uint8))
            for k in ref[4]:
                assert np.array_equal(ref[4][k].view(np.uint8), got[4][k].view(np.uint8)), k
    finally:
        ns.close()


@pytest.mark.gpu
def test_native_and_python_drivers_write_the_same_denoised_png(tmp_path):
    from PIL import Image
    from firework_b200.__main__ import main
    from firework_b200.build import CLI
    scene = CONFIGS["conics"].path()
    args = ["--scene-file", scene, "-s", "8", "--denoise", "--width", "160", "--height", "90", "--seed", "11"]
    out_native, out_py = str(tmp_path / "native.png"), str(tmp_path / "py.png")
    r = subprocess.run([CLI] + args + ["-o", out_native], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    assert main(args + ["-o", out_py]) == 0
    a = np.asarray(Image.open(out_native).convert("RGB"))
    b = np.asarray(Image.open(out_py).convert("RGB"))
    assert a.shape == (90, 160, 3) and np.array_equal(a, b) and a.std() > 5


@pytest.mark.gpu
def test_cpp_mirror_renders_what_the_python_mirror_renders_denoised(tmp_path):
    from PIL import Image
    from test_host import _build_example
    from firework_b200 import scenes
    exe = _build_example("cornell_box", tmp_path)
    out = str(tmp_path / "cb.png")
    r = subprocess.run([exe, "-s", "8", "--width", "72", "--height", "64", "--seed", "5", "--denoise", "-o", out],
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    renderer = CONFIGS["cornell_box"].renderer(width=72, height=64, samples=8, seed=5).denoise()
    want = renderer.render(scenes.cornell_box())
    assert np.array_equal(np.asarray(Image.open(out).convert("RGB")), want)
    assert renderer.last_stats["denoised"].shape == (64, 72, 3)
