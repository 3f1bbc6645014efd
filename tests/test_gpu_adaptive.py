"""Adaptive sampling (fw_render_adaptive): a pixel that received k samples holds, bit for bit, the fp32 sum and the u8 value of
fw_render at samples = k; the sample counts and errors are the ones a numpy replay of the schedule and the stop rule gives.
Argument checks and the drivers' refusals need no device; everything else is marked gpu."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import CONFIGS, REPO, native_scene, params_for, scene_text

CAP, MIN = 64, 4


# ---- numpy replay of the schedule and the stop rule (include/firework_b200.h, DESIGN.md §11) ----------------------------
def luminance(rad):
    """Per-sample luminance in fp64 from fp32 radiance (..., 3): (0.2126 r + 0.7152 g) + 0.0722 b."""
    r, g, b = (rad[..., k].astype(np.float64) for k in range(3))
    return (0.2126 * r + 0.7152 * g) + 0.0722 * b


def relative_error(A, B, n, floor):
    n = np.asarray(n, np.float64)
    with np.errstate(divide="ignore", invalid="ignore"):
        mean = A / n
        var = (B - A * mean) / (n - 1.0)
        var = np.where(var < 0.0, 0.0, var)          # max(0, var), NaN kept
        am = np.abs(mean)
        den = np.where(am < floor, floor, am)        # max(|mean|, floor), NaN kept
        return np.sqrt(var / n) / den


def replay(Y, cap, min_samples, threshold, floor):
    """Y: (samples, npix) fp64 luminance.  Returns (counts, err as float32, var at the end, active count per round)."""
    threshold, floor = float(np.float32(threshold)), float(np.float32(floor))   # the device sees the fp32 arguments
    npix = Y.shape[1]
    A, B = np.zeros(npix), np.zeros(npix)
    count = np.zeros(npix, np.uint32)
    active = np.arange(npix)
    n_prev, n = 0, min(min_samples, cap)
    rounds = []
    while True:
        rounds.append(len(active))
        for s in range(n_prev, n):
            y = Y[s, active]
            A[active] = A[active] + y
            B[active] = B[active] + y * y
        count[active] = n
        if n == cap:
            break
        err = relative_error(A[active], B[active], n, floor)
        with np.errstate(invalid="ignore"):
            stop = (n >= 2) & (err <= threshold)
        active = active[~stop]
        if len(active) == 0:
            break
        n_prev, n = n, min(2 * n, cap)
    with np.errstate(divide="ignore", invalid="ignore"):
        var = (B - A * (A / count)) / (count - 1.0)
    return count, relative_error(A, B, count, floor).astype(np.float32), var, rounds


def adaptive_params(name, w, h, cap, seed=3):
    return params_for(name, w, h, cap, seed=seed)


def uniform(ns, name, w, h, k, seed=3):
    rgb, s, _ = ns.render(params_for(name, w, h, k, seed=seed))
    return rgb, s


# ---- argument checks: no device needed ---------------------------------------------------------------------------------
def test_adaptive_arguments_are_checked_before_any_cuda_call():
    from firework_b200 import _native as N
    from firework_b200.engine import NativeScene
    L = N.lib()
    ns = NativeScene(scene_text("cornell_box"), commit=False)
    try:
        def call(p, ad, scene=ns._h):
            return L.fw_render_adaptive(scene, C.byref(p) if p is not None else None, C.byref(ad) if ad is not None else None,
                                        None, None, None, None, None, None)
        good = N.FwAdaptive(4, 0.05, 0.01)
        p = params_for("cornell_box", 16, 16, 32)
        assert call(p, good, scene=None) == -5                              # FW_ERR_ARG
        assert call(None, good) == -5
        assert call(p, None) == -5
        for ad in (N.FwAdaptive(0, 0.05, 0.01), N.FwAdaptive(4, -0.01, 0.01), N.FwAdaptive(4, float("nan"), 0.01),
                   N.FwAdaptive(4, float("inf"), 0.01), N.FwAdaptive(4, 0.05, 0.0), N.FwAdaptive(4, 0.05, -1.0),
                   N.FwAdaptive(4, 0.05, float("nan")), N.FwAdaptive(4, 0.05, float("inf"))):
            assert call(p, ad) == -5, (ad.min_samples, ad.threshold, ad.floor)
        for begin, count in ((1, 31), (0, 16), (4, 32)):                    # the adaptive render owns the sample range
            assert call(params_for("cornell_box", 16, 16, 32, sample_begin=begin, sample_count=count), good) == -5
        for field in ("width", "height", "samples"):
            q = params_for("cornell_box", 16, 16, 32)
            setattr(q, field, 0)
            assert call(q, good) == -5, field
        assert call(p, good) == -6                                          # FW_ERR_STATE: not committed
        assert call(p, N.FwAdaptive(1, 0.0, 1e-6)) == -6                     # limits of the valid range are accepted
    finally:
        ns.close()


def test_drivers_refuse_adaptive_with_checkpoint_chunk_or_several_gpus(tmp_path):
    from firework_b200.build import CLI
    scene = CONFIGS["cornell_box"].path()
    base = [CLI, "--scene-file", scene, "-s", "8", "--target-error", "0.1", "-o", str(tmp_path / "x.png")]
    for extra, what in ((["--checkpoint", str(tmp_path / "a.fwck")], "--checkpoint"), (["--chunk", "4"], "--chunk"),
                        (["--gpus", "2"], "--gpus")):
        r = subprocess.run(base + extra, capture_output=True, text=True)
        assert r.returncode != 0 and what in r.stderr, (extra, r.stderr)
    r = subprocess.run(base[:-4] + ["--target-error", "-1"], capture_output=True, text=True)
    assert r.returncode != 0 and "--target-error" in r.stderr
    assert not os.path.exists(tmp_path / "x.png")
    for extra in (["--checkpoint", str(tmp_path / "b.fwck")], ["--chunk", "4"]):
        r = subprocess.run([sys.executable, "-m", "firework_b200", "--scene-file", scene, "-s", "8", "--target-error", "0.1"] + extra,
                           capture_output=True, text=True, cwd=REPO)
        assert r.returncode != 0 and "--target-error can not be combined" in r.stderr, r.stderr
    assert not os.path.exists(tmp_path / "b.fwck")


def test_renderer_refuses_adaptive_on_several_gpus():
    from firework_b200 import scenes
    r = CONFIGS["cornell_box"].renderer(width=8, height=8, samples=4, seed=0).adaptive(0.1).gpus(2)
    with pytest.raises(ValueError, match="one GPU"):
        r.render(scenes.cornell_box())


# ---- on the device ----------------------------------------------------------------------------------------------------
def _threshold_with_three_counts(ns, p, thresholds):
    for t in thresholds:
        _, _, counts, _, st = ns.render_adaptive(p, t, MIN, want_rgb=False, want_sum=False)
        if len(np.unique(counts)) >= 3:
            return t
    return None


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["cornell_box", "random_spheres", "suzanne", "hdri_test", "volume"])
def test_each_pixel_equals_the_uniform_render_at_its_count(name):
    """The core promise: for every distinct count k, the pixels with count k hold the fw_render(samples = k) sums, bit for bit,
    and its u8 values."""
    w, h = 48, 36
    ns = native_scene(name)
    try:
        p = adaptive_params(name, w, h, CAP)
        t = _threshold_with_three_counts(ns, p, (0.3, 0.2, 0.1, 0.05, 0.02, 0.01))
        assert t is not None, f"{name}: no threshold leaves three distinct sample counts"
        rgb, s, counts, err, st = ns.render_adaptive(p, t, MIN)
        ks = np.unique(counts)
        assert len(ks) >= 3
        assert st["samples"] == int(counts.sum())
        assert st["rounds"] >= 3 and st["active"][0] == w * h
        for k in ks:
            m = counts == k
            urgb, us = uniform(ns, name, w, h, int(k))
            assert np.array_equal(s[m].view(np.uint32), us[m].view(np.uint32)), f"{name}: sums differ at count {k}"
            assert np.array_equal(rgb[m], urgb[m]), f"{name}: u8 differs at count {k}"
    finally:
        ns.close()


@pytest.fixture(scope="module")
def cornell_samples():
    """Every sample's radiance of cornell_box at 64x48: the sum of a one-sample render is that sample."""
    w, h = 64, 48
    ns = native_scene("cornell_box")
    rad = np.empty((CAP, h, w, 3), np.float32)
    for s in range(CAP):
        _, part, _ = ns.render(params_for("cornell_box", w, h, CAP, seed=3, sample_begin=s, sample_count=1), want_rgb=False)
        rad[s] = part
    yield ns, rad
    ns.close()


@pytest.mark.gpu
@pytest.mark.parametrize("threshold,min_samples", [(0.1, MIN), (0.05, 1), (0.02, 8)])
def test_counts_and_errors_match_a_numpy_replay(cornell_samples, threshold, min_samples):
    ns, rad = cornell_samples
    h, w = rad.shape[1:3]
    Y = luminance(rad).reshape(CAP, -1)
    want_counts, want_err, _, rounds = replay(Y, CAP, min_samples, threshold, 0.01)
    _, s, counts, err, st = ns.render_adaptive(adaptive_params("cornell_box", w, h, CAP), threshold, min_samples)
    assert np.array_equal(counts.reshape(-1), want_counts)
    np.testing.assert_array_equal(err.reshape(-1), want_err)
    assert st["active"] == rounds and st["rounds"] == len(rounds)
    assert len(np.unique(counts)) >= 3
    # the sums are the fp32 sums of each pixel's first `count` samples, added in sample order
    acc = np.zeros((h, w, 3), np.float32)
    want_sum = np.zeros((h, w, 3), np.float32)
    for k in range(CAP):
        acc = acc + rad[k]
        want_sum[counts == k + 1] = acc[counts == k + 1]
    assert np.array_equal(s.view(np.uint32), want_sum.view(np.uint32))


@pytest.mark.gpu
def test_limits_of_the_stop_rule(cornell_samples):
    ns, rad = cornell_samples
    h, w = rad.shape[1:3]
    p = adaptive_params("cornell_box", w, h, CAP)
    Y = luminance(rad).reshape(CAP, -1)
    # min_samples == samples: one round, exactly fw_render
    rgb, s, counts, err, st = ns.render_adaptive(p, 0.05, CAP)
    urgb, us = uniform(ns, "cornell_box", w, h, CAP)
    assert st["rounds"] == 1 and np.all(counts == CAP) and st["samples"] == w * h * CAP
    assert np.array_equal(s.view(np.uint32), us.view(np.uint32)) and np.array_equal(rgb, urgb)
    # a huge threshold: every pixel with a finite error stops at min_samples
    _, _, counts, err, _ = ns.render_adaptive(p, 1e30, MIN)
    want, _, _, _ = replay(Y, CAP, MIN, 1e30, 0.01)
    assert np.array_equal(counts.reshape(-1), want)
    assert np.all(counts[np.isfinite(err)] == MIN)
    # threshold 0: only pixels whose variance is exactly 0 stop early (the light is a constant 15)
    _, _, counts, err, _ = ns.render_adaptive(p, 0.0, MIN)
    want, _, var, _ = replay(Y, CAP, MIN, 0.0, 0.01)
    assert np.array_equal(counts.reshape(-1), want)
    early = counts.reshape(-1) < CAP
    assert early.any() and np.all(var[early] == 0.0) and np.all(err.reshape(-1)[early] == 0.0)
    # min_samples = 1: the first round gives no estimate (n = 1), the second one decides
    _, _, counts, err, st = ns.render_adaptive(p, 0.1, 1)
    want, want_err, _, rounds = replay(Y, CAP, 1, 0.1, 0.01)
    assert np.array_equal(counts.reshape(-1), want) and st["active"][:2] == [w * h, w * h]
    np.testing.assert_array_equal(err.reshape(-1), want_err)


@pytest.mark.gpu
def test_results_do_not_depend_on_the_launch_geometry():
    """Pixel tiles and sample chunks over the active list (small batches), a list that is not a multiple of 128 and a list of one
    pixel give the same pixels as the default batch; two runs are identical."""
    from firework_b200.engine import NativeScene
    w, h = 37, 29                                          # 1073 pixels
    ns = native_scene("random_spheres")
    try:
        p = adaptive_params("random_spheres", w, h, CAP)
        ref = ns.render_adaptive(p, 0.05, MIN)
        again = ns.render_adaptive(p, 0.05, MIN)
        assert any(a % 128 for a in ref[4]["active"]) and len(np.unique(ref[2])) >= 3
        for paths in (1000, 300, 32):                      # tiles of the list x one sample per batch ... chunks of samples
            ns.set_batch_paths(paths)
            got = ns.render_adaptive(p, 0.05, MIN)
            for a, b in zip(ref[:4], got[:4]):
                assert np.array_equal(a.view(np.uint8), b.view(np.uint8)), paths
            assert got[4]["active"] == ref[4]["active"]
        ns.set_batch_paths(0)
        for a, b in zip(ref[:4], again[:4]):
            assert np.array_equal(a.view(np.uint8), b.view(np.uint8))
    finally:
        ns.close()
    # one pixel: the active list has one entry in every round (the sky behind random_spheres never gives two equal samples of a
    # pixel that spans the whole view, so threshold 0 keeps it going to the cap)
    ns = NativeScene(scene_text("random_spheres"))
    try:
        p = adaptive_params("random_spheres", 1, 1, 32)
        rgb, s, counts, err, st = ns.render_adaptive(p, 0.0, 2)
        assert set(st["active"]) == {1} and st["rounds"] == 5 and counts[0, 0] == 32   # 2, 4, 8, 16, 32
        urgb, us = uniform(ns, "random_spheres", 1, 1, 32)
        assert np.array_equal(s.view(np.uint32), us.view(np.uint32)) and np.array_equal(rgb, urgb)
    finally:
        ns.close()


@pytest.mark.gpu
def test_native_and_python_drivers_write_the_same_adaptive_png(tmp_path):
    from PIL import Image
    from firework_b200.__main__ import main
    from firework_b200.build import CLI
    scene = CONFIGS["conics"].path()
    args = ["--scene-file", scene, "-s", "32", "--target-error", "0.1", "--min-samples", "4", "--width", "160", "--height", "90",
            "--seed", "11"]
    out_native, out_py = str(tmp_path / "native.png"), str(tmp_path / "py.png")
    r = subprocess.run([CLI] + args + ["-o", out_native], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    assert "Adaptive: " in r.stdout and "spp mean (cap 32)" in r.stdout
    assert main(args + ["-o", out_py]) == 0
    a = np.asarray(Image.open(out_native).convert("RGB"))
    b = np.asarray(Image.open(out_py).convert("RGB"))
    assert a.shape == (90, 160, 3) and np.array_equal(a, b) and a.std() > 5


@pytest.mark.gpu
def test_cpp_mirror_renders_what_the_python_mirror_renders_adaptively(tmp_path):
    from PIL import Image
    from test_host import _build_example
    from firework_b200 import scenes
    exe = _build_example("cornell_box", tmp_path)
    out = str(tmp_path / "cb.png")
    r = subprocess.run([exe, "-s", "32", "--width", "72", "--height", "64", "--seed", "5", "--target-error", "0.1", "--min-samples", "4",
                        "-o", out], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    renderer = CONFIGS["cornell_box"].renderer(width=72, height=64, samples=32, seed=5).adaptive(0.1, 4)
    want = renderer.render(scenes.cornell_box())
    assert np.array_equal(np.asarray(Image.open(out).convert("RGB")), want)
    counts = renderer.last_stats["counts"]
    assert counts.min() >= 4 and counts.max() <= 32 and len(np.unique(counts)) >= 2
