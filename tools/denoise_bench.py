"""What the denoiser buys, measured: uniform renders at 16 / 64 / 256 spp against denoised renders (fw_render_denoised, default
settings) at the same spp, each compared with a 4096-spp uniform reference (RMSE of the linear per-pixel mean), with device time;
the AOV pass and the filter timed on their own; the fraction of pixels whose variance estimate is exactly 0 at 16 spp.

    python tools/denoise_bench.py [--out profiles/denoise_bench.json] [--ref-spp 4096] [--scenes cornell_box,part2_all,suzanne]

equal_error_time_ratio = (device ms a uniform render needs for the same RMSE) / (denoised device ms): > 1 means the denoised render is
faster at equal error.  The uniform time at a given RMSE comes from a least-squares fit of log(ms) against log(RMSE) over the
uniform renders of the scene (`in_range` says whether that is an interpolation).  The filter's kernel time is the sum of its
kernels' durations in a torch.profiler trace of one fw_denoise_host call (the call's host copies are not part of it); it is also
taken at 3840x2160.  The card's name and power limit are read in the same run."""
import argparse
import gzip
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from firework_b200.engine import DENOISE_DEFAULTS, NativeScene, denoise  # noqa: E402
from firework_b200.scenes import CONFIGS, SCENE_DIR  # noqa: E402

SIZES = {"cornell_box": (300, 300), "part2_all": (1920, 1080), "suzanne": (1920, 1080)}
SPP = (16, 64, 256)


def card():
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=30)
        name, power, clock = [x.strip() for x in r.stdout.strip().splitlines()[0].split(",")]
        return {"name": name, "power_limit": power, "max_sm_clock": clock}
    except Exception as e:  # the numbers still stand, without the card's description
        return {"error": str(e)}


def rmse(mean, ref):
    d = mean.astype(np.float64) - ref
    return float(np.sqrt(np.mean(d * d)))


def filter_kernel_ms(args, reps=3):
    """Sum of the filter's kernel durations (pack, a-trous iterations, unpack) of one fw_denoise_host call, best of `reps`."""
    try:
        from torch.profiler import ProfilerActivity, profile
    except Exception as e:
        return {"error": f"torch.profiler unavailable: {e}"}
    denoise(*args)                                                         # warm-up
    best = None
    for _ in range(reps):
        c0 = time.perf_counter()
        denoise(*args)
        wall = (time.perf_counter() - c0) * 1e3
        try:
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                denoise(*args)
            kern = {}
            for ev in prof.key_averages():
                if "atrous" in ev.key or "denoise_" in ev.key:
                    t = getattr(ev, "device_time_total", None)
                    kern[ev.key] = (t if t is not None else ev.cuda_time_total) / 1e3
        except Exception as e:
            return {"error": f"profiler: {e}", "wall_ms_with_copies": wall}
        tot = sum(kern.values())
        if best is None or tot < best["ms"]:
            best = {"ms": tot, "atrous_ms": sum(v for k, v in kern.items() if "atrous" in k), "kernels": kern,
                    "wall_ms_with_copies": wall}
    return best


def prefiltered(v):
    """The filter's 3x3 Gaussian of the variance (outside taps dropped, weights renormalised); every tap is finite here."""
    h, w = v.shape
    g1 = np.array([0.25, 0.5, 0.25])
    s, wsum = np.zeros((h, w)), np.zeros((h, w))
    for dy in (-1, 0, 1):
        for dx in (-1, 0, 1):
            ys, ye, xs, xe = max(0, -dy), min(h, h - dy), max(0, -dx), min(w, w - dx)
            s[ys:ye, xs:xe] += g1[dx + 1] * g1[dy + 1] * v[ys + dy:ye + dy, xs + dx:xe + dx]
            wsum[ys:ye, xs:xe] += g1[dx + 1] * g1[dy + 1]
    return s / wsum


def run_scene(name, ref_spp):
    cfg = CONFIGS[name]
    w, h = SIZES[name]
    p = cfg.path()
    text = (gzip.open(p, "rt") if p.endswith(".gz") else open(p)).read()
    ns = NativeScene(text, asset_dir=os.path.join(SCENE_DIR, "assets"))

    def params(spp, count=None):
        return cfg.renderer(width=w, height=h, samples=spp, seed=1).params(sample_count=count)

    t0 = time.time()
    _, ref_sum, st = ns.render(params(ref_spp), want_rgb=False)
    ref = ref_sum.astype(np.float64) / ref_spp
    out = {"size": [w, h], "ref_spp": ref_spp, "ref_ms": st["ms_device"], "uniform": [], "denoised": []}
    ns.render(params(SPP[0]), want_rgb=False)                              # warm-up
    for spp in SPP:
        best = None
        for _ in range(2):
            _, s, st = ns.render(params(spp), want_rgb=False)
            best = st["ms_device"] if best is None else min(best, st["ms_device"])
        out["uniform"].append({"spp": spp, "ms": best, "rmse": rmse(s / spp, ref)})
    ns.render_denoised(params(SPP[0]), want_rgb=False)                     # warm-up
    for spp in SPP:
        best = None
        for _ in range(2):
            _, s, den, var, aov, st = ns.render_denoised(params(spp), want_rgb=False)
            best = st["ms_device"] if best is None else min(best, st["ms_device"])
        noisy = s / np.float32(spp)
        r = {"spp": spp, "ms": best, "rmse": rmse(den, ref), "rmse_noisy_mean": rmse(noisy, ref)}
        if spp == SPP[0]:
            zero = var == 0
            gp_zero = prefiltered(var.astype(np.float64)) == 0
            moved = np.abs(den.astype(np.float64) - noisy).max(axis=2) > 1e-6
            r["zero_variance"] = {
                "fraction_v_zero": float(zero.mean()),
                "fraction_prefiltered_zero": float(gp_zero.mean()),
                "fraction_of_v_zero_pixels_changed_by_filter": float(moved[zero].mean()) if zero.any() else None,
                "fraction_of_other_pixels_changed_by_filter": float(moved[~zero].mean()) if (~zero).any() else None,
                "rmse_v_zero_pixels_noisy": rmse(noisy[zero], ref[zero]) if zero.any() else None,
                "rmse_v_zero_pixels_denoised": rmse(den[zero], ref[zero]) if zero.any() else None,
            }
            filter_args = (noisy, var, aov["albedo"], aov["normal"], aov["depth"])
        out["denoised"].append(r)
    aov_ms = None
    ns.render_aov(params(SPP[0], DENOISE_DEFAULTS["aov_samples"]))         # warm-up
    for _ in range(3):
        _, st = ns.render_aov(params(SPP[0], DENOISE_DEFAULTS["aov_samples"]))
        aov_ms = st["ms_device"] if aov_ms is None else min(aov_ms, st["ms_device"])
    out["aov_pass_ms"] = aov_ms
    out["aov_samples"] = DENOISE_DEFAULTS["aov_samples"]
    out["filter"] = filter_kernel_ms(filter_args)
    ns.close()
    x = np.log([u["rmse"] for u in out["uniform"]])
    y = np.log([u["ms"] for u in out["uniform"]])
    b, a = np.polyfit(x, y, 1)
    for r in out["denoised"]:
        uni_ms = float(np.exp(a + b * np.log(r["rmse"])))
        r["uniform_ms_at_equal_rmse"] = uni_ms
        r["equal_error_time_ratio"] = uni_ms / r["ms"]
        r["in_range"] = bool(x.min() <= np.log(r["rmse"]) <= x.max())
    out["fit_log_ms_vs_log_rmse"] = [float(a), float(b)]
    out["seconds"] = time.time() - t0
    return out


def filter_4k():
    rng = np.random.default_rng(0)
    h, w = 2160, 3840
    color = rng.random((h, w, 3), np.float32)
    var = (rng.random((h, w), np.float32) * 0.01).astype(np.float32)
    albedo = rng.random((h, w, 3), np.float32)
    normal = np.zeros((h, w, 3), np.float32)
    normal[..., 2] = 1
    depth = (1 + rng.random((h, w), np.float32)).astype(np.float32)
    return filter_kernel_ms((color, var, albedo, normal, depth))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="denoise_bench.json")
    ap.add_argument("--ref-spp", type=int, default=4096)
    ap.add_argument("--scenes", default="cornell_box,part2_all,suzanne")
    opt = ap.parse_args()
    res = {"card": card(), "spp": list(SPP), "settings": DENOISE_DEFAULTS, "scenes": {}}
    for name in opt.scenes.split(","):
        res["scenes"][name] = r = run_scene(name, opt.ref_spp)
        print(f"{name} {r['size'][0]}x{r['size'][1]} (reference {r['ref_spp']} spp, {r['seconds']:.0f} s)  AOV pass {r['aov_pass_ms']:.2f} ms  "
              f"filter {r['filter'].get('ms', float('nan')):.2f} ms", flush=True)
        for u, d in zip(r["uniform"], r["denoised"]):
            print(f"  {u['spp']:4d} spp  uniform {u['ms']:8.1f} ms rmse {u['rmse']:.5f}   denoised {d['ms']:8.1f} ms rmse {d['rmse']:.5f}  "
                  f"equal-error time ratio {d['equal_error_time_ratio']:.2f}{'' if d['in_range'] else ' (extrapolated)'}", flush=True)
        print(f"  16 spp zero variance: {json.dumps(r['denoised'][0]['zero_variance'])}", flush=True)
    res["filter_3840x2160"] = filter_4k()
    print(f"filter at 3840x2160: {json.dumps(res['filter_3840x2160'])}", flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(opt.out)), exist_ok=True)
    with open(opt.out, "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
