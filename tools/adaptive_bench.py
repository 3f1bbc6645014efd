"""What adaptive sampling buys, measured: uniform renders at a few spp against adaptive renders at a few thresholds, each
compared with a high-spp uniform reference (RMSE of the linear per-pixel mean), with device time and samples spent.

    python tools/adaptive_bench.py [--out profiles/adaptive_bench.json] [--ref-spp 4096] [--scenes cornell_box,part2_all,suzanne]

equal_error_time_ratio = (device ms a uniform render needs for the same RMSE) / (adaptive device ms): > 1 means adaptive sampling
is faster at equal error, < 1 that it is slower.  The uniform time at a given RMSE comes from a least-squares fit of
log(ms) against log(RMSE) over the uniform renders of the scene (interpolation inside their range, extrapolation outside it:
`in_range` says which).  The card's name and power limit are read in the same run."""
import argparse
import gzip
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from firework_b200.engine import NativeScene  # noqa: E402
from firework_b200.scenes import CONFIGS, SCENE_DIR  # noqa: E402

SIZES = {"cornell_box": (300, 300), "part2_all": (1920, 1080), "suzanne": (1920, 1080)}
UNIFORM_SPP = (16, 32, 64, 128, 256)
THRESHOLDS = (0.2, 0.1, 0.05, 0.03)
MIN_SAMPLES, CAP = 16, 1024


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


def run_scene(name, ref_spp):
    cfg = CONFIGS[name]
    w, h = SIZES[name]
    p = cfg.path()
    text = (gzip.open(p, "rt") if p.endswith(".gz") else open(p)).read()
    ns = NativeScene(text, asset_dir=os.path.join(SCENE_DIR, "assets"))

    def params(spp):
        return cfg.renderer(width=w, height=h, samples=spp, seed=1).params()

    t0 = time.time()
    _, ref_sum, st = ns.render(params(ref_spp), want_rgb=False)
    ref = ref_sum.astype(np.float64) / ref_spp
    out = {"size": [w, h], "ref_spp": ref_spp, "ref_ms": st["ms_device"], "uniform": [], "adaptive": []}
    ns.render(params(UNIFORM_SPP[0]), want_rgb=False)                    # warm-up
    for spp in UNIFORM_SPP:
        best = None
        for _ in range(2):
            _, s, st = ns.render(params(spp), want_rgb=False)
            best = st["ms_device"] if best is None else min(best, st["ms_device"])
        out["uniform"].append({"spp": spp, "samples": st["samples"], "ms": best, "rmse": rmse(s / spp, ref)})
    ns.render_adaptive(params(CAP), THRESHOLDS[0], MIN_SAMPLES, want_rgb=False)   # warm-up
    for t in THRESHOLDS:
        best, wall = None, None
        for _ in range(2):
            c0 = time.perf_counter()
            _, s, counts, err, st = ns.render_adaptive(params(CAP), t, MIN_SAMPLES, want_rgb=False)
            c1 = time.perf_counter()
            if best is None or st["ms_device"] < best:
                best, wall = st["ms_device"], (c1 - c0) * 1e3
        mean = s / counts[..., None].astype(np.float32)
        out["adaptive"].append({"threshold": t, "min_samples": MIN_SAMPLES, "cap": CAP, "samples": st["samples"],
                                "mean_spp": st["samples"] / (w * h), "rounds": st["rounds"], "active": st["active"],
                                "ms": best, "wall_ms": wall, "rmse": rmse(mean, ref),
                                "pixels_at_cap": int((counts == CAP).sum())})
    ns.close()
    # equal-error time: log(ms) = a + b log(rmse) over the uniform renders
    x = np.log([u["rmse"] for u in out["uniform"]])
    y = np.log([u["ms"] for u in out["uniform"]])
    b, a = np.polyfit(x, y, 1)
    for r in out["adaptive"]:
        uni_ms = float(np.exp(a + b * np.log(r["rmse"])))
        r["uniform_ms_at_equal_rmse"] = uni_ms
        r["equal_error_time_ratio"] = uni_ms / r["ms"]
        r["in_range"] = bool(x.min() <= np.log(r["rmse"]) <= x.max())
    out["fit_log_ms_vs_log_rmse"] = [float(a), float(b)]
    out["seconds"] = time.time() - t0
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="adaptive_bench.json")
    ap.add_argument("--ref-spp", type=int, default=4096)
    ap.add_argument("--scenes", default="cornell_box,part2_all,suzanne")
    opt = ap.parse_args()
    res = {"card": card(), "uniform_spp": list(UNIFORM_SPP), "thresholds": list(THRESHOLDS), "scenes": {}}
    for name in opt.scenes.split(","):
        res["scenes"][name] = r = run_scene(name, opt.ref_spp)
        print(f"{name} {r['size'][0]}x{r['size'][1]} (reference {r['ref_spp']} spp, {r['seconds']:.0f} s)", flush=True)
        for u in r["uniform"]:
            print(f"  uniform  {u['spp']:5d} spp            {u['ms']:9.1f} ms  rmse {u['rmse']:.5f}")
        for v in r["adaptive"]:
            print(f"  adaptive e={v['threshold']:<5} {v['mean_spp']:7.1f} spp mean {v['ms']:9.1f} ms  rmse {v['rmse']:.5f}  "
                  f"equal-error time ratio {v['equal_error_time_ratio']:.2f}{'' if v['in_range'] else ' (extrapolated)'}  "
                  f"rounds {v['rounds']}", flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(opt.out)), exist_ok=True)
    with open(opt.out, "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
