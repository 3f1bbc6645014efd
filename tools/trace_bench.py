"""What tracing caller-supplied rays costs against the camera: fw_trace_rays_device fed with fw_render's own camera rays (per-sample
layout, uploaded once) against fw_render at the same size and spp, with the two arms alternated.

    python tools/trace_bench.py [--out trace_bench.json] [--reps 5] [--scenes part2_all,suzanne,cornell_box]

Both arms report the CUDA-event time of their device work (fw_stats.ms_device: the batch loop from the first raygen to the last
tally); the trace arm reads 24 bytes of ray per path where the render's raygen computes the camera ray.  Each scene also records
whether the trace's sums equal the render's bit for bit.  The card's name and power limit are read in the same run."""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from firework_b200.engine import NativeScene  # noqa: E402
from firework_b200.scenes import CONFIGS  # noqa: E402

WORKLOADS = {"part2_all": (1920, 1080, 64), "suzanne": (1920, 1080, 64), "cornell_box": (300, 300, 1024)}


def card():
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=30)
        name, power, clock = [x.strip() for x in r.stdout.strip().splitlines()[0].split(",")]
        return {"name": name, "power_limit": power, "max_sm_clock": clock}
    except Exception as e:  # the numbers still stand, without the card's description
        return {"error": str(e)}


def run_scene(name, reps):
    import torch
    w, h, spp = WORKLOADS[name]
    cfg = CONFIGS[name]
    ns = NativeScene.from_scene(cfg.load(), 0)
    try:
        p = cfg.renderer(width=w, height=h, samples=spp, seed=0).params()
        npix = w * h
        o = torch.empty((spp, npix, 3), dtype=torch.float32, device="cuda")
        d = torch.empty_like(o)
        for s in range(spp):                                          # fw_render's camera rays, uploaded once
            ho, hd = ns.primary_rays(p, s)
            o[s].copy_(torch.from_numpy(ho))
            d[s].copy_(torch.from_numpy(hd))
        total = torch.zeros((npix, 3), dtype=torch.float32, device="cuda")
        stream = torch.cuda.Stream()
        stream.wait_stream(torch.cuda.current_stream())
        torch.cuda.synchronize()

        def trace():
            total.zero_()
            torch.cuda.synchronize()
            return ns.trace_rays_device(o.data_ptr(), d.data_ptr(), npix, total.data_ptr(), stream.cuda_stream, per_sample=True,
                                        sample_count=spp, seed=0, use_bvh=cfg.use_bvh)

        def render():
            return ns.render(p, want_rgb=False)
        render_sum = render()[1]                                      # warm-up of both arms
        trace()
        identical = bool(np.array_equal(total.cpu().numpy().view(np.uint32), render_sum.reshape(-1, 3).view(np.uint32)))
        arms = {"render": [], "trace": []}
        for _ in range(reps):                                         # alternated
            arms["render"].append(render()[2]["ms_device"])
            arms["trace"].append(trace()["ms_device"])
        res = {"size": [w, h], "spp": spp, "use_bvh": cfg.use_bvh, "trace_sums_equal_render_sums": identical,
               "ray_bytes_per_path": 24, "ray_buffer_bytes": 2 * o.numel() * 4}
        for arm, ms in arms.items():
            res[arm] = {"ms_device": ms, "min_ms": min(ms), "median_ms": float(np.median(ms)),
                        "msamples_per_s_at_min": npix * spp / (min(ms) * 1e3)}
        res["trace_over_render_min"] = res["trace"]["min_ms"] / res["render"]["min_ms"]
        res["trace_over_render_median"] = res["trace"]["median_ms"] / res["render"]["median_ms"]
        return res
    finally:
        ns.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="trace_bench.json")
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--scenes", default="part2_all,suzanne,cornell_box")
    opt = ap.parse_args()
    res = {"card": card(), "scenes": {}}
    for name in opt.scenes.split(","):
        res["scenes"][name] = r = run_scene(name, opt.reps)
        print(f"{name} {r['size'][0]}x{r['size'][1]} x {r['spp']} spp  render {r['render']['min_ms']:.2f} / {r['render']['median_ms']:.2f} ms  "
              f"trace {r['trace']['min_ms']:.2f} / {r['trace']['median_ms']:.2f} ms (min / median)  ratio {r['trace_over_render_median']:.4f}  "
              f"bit-identical {r['trace_sums_equal_render_sums']}", flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(opt.out)), exist_ok=True)
    with open(opt.out, "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
