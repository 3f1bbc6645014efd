"""`python -m firework_b200 --scene-file X.yml -s N [-o out.png] [-n name]` — the reference's CLI
(src/main.rs:6-62) on the GPU path: same flags, same hard-coded camera ((0,30,50) -> origin, fov 40), 960x540,
BVH on.  `-o` writes a PNG (window.rs:59-66 `save_image`); without it the image is written to `<name>.png`
(there is no window here).  Extra flags: --checkpoint FILE resumes / saves the fp32 sample sums so that a long
render can be interrupted (the reference's 3.36 h render has no intermediate save, README.md:16); --target-error E renders each
pixel until its relative standard error is <= E (adaptive sampling, `-s` is the cap per pixel, --min-samples the first round);
--denoise filters the render with first-hit albedo / normal / depth as guides (fw_render_denoised, default settings)."""
import argparse
import os
import sys
import time

import numpy as np

from . import CameraSettings, Renderer, Scene
from .progressive import render_progressive


def main(argv=None):
    ap = argparse.ArgumentParser(prog="firework")
    ap.add_argument("--scene-file", required=True)
    ap.add_argument("-n", "--name", default=None)
    ap.add_argument("-s", "--samples", type=int, required=True)
    ap.add_argument("-o", "--output", default=None)
    ap.add_argument("--checkpoint", default=None, help="npz file holding the fp32 sums + samples done (resume / save)")
    ap.add_argument("--chunk", type=int, default=0, help="samples per progressive step (default: all at once)")
    ap.add_argument("--width", type=int, default=960)
    ap.add_argument("--height", type=int, default=540)
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--target-error", type=float, default=None,
                    help="adaptive sampling: render each pixel until its relative standard error <= this (-s is the cap)")
    ap.add_argument("--min-samples", type=int, default=16, help="adaptive sampling: samples of the first round (default 16)")
    ap.add_argument("--denoise", action="store_true",
                    help="filter the render with first-hit albedo / normal / depth as guides (-s >= 2)")
    opt = ap.parse_args(argv)
    if opt.denoise:
        # a denoised render owns its sample range: no chunks, no checkpoint, no adaptive schedule
        if opt.checkpoint or opt.chunk or opt.target_error is not None:
            ap.error("--denoise can not be combined with --checkpoint, --chunk or --target-error")
        if opt.samples < 2:
            ap.error("--denoise needs --samples >= 2")
    if opt.target_error is not None:
        # an adaptive render owns its sample schedule: it can not be split into chunks or resumed from a checkpoint
        if opt.checkpoint or opt.chunk:
            ap.error("--target-error can not be combined with --checkpoint or --chunk")
        if not (opt.target_error >= 0.0) or opt.target_error == float("inf") or opt.min_samples < 1:
            ap.error("--target-error must be finite and >= 0, --min-samples >= 1")

    scene = Scene.from_file(opt.scene_file)
    camera = CameraSettings.default().cam_pos((0.0, 30.0, 50.0)).look_at((0.0, 0.0, 0.0)).field_of_view(40.0)
    renderer = (Renderer.default().width(opt.width).height(opt.height).samples(opt.samples).use_bvh(True)
                .camera(camera).seed(opt.seed))
    start = time.time()
    if opt.denoise:
        rgb = renderer.denoise().render(scene)
        print(f"Finished Rendering in {int(time.time() - start)} s")
    elif opt.target_error is not None:
        rgb = renderer.adaptive(opt.target_error, opt.min_samples).render(scene)
        st = renderer.last_stats
        print(f"Finished Rendering in {int(time.time() - start)} s")
        print(f"Adaptive: {st['samples']} samples in {st['rounds']} rounds, {st['samples'] / (opt.width * opt.height):.2f} spp mean "
              f"(cap {opt.samples})")
    else:
        rgb, info = render_progressive(scene, renderer, checkpoint=opt.checkpoint, chunk=opt.chunk or opt.samples)
        print(f"Finished Rendering in {int(time.time() - start)} s")
    name = opt.name or "Firework Render"
    out = opt.output or (name.replace(" ", "_") + ".png")
    print(f"Saving image to {out!r}")
    from PIL import Image
    Image.fromarray(rgb).save(out)
    return 0


if __name__ == "__main__":
    sys.exit(main())
