"""Render a workload twice with the same build; report pixels whose fp32 sums differ from run to run."""
import os, sys, gzip
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
from firework_b200.engine import NativeScene
from firework_b200.scenes import CONFIGS, SCENE_DIR
name, w, h, spp = sys.argv[1], int(sys.argv[2]), int(sys.argv[3]), int(sys.argv[4])
cfg = CONFIGS[name]; p = cfg.path()
text = (gzip.open(p, "rt") if p.endswith(".gz") else open(p)).read()
def render():
    ns = NativeScene(text, asset_dir=os.path.join(SCENE_DIR, "assets"))
    _, s, st = ns.render(cfg.renderer(width=w, height=h, samples=spp, seed=2).params(), want_rgb=False)
    ns.close()
    return s, st
a, sa = render(); b, sb = render()
print("rays", sa["rays"], sb["rays"])
da = ~((a == b) | (np.isnan(a) & np.isnan(b)))
print("run vs run: differing values", int(da.sum()), "pixels", np.argwhere(da.any(2))[:10].tolist())
for yx in np.argwhere(da.any(2))[:5]:
    print("   ", yx, a[tuple(yx)], b[tuple(yx)])
