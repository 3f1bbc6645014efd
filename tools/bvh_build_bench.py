"""Host against device BVH builds: fw_bvh_build over mesh-like boxes (small boxes scattered over a sphere, 1e4 to 4e6 of them) and
over part2_all's top-level tree, and fw_scene_commit of generated triangle-soup scenes with host-built and device-built trees.

    python tools/bvh_build_bench.py [--out profiles/r06_bvh_build_bench.json] [--reps 3]

Wall times are host clocks around the synchronous calls (the device arm includes its uploads and read-backs and the host's
O(n) box and collapse stages).  Commit times are medians over --reps commits after a warm-up.  `kernels_ms` is the CUDA time of the device build's kernels and copies in one call, summed
from torch.profiler.  Every device result is compared with the host's, byte for byte.  The card's name and power limit are
read in the same run."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, REPO)
from firework_b200 import _native as N  # noqa: E402
from firework_b200.engine import NativeScene, bvh_build  # noqa: E402

SIZES = [2000, 3000, 4000, 6000, 8000, 10000, 16384, 30000, 100000, 300000, 1000000, 2000000, 4000000]
COMMIT_SIZES = [4000, 8192, 10000, 30000, 100000, 1000000]


def card():
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=30)
        name, power, clock = [x.strip() for x in r.stdout.strip().splitlines()[0].split(",")]
        return {"name": name, "power_limit": power, "max_sm_clock": clock}
    except Exception as e:  # the numbers still stand, without the card's description
        return {"error": str(e)}


def cloud(n, seed):
    rng = np.random.default_rng(seed)
    d = rng.normal(size=(n, 3))
    c = 100.0 * d / np.linalg.norm(d, axis=1, keepdims=True)
    h = rng.random((n, 3)) + 1e-3
    return np.concatenate([c - h, c + h], axis=1).astype(np.float32)


def timed(f, reps):
    ts, out = [], None
    for _ in range(reps):
        t0 = time.perf_counter()
        out = f()
        ts.append((time.perf_counter() - t0) * 1e3)
    return float(np.median(ts)), out


def kernel_ms(f):
    import torch
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        f()
        torch.cuda.synchronize()
    total = 0.0
    for e in prof.events():
        if e.device_type == torch.autograd.DeviceType.CUDA:
            total += e.device_time_total if hasattr(e, "device_time_total") else e.cuda_time_total
    return total / 1e3


def same(a, b):
    return bool(np.array_equal(a["items"], b["items"]) and a["info"] == b["info"] and a["root_box"].tobytes() == b["root_box"].tobytes()
                and a["nodes"].tobytes() == b["nodes"].tobytes())


def probe(boxes, reps):
    n = len(boxes)
    hr = 1 if n >= 1000000 else reps
    host_ms, host = timed(lambda: bvh_build(boxes, device=-1), hr)
    bvh_build(boxes, device=0)   # warm: module load, memory pool
    dev_ms, dev = timed(lambda: bvh_build(boxes, device=0), reps)
    return {"n": n, "host_ms": host_ms, "device_ms": dev_ms, "kernels_ms": kernel_ms(lambda: bvh_build(boxes, device=0)),
            "speedup": host_ms / dev_ms, "identical": same(host, dev), "wide_nodes": host["info"]["nodes"]}


def soup_yaml(n, seed):
    """A scene of one TriangleMesh of n small triangles over a sphere, written straight in the scene format."""
    b = cloud(n, seed)
    v = np.stack([b[:, :3], np.concatenate([b[:, 3:4], b[:, 1:3]], axis=1), np.concatenate([b[:, 0:1], b[:, 4:6]], axis=1)], axis=1)
    v = v.reshape(-1, 3).astype(np.float64)
    verts = "".join("        - x: %r\n          y: %r\n          z: %r\n" % (float(x), float(y), float(z)) for x, y, z in v)
    ind = "".join("        - %d\n" % i for i in range(3 * n))
    return ("---\nrender_objects:\n  - obj:\n      object_type: TriangleMesh\n      indicies:\n" + ind + "      verts:\n" + verts +
            "      normals: ~\n      uvs: ~\n      material: 0\n    position:\n      x: 0.0\n      y: 0.0\n      z: 0.0\n"
            "    rotation:\n      s: 1.0\n      bv:\n        xy: 0.0\n        xz: 0.0\n        yz: 0.0\n    flip_normals: false\n"
            "materials:\n  - material: LambertianMat\n    albedo:\n      texture: ConstantTexture\n      color:\n"
            "        x: 0.5\n        y: 0.5\n        z: 0.5\nenvironment:\n  environment: ColorEnv\n  color:\n    x: 0.0\n    y: 0.0\n    z: 0.0\n")


def commit(text, reps):
    def host():
        s = NativeScene(text, commit=False)
        s.build_host()
        s.commit()
        return s

    def dev():
        return NativeScene(text)
    out = {}
    dev().close()   # warm: the device build's module and memory pool
    for arm, f in (("host_trees", host), ("device_trees", dev)):
        ts = []
        for _ in range(reps):
            t0 = time.perf_counter()
            s = f()
            ts.append((time.perf_counter() - t0) * 1e3)
            out[arm] = (s.bvh_nodes()[0].tobytes(), s.mesh_leaf_order(0).tobytes(), s.device_bytes())
            s.close()
        out[arm + "_ms"] = float(np.median(ts))
    out["identical"] = out.pop("host_trees") == out.pop("device_trees")
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(REPO, "profiles", "r06_bvh_build_bench.json"))
    ap.add_argument("--reps", type=int, default=3)
    a = ap.parse_args()
    res = {"card": card(), "probe": [], "commit": []}
    for n in SIZES:
        r = probe(cloud(n, n), a.reps)
        print(json.dumps(r), flush=True)
        res["probe"].append(r)
    from firework_b200.scenes import CONFIGS
    ns = NativeScene.from_scene(CONFIGS["part2_all"].load(), 0)
    top = ns.object_aabbs()
    ns.close()
    r = probe(top, a.reps)
    r["tree"] = "part2_all top level"
    print(json.dumps(r), flush=True)
    res["probe"].append(r)
    for n in COMMIT_SIZES:
        text = soup_yaml(n, n)
        r = {"triangles": n, **commit(text, 1 if n >= 1000000 else a.reps)}
        print(json.dumps(r), flush=True)
        res["commit"].append(r)
    os.makedirs(os.path.dirname(a.out), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
