"""Device BVH builds (fw_bvh_build on a CUDA device, and fw_scene_commit for large trees) against the host build, byte for
byte: item order, wide nodes, root box and {nodes, root code, wide depth, binary depth}."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import ALL_SCENES, REPO, asset_loader, native_scene, scene_doc
from firework_b200 import _native as N
from firework_b200.engine import NativeScene, bvh_build

DEVICE_MIN_ITEMS = 8192   # kDeviceBvhMinItems (scene_host.h): fw_scene_commit builds trees this large on the device


def _cloud(n, seed, spread=100.0, size=1.0):
    """Small boxes scattered over a sphere's surface, like a mesh's triangles."""
    rng = np.random.default_rng(seed)
    d = rng.normal(size=(n, 3))
    c = spread * d / np.linalg.norm(d, axis=1, keepdims=True)
    h = size * rng.random((n, 3)) + 1e-3
    return np.concatenate([c - h, c + h], axis=1).astype(np.float32)


def _same(a, b):
    assert np.array_equal(a["items"], b["items"])
    assert a["info"] == b["info"]
    assert a["root_box"].tobytes() == b["root_box"].tobytes()
    assert a["nodes"].tobytes() == b["nodes"].tobytes()


def _check(boxes, unbounded=None):
    host = bvh_build(boxes, unbounded, device=-1)
    dev = bvh_build(boxes, unbounded, device=0)
    _same(dev, host)
    return host


def _mesh_boxes(doc):
    """Triangle boxes of every TriangleMesh in a scene document (also inside a ConstantMedium)."""
    out = []

    def walk(x):
        if isinstance(x, dict):
            if "indicies" in x and "verts" in x:
                v = np.array([[p["x"], p["y"], p["z"]] for p in x["verts"]], np.float32)
                t = v[np.array(x["indicies"], np.int64).reshape(-1, 3)]
                out.append(np.concatenate([t.min(axis=1), t.max(axis=1)], axis=1))
            for y in x.values():
                walk(y)
        elif isinstance(x, list):
            for y in x:
                walk(y)
    walk(doc)
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("name", ALL_SCENES)
def test_scene_trees_match_host(name):
    ns = native_scene(name, commit=False)
    ns.build_host()
    n = ns.num_objects()
    top = np.zeros((n, 6), np.float32)
    for i in range(n):
        N.check(N.lib().fw_scene_object_aabb(ns._h, i, N.ptr(top[i])))
    ns.close()
    _check(top)
    for boxes in _mesh_boxes(scene_doc(name)):
        _check(boxes)


@pytest.mark.gpu
def test_random_clouds_match_host():
    sizes = list(range(1, 65)) + [m for k in range(7, 18) for m in (2 ** k - 1, 2 ** k, 2 ** k + 1)] + [100000, 1000000]
    for n in sizes:
        _check(_cloud(n, seed=n))


@pytest.mark.gpu
def test_degenerate_inputs_match_host():
    # all centroids equal: both sorts must keep the input order at every level
    for n in (5, 1000, 3000, 40000):
        _check(np.tile(np.array([[-1, -2, -3, 1, 2, 3]], np.float32), (n, 1)))
        rng = np.random.default_rng(n)
        h = rng.random((n, 3)).astype(np.float32)   # same centre, different extents
        _check(np.concatenate([-h, h], axis=1))
    # +-0.0 centroids and subnormals: -0.0 and +0.0 tie under `<`
    rng = np.random.default_rng(7)
    for n in (33, 2500, 70000):
        vals = np.array([0.0, -0.0, 1e-45, -1e-45, 1e-40, -1e-40, 1e-38], np.float32)
        c = vals[rng.integers(0, len(vals), (n, 3))]
        _check(np.concatenate([c, c], axis=1))
        _check(np.concatenate([c - vals[rng.integers(0, 5, (n, 3))], c], axis=1))
    # boxes near 1e30: areas overflow, every cost is inf or NaN and the (2, n/2) fallback applies
    for n in (17, 5000, 50000):
        b = _cloud(n, seed=n, spread=1e30, size=1e30)
        _check(b)
    # unbounded flags and one-sided infinite boxes
    for n in (9, 4000, 60000):
        b = _cloud(n, seed=n + 1)
        u = (np.random.default_rng(n).random(n) < 0.1).astype(np.uint8)
        idx = np.random.default_rng(n + 2).integers(0, n, max(1, n // 50))
        b[idx, 0] = -np.inf
        b[idx[::2], 4] = np.inf
        _check(b, u)
    # a geometric series of sizes: the SAH peels one leaf per level until the depth limit forces balanced splits
    for n in (60, 200, 30000):
        i = np.arange(n, dtype=np.float64)
        lo = np.stack([1.2 ** (i % 400), np.zeros(n), np.zeros(n)], axis=1)
        hi = lo * 2 + 1
        _check(np.concatenate([lo, hi], axis=1).astype(np.float32))


@pytest.mark.gpu
def test_nan_centroid_gives_the_host_error():
    """A node sorts its items on axis depth % 3 only, so a NaN on an axis none of an item's nodes sorts on is no error
    (n = 1 sorts x alone); wherever the host refuses a tree the device must give the same code and message."""
    refused = 0
    for n, where in ((1, 0), (3, 2), (5, 4), (6, 5), (5000, 1234), (60000, 59999)):
        for axis in range(6):
            b = _cloud(n, seed=n)
            b[where, axis] = np.nan
            out = []
            for device in (-1, 0):
                try:
                    out.append(bvh_build(b, device=device))
                except N.FireworkError as e:
                    out.append((e.code, str(e)))
            if isinstance(out[0], tuple):
                refused += 1
                assert out[0] == out[1] and out[0][0] == -2 and "NaN centroid; bvh.rs:34" in out[0][1]
            else:
                _same(out[1], out[0])
    assert refused >= 20


@pytest.mark.gpu
def test_reference_interior_matches_host():
    prog = ("import sys; sys.path.insert(0, %r); sys.path.insert(0, %r)\n"
            "from test_gpu_bvh_build import _check, _cloud\n"
            "for n in (1, 2, 7, 64, 1025, 40000, 300000):\n"
            "    _check(_cloud(n, seed=n))\n"
            "print('ok')\n" % (REPO, os.path.join(REPO, "tests")))
    out = subprocess.run([sys.executable, "-c", prog], env=dict(os.environ, FW_BVH_SAH="0"), capture_output=True, text=True)
    assert out.returncode == 0 and out.stdout.strip().endswith("ok"), out.stderr[-2000:]


@pytest.mark.gpu
def test_device_builds_are_deterministic():
    b = _cloud(300000, seed=11)
    _same(bvh_build(b, device=0), bvh_build(b, device=0))


def _mesh_scene(n_side, seed):
    """A render object per mesh: a bumpy grid of 2 (n_side - 1)^2 triangles and a sphere, under a sky."""
    from firework_b200.scenes import (LambertianMat, RenderObject, Scene, SkyEnv, Sphere, TriangleMesh, Vec3)
    rng = np.random.default_rng(seed)
    scene = Scene.new()
    scene.set_environment(SkyEnv.default())
    mat = scene.add_material(LambertianMat.with_color(Vec3(0.4, 0.5, 0.6)))
    h = rng.random((n_side, n_side)).astype(np.float32)
    verts = [(np.float32(x * 0.1 - n_side * 0.05), h[y, x] * np.float32(0.05), np.float32(y * 0.1 - n_side * 0.05))
             for y in range(n_side) for x in range(n_side)]
    ind = []
    for y in range(1, n_side):
        for x in range(1, n_side):
            ind += [(y - 1) * n_side + x - 1, y * n_side + x, (y - 1) * n_side + x]
            ind += [(y - 1) * n_side + x - 1, y * n_side + x - 1, y * n_side + x]
    scene.add_object(RenderObject.new(TriangleMesh(verts, ind, None, None, mat)))
    scene.add_object(RenderObject.new(Sphere(1.0, mat)).position(0.0, 1.5, 0.0))
    return scene


class _device_kernels:
    """The set of device-build kernels (kernels_build.cu) that ran inside the block, from torch.profiler's CUDA activity."""
    NAMES = ("leaf_local_kernel", "sah_tile_cost_kernel", "merge_kernel", "tile_sort_kernel")

    def __enter__(self):
        import torch
        from torch.profiler import ProfilerActivity, profile
        self.torch = torch
        self.prof = profile(activities=[ProfilerActivity.CUDA])
        self.prof.__enter__()
        self.found = set()
        return self.found

    def __exit__(self, *exc):
        self.torch.cuda.synchronize()
        self.prof.__exit__(*exc)
        for e in self.prof.events():
            self.found |= {k for k in self.NAMES if k in e.name}
        return False


def _introspect(ns):
    top = ns.top_leaf_order()
    meshes = [ns.mesh_leaf_order(0)]
    nodes, root = ns.bvh_nodes()
    return top, meshes, nodes, root, ns.walk_info(), ns.device_bytes()


@pytest.mark.gpu
@pytest.mark.parametrize("n_side", [100, 200])
def test_commit_builds_large_trees_as_the_host_does(n_side):
    assert 2 * (n_side - 1) ** 2 >= DEVICE_MIN_ITEMS
    text = _mesh_scene(n_side, seed=n_side).to_yaml()
    with _device_kernels() as host_side:
        a = NativeScene(text, commit=False)
        a.build_host()     # host trees; the commit below uploads them
        a.commit()
    with _device_kernels() as device_side:
        b = NativeScene(text)   # the mesh's tree is built on the device
    assert not host_side and {"leaf_local_kernel", "sah_tile_cost_kernel"} <= device_side
    ra, rb = _introspect(a), _introspect(b)
    for x, y in zip(ra, rb):
        if isinstance(x, tuple) or isinstance(x, list):
            assert len(x) == len(y) and all(np.array_equal(np.asarray(p), np.asarray(q)) for p, q in zip(x, y))
        elif isinstance(x, np.ndarray):
            assert x.tobytes() == y.tobytes()
        else:
            assert x == y
    a.close()
    b.close()


@pytest.mark.gpu
def test_render_of_device_built_scene_matches_oracle_first_hit():
    from firework_b200.scenes import CONFIGS
    from firework_b200.serde_yaml import loads
    from oracle.oracle import OracleScene
    text = _mesh_scene(120, seed=3).to_yaml()
    ns = NativeScene(text)
    orc = OracleScene(loads(text), True, asset_loader=asset_loader)
    params = CONFIGS["suzanne"].renderer(width=64, height=48, samples=1, seed=1).params()
    for k, (p, q) in enumerate(zip((0.0, 4.0, 9.0), (0.0, 0.0, 0.0))):
        params.cam_pos[k], params.look_at[k] = p, q
    o, d = orc.primary_rays(params, 0)
    r = orc.first_hit(o, d, seed=1)
    for g in (ns.first_hit(o, d, True, seed=1), ns.first_hit_wavefront(o, d, True, seed=1)):
        assert np.array_equal(g["obj"], r["obj"]) and np.array_equal(g["prim"], r["prim"])
    assert (r["obj"] == 0).sum() > 100   # the rays do reach the mesh
    ns.close()


def test_argument_errors_come_before_any_cuda_call():
    L = N.lib()
    b = np.zeros((4, 6), np.float32)
    items, root, info = np.zeros(4, np.int32), np.zeros(6, np.float32), np.zeros(4, np.int32)
    assert L.fw_bvh_build(0, 0, N.ptr(b), None, N.ptr(items), None, 0, N.ptr(root), N.ptr(info)) == -5
    assert L.fw_bvh_build(0, 4, None, None, N.ptr(items), None, 0, N.ptr(root), N.ptr(info)) == -5
    assert L.fw_bvh_build(0, 4, N.ptr(b), None, None, None, 0, N.ptr(root), N.ptr(info)) == -5
    assert L.fw_bvh_build(0, 4, N.ptr(b), None, N.ptr(items), None, -1, N.ptr(root), N.ptr(info)) == -5
    assert L.fw_bvh_build(-2, 4, N.ptr(b), None, N.ptr(items), None, 0, N.ptr(root), N.ptr(info)) == -5


def test_host_probe_matches_the_scene_build():
    """fw_bvh_build(device = -1) is the tree fw_scene_build_host makes: the top-level tree of every scene."""
    for name in ALL_SCENES:
        ns = native_scene(name, commit=False)
        ns.build_host()
        n = ns.num_objects()
        top = np.zeros((n, 6), np.float32)
        for i in range(n):
            N.check(N.lib().fw_scene_object_aabb(ns._h, i, N.ptr(top[i])))
        t = bvh_build(top, device=-1)
        nodes, root = ns.bvh_nodes()
        assert np.array_equal(t["items"], ns.top_leaf_order())
        assert t["info"]["root_code"] == root
        # boxes and codes; the unbounded flags (row 7) are the scene's, which this call was not given
        assert nodes[: t["info"]["nodes"], :7].tobytes() == t["nodes"].reshape(-1, 8, 4)[:, :7].tobytes()
        ns.close()
