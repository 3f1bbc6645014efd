"""GPU edge cases: degenerate trees (1 / 2 objects, 1-triangle mesh), ragged sizes, nested shapes, per-face
materials, single samples — each compared with the oracle through the same gates as test_gpu_parity.py."""
import numpy as np
import pytest

from firework_b200.api import (CameraSettings, CheckerTexture, ConstantTexture, Cone, Cylinder, DielectricMat, Disk,
                               EmissiveMat, LambertianMat, MarbleTexture, MetalMat, PerlinNoiseTexture, Rect3d,
                               RenderObject, Renderer, Rotor3, Scene, SkyEnv, Sphere, TriangleMesh, Vec3, XYRect,
                               XZRect, YZRect)
from firework_b200.engine import NativeScene
from oracle.oracle import OracleScene

pytestmark = pytest.mark.gpu


def _renderer(w, h, spp, use_bvh, cam=(3.0, 2.0, 6.0), look=(0.0, 0.5, 0.0), seed=3):
    return (Renderer.default().width(w).height(h).samples(spp).use_bvh(use_bvh).seed(seed)
            .camera(CameraSettings.default().cam_pos(cam).look_at(look).field_of_view(45.0)))


def _compare(scene, w, h, spp, use_bvh, min_close=0.995, **kw):
    ns = NativeScene(scene.to_yaml())
    orc = OracleScene(scene.to_dict(), use_bvh)
    r = _renderer(w, h, spp, use_bvh, **kw)
    p = r.params()
    go, gd = ns.primary_rays(p, 0)
    oo, od = orc.primary_rays(p, 0)
    assert np.array_equal(go, oo) and np.array_equal(gd, od)
    g = ns.first_hit(go, gd, use_bvh, seed=3)
    o = orc.first_hit(go, gd, seed=3)
    assert np.array_equal(g["obj"], o["obj"]) and np.array_equal(g["prim"], o["prim"])
    assert np.array_equal(g["material"], o["material"])
    hit = o["obj"] >= 0
    if hit.any():
        assert (np.abs(g["t"][hit] - o["t"][hit]) / np.abs(o["t"][hit])).max() <= 1e-5
    grgb, gsum, gst = ns.render(p)
    orgb, osum, ost = orc.render(p)
    close = np.all((np.abs(gsum - osum) <= 1e-4 * np.maximum(np.abs(osum), 1e-3)) | (np.isnan(gsum) & np.isnan(osum)), axis=2)
    assert close.mean() >= min_close, f"{(~close).sum()} / {close.size} pixels differ"
    assert gst["samples"] == w * h * spp
    ns.close()
    return g, o


def _base_scene():
    s = Scene.new()
    s.set_environment(SkyEnv.default())
    return s


@pytest.mark.parametrize("use_bvh", [True, False])
@pytest.mark.parametrize("n_objects", [1, 2, 3])
def test_tiny_trees(use_bvh, n_objects):
    """1 object = Leaf root, 2 = DoubleLeaf root, 3 = Branch(Leaf, DoubleLeaf) (bvh.rs:37-69)."""
    s = _base_scene()
    m = s.add_material(LambertianMat.with_color(Vec3(0.6, 0.3, 0.2)))
    g = s.add_material(MetalMat(Vec3(0.8, 0.8, 0.8), 0.1))
    s.add_object(RenderObject.new(Sphere(1.0, m)).position(0.0, 1.0, 0.0))
    if n_objects >= 2:
        s.add_object(RenderObject.new(XZRect(-5.0, 5.0, -5.0, 5.0, 0.0, g)))
    if n_objects >= 3:
        s.add_object(RenderObject.new(Sphere(0.5, g)).position(1.5, 0.5, 1.0))
    _compare(s, 67, 41, 3, use_bvh)


@pytest.mark.parametrize("w,h,spp", [(1, 1, 1), (1, 7, 2), (33, 1, 5), (31, 17, 1), (129, 65, 2)])
def test_ragged_image_sizes(w, h, spp):
    s = _base_scene()
    m = s.add_material(LambertianMat(CheckerTexture.with_colors(Vec3(0.1, 0.1, 0.1), Vec3(0.9, 0.9, 0.9), 4.0)))
    d = s.add_material(DielectricMat(1.5))
    s.add_object(RenderObject.new(XZRect(-8.0, 8.0, -8.0, 8.0, 0.0, m)))
    s.add_object(RenderObject.new(Sphere(1.0, d)).position(0.0, 1.0, 0.0))
    s.add_object(RenderObject.new(Sphere(0.4, m)).position(-1.5, 0.4, 1.0))
    _compare(s, w, h, spp, True, min_close=0.99 if w * h > 4 else 1.0)


def _mesh_layout(top_meshes, medium_mesh, n_spheres):
    """A floor, `top_meshes` tetrahedra (4 triangles: an interior mesh root, which the mesh walk needs), optionally one more
    as the boundary of a ConstantMedium, and `n_spheres` small spheres (over 32 objects: more than 16 top-level leaves)."""
    s = _base_scene()
    red = s.add_material(LambertianMat.with_color(Vec3(0.8, 0.2, 0.2)))
    grey = s.add_material(LambertianMat.with_color(Vec3(0.5, 0.5, 0.5)))
    s.add_object(RenderObject.new(XZRect(-6.0, 6.0, -6.0, 6.0, 0.0, grey)))
    v = [[0, 0, 0], [1, 0, 0], [0.5, 0, 0.9], [0.5, 0.9, 0.4]]
    tet = [0, 2, 1, 0, 1, 3, 1, 2, 3, 2, 0, 3]
    for k in range(top_meshes):
        s.add_object(RenderObject.new(TriangleMesh(v, tet, None, None, red)).position(-2.0 + 1.5 * k, 0.1, 0.0)
                     .rotate(Rotor3.from_rotation_xz(0.3 * k)))
    if medium_mesh:
        s.add_volume(RenderObject.new(TriangleMesh(v, tet, None, None, red)).position(1.5, 0.1, 0.5), 2.0,
                     ConstantTexture(Vec3(0.2, 0.4, 0.9)))
    for x, z in np.random.default_rng(5).uniform((-4.0, -4.0), (4.0, -1.5), (n_spheres, 2)):
        s.add_object(RenderObject.new(Sphere(0.15, grey)).position(float(x), 0.15, float(z)))
    return s


@pytest.mark.parametrize("use_bvh", [True, False])
def test_meshes_small_and_nested_in_media(use_bvh):
    """1- and 2-triangle meshes (Leaf / DoubleLeaf mesh roots), a mesh with normals + uvs, and ConstantMedium
    wrapping a mesh and a box (volume.rs generic over the boundary shape).  Then the other mesh layouts an extend kernel is
    chosen by: a mesh only inside a medium, and meshes the mesh walk serves, with and without one inside a medium, under a
    top-level tree of at most and of more than 16 leaves (linear scan: the larger scenes' programs do not fit
    kernel-parameter space, so the object loop runs)."""
    s = _base_scene()
    red = s.add_material(LambertianMat.with_color(Vec3(0.8, 0.2, 0.2)))
    grey = s.add_material(LambertianMat.with_color(Vec3(0.5, 0.5, 0.5)))
    s.add_object(RenderObject.new(XZRect(-6.0, 6.0, -6.0, 6.0, 0.0, grey)))
    tri = TriangleMesh([[0, 0, 0], [1, 0, 0], [0, 1, 0]], [0, 1, 2], None, None, red)
    s.add_object(RenderObject.new(tri).position(-2.0, 0.2, 0.0))
    quad = TriangleMesh([[0, 0, 0], [1, 0, 0], [1, 1, 0], [0, 1, 0]], [0, 1, 2, 0, 2, 3],
                        [[0, 0, 1]] * 4, [[0, 0], [1, 0], [1, 1], [0, 1]], red)
    s.add_object(RenderObject.new(quad).position(0.0, 0.2, 0.0).rotate(Rotor3.from_rotation_xz(0.5)))
    # a closed tetrahedron as medium boundary
    v = [[0, 0, 0], [1, 0, 0], [0.5, 0, 0.9], [0.5, 0.9, 0.4]]
    tet = TriangleMesh(v, [0, 2, 1, 0, 1, 3, 1, 2, 3, 2, 0, 3], None, None, red)
    s.add_volume(RenderObject.new(tet).position(1.5, 0.1, 0.5), 2.0, ConstantTexture(Vec3(0.2, 0.4, 0.9)))
    s.add_volume(RenderObject.new(Rect3d.with_size(Vec3(1.0, 1.0, 1.0), grey)).position(-0.5, 0.0, -2.5), 1.5,
                 ConstantTexture(Vec3(0.9, 0.9, 0.9)))
    _compare(s, 96, 64, 4, use_bvh)
    for top_meshes, medium_mesh, n_spheres in ((0, True, 0), (2, True, 0), (2, True, 100), (2, False, 100)):
        _compare(_mesh_layout(top_meshes, medium_mesh, n_spheres), 64, 40, 2, use_bvh)


@pytest.mark.parametrize("use_bvh", [True, False])
def test_conics_textures_and_rotations(use_bvh):
    s = _base_scene()
    marble = s.add_material(LambertianMat(MarbleTexture(4, 3.0)))
    perlin = s.add_material(LambertianMat(PerlinNoiseTexture(2.5)))
    light = s.add_material(EmissiveMat.with_color(Vec3(4.0, 4.0, 4.0)))
    metal = s.add_material(MetalMat(Vec3(0.7, 0.6, 0.5), 0.3))
    s.add_object(RenderObject.new(XZRect(-8.0, 8.0, -8.0, 8.0, 0.0, perlin)))
    s.add_object(RenderObject.new(Cylinder.partial(0.7, 1.5, 270.0, marble)).position(-2.0, 0.0, 0.0)
                 .rotate(Rotor3.from_rotation_xy(0.4)))
    s.add_object(RenderObject.new(Cone(0.8, 1.6, metal)).position(0.0, 0.0, 0.5))
    s.add_object(RenderObject.new(Disk.partial(1.0, 300.0, 0.3, marble)).position(2.0, 0.8, 0.0)
                 .rotate(Rotor3.from_rotation_yz(0.7)))
    s.add_object(RenderObject.new(XYRect(-1.0, 1.0, 2.0, 3.0, -2.0, light)).flip_normals())
    s.add_object(RenderObject.new(YZRect(0.0, 1.0, -1.0, 1.0, 3.0, metal)).rotate(Rotor3.from_rotation_xz(-0.3)))
    # rotation below the 0.999 cos-trace threshold: the ray is NOT rotated but the hit is (scene.rs:242-258)
    s.add_object(RenderObject.new(Rect3d.with_size(Vec3(0.6, 0.6, 0.6), marble)).position(0.5, 0.0, 2.0)
                 .rotate(Rotor3.from_rotation_xz(0.02)))
    _compare(s, 120, 80, 4, use_bvh, min_close=0.98)   # sin / atan2 / acos heavy: a few more ulp-flipped pixels


def test_rect3d_faces_with_their_own_materials():
    """A deserialised Rect3d may carry a different material per face (rect3d.rs:10-15 stores plain rects)."""
    s = _base_scene()
    mats = [s.add_material(LambertianMat.with_color(Vec3(*c))) for c in
            [(0.9, 0.1, 0.1), (0.1, 0.9, 0.1), (0.1, 0.1, 0.9), (0.9, 0.9, 0.1), (0.1, 0.9, 0.9), (0.9, 0.1, 0.9)]]
    emis = s.add_material(EmissiveMat.with_color(Vec3(2.0, 2.0, 2.0)))
    box = Rect3d.with_size(Vec3(1.0, 1.0, 1.0), mats[0])
    for i, (_tag, face) in enumerate(box.faces):
        face.material = mats[i] if i != 2 else emis
    s.add_object(RenderObject.new(box).position(-0.5, 0.0, -0.5).rotate(Rotor3.from_rotation_xz(0.6)))
    s.add_object(RenderObject.new(XZRect(-5.0, 5.0, -5.0, 5.0, 0.0, mats[3])))
    for use_bvh in (True, False):
        g, o = _compare(s, 80, 60, 4, use_bvh)
        assert len(set(o["material"][o["obj"] == 0].tolist())) >= 2


def test_many_objects_deep_tree():
    """4097 spheres: a 13-level reference tree (7 wide levels); exercises the traversal stack bound."""
    rng = np.random.default_rng(1)
    s = _base_scene()
    m = s.add_material(LambertianMat.with_color(Vec3(0.5, 0.6, 0.7)))
    for p in rng.uniform(-6, 6, (4097, 3)):
        s.add_object(RenderObject.new(Sphere(0.12, m)).position(float(p[0]), float(p[1]), float(p[2])))
    _compare(s, 96, 64, 2, True, cam=(0.0, 0.0, 16.0), look=(0.0, 0.0, 0.0))


def test_zero_samples_and_bad_arguments():
    from firework_b200._native import FireworkError
    s = _base_scene()
    m = s.add_material(LambertianMat.with_color(Vec3(0.5, 0.5, 0.5)))
    s.add_object(RenderObject.new(Sphere(1.0, m)))
    ns = NativeScene(s.to_yaml())
    p = _renderer(8, 8, 4, True).params(sample_begin=0, sample_count=0)
    rgb, sm, st = ns.render(p)
    assert not sm.any() and st["rays"] == 0
    bad = _renderer(8, 8, 4, True).params()
    bad.width = 0
    with pytest.raises(FireworkError):
        ns.render(bad)
    ns.close()


def _linear_scene(n_spheres):
    """A linear-scan scene: n translated spheres + a ground rect + a Rect3d with canonical faces + a rotated one."""
    s = _base_scene()
    m = s.add_material(LambertianMat.with_color(Vec3(0.6, 0.3, 0.2)))
    g = s.add_material(MetalMat(Vec3(0.8, 0.8, 0.8), 0.1))
    rng = np.random.default_rng(9)
    for i in range(n_spheres):
        x, z = rng.uniform(-3.0, 3.0, 2)
        s.add_object(RenderObject.new(Sphere(0.25, m if i % 2 else g)).position(float(x), 0.25, float(z)))
    s.add_object(RenderObject.new(XZRect(-6.0, 6.0, -6.0, 6.0, 0.0, m)))
    s.add_object(RenderObject.new(Rect3d.with_size(Vec3(0.8, 1.2, 0.8), g)).position(-1.0, 0.0, 1.0))
    s.add_object(RenderObject.new(Rect3d.with_size(Vec3(0.6, 0.6, 0.6), m)).rotate(Rotor3.from_rotation_xz(0.6)).position(1.2, 0.0, 0.5))
    return s


def test_linear_program_and_object_loop_kernels_agree(monkeypatch):
    """Linear-scan scenes run the LinProgram kernels when the program fits kernel-parameter space, and the object-loop
    kernels otherwise (or with FW_LINEAR_PROGRAM=0).  Both must give the oracle's result, and each other's, bit for bit."""
    small = _linear_scene(6)
    ns = NativeScene(small.to_yaml())
    words = ns.linear_program()
    assert 0 < len(words) <= 160
    p = _renderer(64, 40, 4, False).params()
    _, sum_prog, _ = ns.render(p)
    o, d = ns.primary_rays(p, 0)
    hit_prog = ns.first_hit(o, d, False, seed=3)
    ns.close()
    monkeypatch.setenv("FW_LINEAR_PROGRAM", "0")
    ns2 = NativeScene(small.to_yaml())
    _, sum_loop, _ = ns2.render(p)
    hit_loop = ns2.first_hit(o, d, False, seed=3)
    ns2.close()
    monkeypatch.delenv("FW_LINEAR_PROGRAM")
    assert np.array_equal(sum_prog, sum_loop, equal_nan=True)
    for k in ("obj", "prim", "material", "t", "point", "normal"):
        assert np.array_equal(hit_prog[k], hit_loop[k], equal_nan=True), k
    _compare(small, 64, 40, 4, False)
    # too many items for kernel-parameter space: the object-loop kernels take over by themselves
    big = _linear_scene(120)
    nb = NativeScene(big.to_yaml(), commit=False)
    nb.build_host()
    assert len(nb.linear_program()) > 160
    nb.close()
    _compare(big, 48, 30, 2, False)


def test_black_environment_miss_shortcut_is_exact(monkeypatch):
    """part2_all and volume-like scenes have a black ColorEnv but procedural (noise) textures, so the miss kernel can not be
    dropped statically; it returns at once unless a shade kernel flagged a non-finite / huge attenuation in the batch
    (kernels_shade.cu miss_kernel<BLACK_ENV>).  The shortcut must not change a single bit of the sums."""
    from conftest import native_scene, params_for
    p = params_for("part2_all", 320, 180, 24, seed=6)
    monkeypatch.setenv("FW_BLACK_ENV_SKIP", "0")
    ns = native_scene("part2_all")
    _, full, st_full = ns.render(p, want_rgb=False)
    ns.close()
    monkeypatch.setenv("FW_BLACK_ENV_SKIP", "1")
    ns = native_scene("part2_all")
    _, fast, st_fast = ns.render(p, want_rgb=False)
    ns.close()
    assert st_full["rays"] == st_fast["rays"]
    assert np.array_equal(np.isnan(full), np.isnan(fast))
    ok = ~np.isnan(full)
    assert np.array_equal(full[ok], fast[ok])


def _store_stats():
    from firework_b200.engine import texture_store_stats
    return texture_store_stats()


def test_texture_store_shares_resident_texels_and_sees_changed_content(monkeypatch):
    """Texture store (api.cu): a second scene handed the same HDR map / image shares the resident array (no upload, identical
    image, also while the first scene is still alive); changed texels of the same geometry are uploaded again and the image
    follows them; FW_TEXTURE_CACHE=0 uploads every time and gives the same images."""
    from conftest import params_for, scene_text
    from firework_b200.assets import synthetic_hdr
    from firework_b200.engine import release_cached_memory
    release_cached_memory()
    hdr_a = synthetic_hdr(512, 256, 3)
    hdr_b = hdr_a.copy()
    hdr_b[:, :256] *= 0.25
    text = scene_text("hdri_test")
    key = [l for l in text.splitlines() if "synthetic_hdr" in l][0].split("value:")[1].strip()
    p = params_for("hdri_test", 200, 100, 8, seed=4)

    def render(hdr, keep=False):
        before = _store_stats()
        ns = NativeScene(text, assets={key: hdr})
        rgb, s, _ = ns.render(p)
        after = _store_stats()
        bytes_up = ns.device_bytes()
        if not keep:
            ns.close()
        return rgb, s, after["hits"] - before["hits"], after["uploads"] - before["uploads"], bytes_up, ns

    rgb1, s1, hit1, up1, bytes1, _ = render(hdr_a)
    assert (hit1, up1) == (0, 1) and bytes1 >= hdr_a.shape[0] * hdr_a.shape[1] * 16
    rgb2, s2, hit2, up2, bytes2, live = render(hdr_a, keep=True)          # same content: shared, nothing uploaded
    assert (hit2, up2) == (1, 0) and bytes2 < 512 * 256 * 16
    assert np.array_equal(s1, s2) and np.array_equal(rgb1, rgb2)
    rgb3, s3, hit3, up3, _, _ = render(hdr_a)                               # ... also while another scene is using the array
    assert (hit3, up3) == (1, 0) and np.array_equal(s1, s3)
    live.close()
    rgb4, s4, hit4, up4, _, _ = render(hdr_b)                               # same geometry, other content: uploaded
    assert (hit4, up4) == (0, 1) and not np.array_equal(s1, s4)
    rgb5, s5, hit5, up5, _, _ = render(hdr_a)                               # the first content again (idle array refilled or kept)
    assert np.array_equal(s1, s5)
    monkeypatch.setenv("FW_TEXTURE_CACHE", "0")
    rgb6, s6, hit6, up6, _, _ = render(hdr_b)
    assert (hit6, up6) == (0, 1) and np.array_equal(s4, s6)
    monkeypatch.delenv("FW_TEXTURE_CACHE")
    # image textures (RGBA8) go through the same store
    pe = params_for("earth", 160, 160, 4, seed=2)
    from conftest import native_scene
    outs = []
    for _ in range(2):
        before = _store_stats()
        ns = native_scene("earth")
        _, s, _ = ns.render(pe, want_rgb=False)
        ns.close()
        after = _store_stats()
        outs.append((s, after["hits"] - before["hits"], after["uploads"] - before["uploads"]))
    assert outs[1][1] >= 1 and outs[1][2] == 0 and np.array_equal(outs[0][0], outs[1][0])
    release_cached_memory()
    assert _store_stats()["arrays"] == 0


def test_idle_contexts_give_their_memory_back_when_an_allocation_fails():
    """Render contexts are cached with their path state (gigabytes at full batch size).  A process that has rendered many large
    scenes must still be able to start a small one next to a live scene: on an allocation failure the idle contexts are
    destroyed and the allocation is retried (api.cu destroy_idle_contexts)."""
    from conftest import native_scene, params_for
    from firework_b200.engine import release_cached_memory
    release_cached_memory()
    # four idle contexts: three grown to a full 128 Mi-path batch (~53 GB each for cornell_box's two materials), the fourth to what
    # was left — the device is nearly full of memory nobody is using
    held = []
    for _ in range(4):
        ns = native_scene("cornell_box")
        ns.render(params_for("cornell_box", 2048, 2048, 32, seed=1), want_rgb=False, want_sum=False)   # 128 Mi paths
        held.append(ns)
    for ns in held:
        ns.close()
    live = native_scene("cornell_box")                               # takes one of them over
    live.render(params_for("cornell_box", 256, 256, 4, seed=1), want_rgb=False, want_sum=False)
    # random_spheres has materials cornell_box lacks: the context it takes over must add their queues at its full capacity
    # (19 GB) — that allocation fails, the idle contexts are released, the render goes through
    small = native_scene("random_spheres")
    rgb, s, _ = small.render(params_for("random_spheres", 96, 64, 4, seed=2))
    assert np.isfinite(s).all() and rgb.std() > 1
    ref = native_scene("random_spheres")
    _, s2, _ = ref.render(params_for("random_spheres", 96, 64, 4, seed=2))
    assert np.array_equal(s, s2)
    small.close(); ref.close(); live.close()
    release_cached_memory()
