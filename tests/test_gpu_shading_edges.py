"""Shading stages against the oracle at their edges: textures, scatter, the production sampler, resolve, environment.

Every output is compared bit for bit (NaN against NaN, any payload).  The only rows allowed to differ are those a test
marks as a transcendental decision flip: the float64 value of the `sinf` / `powf` / `atan2f` / `asinf` input lies within
a few ulp of the decision it feeds (sign of the checker product, Schlick coin, u8 threshold, texel edge).  An excused row
must equal the result of one of the branches that decision chooses between, and each test prints and bounds its count.
Marble has no decision but a continuous `sinf`: its differing rows must lie within 4 ulp of the float64 value on both sides.
"""
import itertools

import numpy as np
import pytest

from firework_b200.api import (CheckerTexture, ColorEnv, ConstantTexture, DielectricMat, EmissiveMat, HdrEnvironment,
                               ImageTexture, IsotropicMat, LambertianMat, MarbleTexture, MetalMat, PerlinNoiseTexture,
                               RenderObject, Scene, SkyEnv, Sphere, TurbulenceTexture, Vec3)
from firework_b200._native import FireworkError
from firework_b200.engine import NativeScene, resolve_host
from oracle import oracle as oracle_mod
from oracle.oracle import OracleScene

pytestmark = pytest.mark.gpu

F = np.float32
ULPS = 4            # "a few ulp": how close to a decision a float64 transcendental input must be for a flip to be excused
MAX_TEX_DEPTH = 64  # FW_MAX_TEXTURE_DEPTH (fw_types.h)


def _same(g, r):
    """Elementwise: bit-equal, or NaN on both sides."""
    g, r = np.asarray(g, F), np.asarray(r, F)
    gn, rn = np.isnan(g), np.isnan(r)
    return (gn == rn) & (gn | (g.view(np.uint32) == r.view(np.uint32)))


def _rows_same(g, r):
    s = _same(g, r)
    return s.reshape(len(s), -1).all(axis=1)


def _nudge(x, k):
    """x moved k float32 ulps (k may be negative)."""
    x = np.asarray(x, F).copy()
    for _ in range(abs(k)):
        x = np.nextafter(x, F(np.inf) if k > 0 else F(-np.inf)).astype(F)
    return x


class _Pair:
    """One scene on the device and in the oracle; images / HDR maps handed to both through `assets`."""

    def __init__(self, materials, env=None, assets=None):
        s = Scene.new()
        self.mat = [s.add_material(m) for m in materials]
        s.add_object(RenderObject.new(Sphere(1.0, 0)))
        if env is not None:
            s.set_environment(env)
        assets = assets or {}
        self.ns = NativeScene(s.to_yaml(), assets=assets)
        self.orc = OracleScene(s.to_dict(), False, asset_loader=lambda path, kind: assets[path])

    def tex(self, m):
        t = self.ns.material_texture(m)
        assert t == self.orc.tex_of_material[m] and t >= 0
        return t

    def close(self):
        self.ns.close()


def _image(w, h, seed):
    rng = np.random.default_rng(seed)
    img = rng.integers(0, 256, (h, w, 4), dtype=np.uint8)
    img[..., 0] = (np.arange(w * h) % 251).reshape(h, w)   # every texel distinct in R for small maps
    return img


# ---- A. textures ------------------------------------------------------------------------------------------------------
IMAGE_SIZES = [(1, 1), (1, 7), (7, 1), (3, 5), (257, 129)]


def _coord_values():
    ints = F([1, 2, -3, 255, 256, 1 << 23, 1 << 24])
    v = [F(0), F(-0.0), F(0.5), F(-0.5), F(2.5), F(-7.25), F(1e-3), F(123.456), F(-254.5), F(255.99),
         F(2.0 ** 31), F(2.0 ** 63), F(1e30), F(-1e30), F(3.4e38), F(np.inf), F(-np.inf), F(np.nan), -F(np.nan), F(1e-45)]
    v += list(ints) + list(-ints) + list(_nudge(ints, 1)) + list(_nudge(ints, -1)) + list(_nudge(-ints, 1))
    return np.array(v, F)


def _points():
    v = _coord_values()
    core = v[[0, 1, 2, 4, 5, 10, 11, 12, 13, 15, 16, 17, 18, 20, 25, 27, 30, 35]]
    grid = np.array(list(itertools.product(core, core, core)), F)
    rng = np.random.default_rng(21)
    rows = [grid]
    for axis in range(3):   # every value on each axis, the other two random
        p = rng.uniform(-20, 20, (len(v), 3)).astype(F)
        p[:, axis] = v
        rows.append(p)
    rows.append(rng.uniform(-50, 50, (4000, 3)).astype(F))
    rows.append(np.floor(rng.uniform(-300, 300, (1000, 3))).astype(F))          # lattice points
    inf, nan = F(np.inf), F(np.nan)
    rows.append(np.array([(inf, 1, 1), (1, inf, 1), (1, 1, -inf), (1e38, 1, 1), (inf, inf, inf), (inf, nan, 1),
                          (nan, inf, 1), (1, 1, nan), (1, 1, -nan)], F))         # the checker's NaN-sign table
    return np.concatenate(rows)


def _uvs(w, h):
    one = F(1)
    u = [F(0), F(-0.0), one, _nudge(one, -1), _nudge(one, 1), F(-0.25), F(1.5), F(np.inf), F(-np.inf), F(np.nan),
         F(1e-30), F(0.5)]
    for n in (w, h):
        e = (np.arange(n + 1) / F(n)).astype(F)
        u += list(e) + list(_nudge(e, 1)) + list(_nudge(e, -1))
    u = np.unique(np.array(u, F).view(np.uint32)).view(F)
    return np.array(list(itertools.product(u, u)), F)


def _texture_cases():
    """(name, texture, leaves) — leaves: the non-checker textures a checker chooses among."""
    c1, c2, c3 = ConstantTexture(Vec3(0.25, 0.5, 0.75)), ConstantTexture(Vec3(1.0, 0.0, 2.0)), ConstantTexture(Vec3(0.1, 0.2, 0.3))
    img = ImageTexture("img_3x5")
    cases = [("constant", c1, [])]
    for s in (0.0, -3.5, 1e-3, 4.0, 100.0):
        cases.append((f"checker_{s}", CheckerTexture(c1, c2, s), [c1, c2]))
    cases.append(("checker_nested", CheckerTexture(CheckerTexture(c1, c2, 2.0), CheckerTexture(img, c3, 0.5), 3.0), [c1, c2, img, c3]))
    for s in (0.0, -2.0, 1e-3, 1.0, 100.0):
        cases.append((f"perlin_{s}", PerlinNoiseTexture(s), []))
    for d in (0, 1, 7, 300):
        for s in ((1.0, -2.5) if d != 7 else (0.0, 1e-3, 1.0, -2.5, 100.0)):
            cases.append((f"turbulence_{d}_{s}", TurbulenceTexture(d, s), []))
            cases.append((f"marble_{d}_{s}", MarbleTexture(d, s), [TurbulenceTexture(d, 1.0)]))
    for w, h in IMAGE_SIZES:
        cases.append((f"image_{w}x{h}", ImageTexture(f"img_{w}x{h}"), []))
    return cases


def _image_assets():
    return {f"img_{w}x{h}": _image(w, h, w * 1000 + h) for w, h in IMAGE_SIZES}


def _checker_flip_rows(scale, pts):
    """Rows where some sinf input scale*coord (float32) lies within ULPS ulp of a multiple of pi (not at 0 itself)."""
    with np.errstate(invalid="ignore", over="ignore"):
        a = (F(scale) * pts).astype(F)
        near = np.abs(np.sin(a.astype(np.float64))) <= ULPS * np.spacing(np.abs(a)).astype(np.float64)
    return (near & np.isfinite(a) & (a != 0)).any(axis=1)


def _marble_reference(scale, pts, turb):
    """0.5 * (1 + sin(arg)) in float64 for the float32 arg = scale*z + 10*turb (turb: the bit-exact Turbulence output)."""
    with np.errstate(invalid="ignore", over="ignore"):
        arg = ((F(scale) * pts[:, 2]).astype(F) + (F(10.0) * turb).astype(F)).astype(F)
        return 0.5 * (1.0 + np.sin(arg.astype(np.float64)))


class _TextureScene(_Pair):
    def __init__(self, cases):
        mats, self.index = [], {}
        for name, tex, leaves in cases:
            self.index[name] = (len(mats), list(range(len(mats) + 1, len(mats) + 1 + len(leaves))))
            mats.append(LambertianMat(tex))
            mats += [LambertianMat(t) for t in leaves]
        super().__init__(mats, assets=_image_assets())


def texture_compare(pair, name, uv, pts, g=None):
    """Device vs oracle for one texture case under the accounting rule; returns the number of excused rows.
    `g` (optional) is a device result obtained another way for the same rows (e.g. a scatter step's attenuation)."""
    m, leaves = pair.index[name]
    tex = pair.tex(m)
    if g is None:
        g = pair.ns.texture_sample(tex, uv, pts)
    r = pair.orc.texture_sample(tex, uv, pts)
    assert np.array_equal(np.isnan(g), np.isnan(r)), f"{name}: NaN outputs differ"
    bad = ~_rows_same(g, r)
    excused = np.zeros(len(r), bool)
    if name.startswith("checker"):
        scales = [float(name.split("_")[1])] if name != "checker_nested" else [3.0, 2.0, 0.5]
        near = np.zeros(len(r), bool)
        for s in scales:
            near |= _checker_flip_rows(s, pts)
        excused = bad & near
        cand = [pair.orc.texture_sample(pair.tex(lm), uv, pts) for lm in leaves]
        for i in np.flatnonzero(excused):    # the flipped row took the other branch: one of the leaves' colours
            assert any(_same(g[i], c[i]).all() for c in cand), (name, pts[i], g[i], r[i])
    elif name.startswith("marble"):
        scale = float(name.split("_")[2])
        turb = pair.orc.texture_sample(pair.tex(leaves[0]), uv, pts)[:, 0]
        ref = _marble_reference(scale, pts, turb)
        tol = 4 * np.spacing(F(1))    # sinf within 2 ulp on each side, plus the two roundings of 0.5 * (1 + s)
        with np.errstate(invalid="ignore"):
            close = (np.abs(g[:, 0] - ref) <= tol) & (np.abs(r[:, 0] - ref) <= tol)
        excused = bad & close
    if (bad & ~excused).any():
        pytest.fail(f"{name}: {(bad & ~excused).sum()} rows differ, e.g.\n" + "\n".join(
            f"uv={uv[i].tolist()} point={pts[i].tolist()}: {g[i].tolist()} vs {r[i].tolist()}" for i in np.flatnonzero(bad & ~excused)[:8]))
    return int(excused.sum())


@pytest.fixture(scope="module")
def texture_pair():
    p = _TextureScene(_texture_cases())
    yield p
    p.close()


def test_textures_at_their_edges(texture_pair):
    pts = _points()
    rng = np.random.default_rng(4)
    uv = rng.uniform(-0.1, 1.1, (len(pts), 2)).astype(F)
    excused = {}
    for name, _, _ in _texture_cases():
        if name.startswith("image"):
            w, h = map(int, name.split("_")[1].split("x"))
            u = _uvs(w, h)
            excused[name] = texture_compare(texture_pair, name, u, np.zeros((len(u), 3), F))
        else:
            excused[name] = texture_compare(texture_pair, name, uv, pts)
    for name in excused:
        if not name.startswith(("checker", "marble")):
            assert excused[name] == 0, name     # no transcendental: bit for bit
    flips = {k: v for k, v in excused.items() if v}
    print(f"texture rows excused ({len(pts)} points per texture): {flips or 'none'}")
    assert sum(v for k, v in excused.items() if k.startswith("checker")) <= 16
    # marble: sinf differs from glibc's by an ulp on several percent of inputs; each such row is held to the float64 value
    assert all(v <= len(pts) * 15 // 100 for k, v in excused.items() if k.startswith("marble"))


def test_checker_nan_sign_follows_the_reference(texture_pair):
    """Non-finite points: the first axis whose sin is NaN decides, with x86's NaN sign (DESIGN.md §3)."""
    inf, nan = F(np.inf), F(np.nan)
    pts = np.array([(inf, 1, 1), (1, inf, 1), (1, 1, -inf), (1e38, 1, 1), (inf, inf, inf), (inf, nan, 1),
                    (nan, inf, 1), (1, 1, nan), (1, 1, -nan), (0, 1, 1), (-0.0, 1, 1), (-inf, 0, 1), (1, inf, nan), (1, nan, -inf)], F)
    want_odd = [True, True, True, True, True, True, False, False, True, False, True, True, True, False]
    m, leaves = texture_pair.index["checker_4.0"]
    uv = np.zeros((len(pts), 2), F)
    odd = texture_pair.orc.texture_sample(texture_pair.tex(leaves[0]), uv, pts)
    for who, out in (("oracle", texture_pair.orc.texture_sample(texture_pair.tex(m), uv, pts)),
                     ("device", texture_pair.ns.texture_sample(texture_pair.tex(m), uv, pts))):
        got = (out == odd).all(axis=1)
        assert got.tolist() == want_odd, (who, [(tuple(p), w) for p, g_, w in zip(pts, got, want_odd) if g_ != w])


def _checker_chain(depth):
    """`depth` textures on one path: depth - 1 nested checkers over a constant."""
    t = ConstantTexture(Vec3(0.2, 0.4, 0.8))
    for _ in range(depth - 1):
        t = CheckerTexture(t, ConstantTexture(Vec3(0.2, 0.4, 0.8)), 1.0)
    return t


def test_texture_tree_depth_limit():
    """The deepest tree the device follows matches the oracle; one level more is refused when the scene loads."""
    pair = _Pair([LambertianMat(_checker_chain(MAX_TEX_DEPTH))])
    try:
        pts = np.random.default_rng(2).uniform(-5, 5, (256, 3)).astype(F)
        uv = np.zeros((256, 2), F)
        t = pair.tex(0)
        g, r = pair.ns.texture_sample(t, uv, pts), pair.orc.texture_sample(t, uv, pts)
        assert np.array_equal(g, r) and np.all(r == F([0.2, 0.4, 0.8]))
    finally:
        pair.close()
    s = Scene.new()
    s.add_material(LambertianMat(_checker_chain(MAX_TEX_DEPTH + 1)))
    s.add_object(RenderObject.new(Sphere(1.0, 0)))
    with pytest.raises(FireworkError, match=f"deeper than {MAX_TEX_DEPTH}"):
        NativeScene(s.to_yaml())


# ---- B. scatter with explicit uniforms --------------------------------------------------------------------------------
NU = 128
SCATTER_TEXTURES = ["constant", "checker_4.0", "checker_nested", "perlin_1.0", "turbulence_7_1.0", "marble_7_1.0", "image_3x5"]


def _hits():
    """(ray_d, normal) pairs: grazing, head-on, inside, TIR sweeps, non-unit / zero normals, extreme magnitudes."""
    rng = np.random.default_rng(8)
    d, n = [], []
    ny = F([0, 1, 0])
    tiny = [0.0, -0.0, 1e-45, -1e-45, 1e-38, -1e-38, 1e-7, -1e-7]
    for nrm in (ny, F([0, 2.5, 0]), F([0.18, 0.0, -0.24])):
        u = nrm / np.linalg.norm(nrm)
        t = np.cross(u, F([0.0, 0.0, 1.0])) if abs(u[2]) < 0.9 else F([1, 0, 0])
        t = (t / np.linalg.norm(t)).astype(F)
        for e in tiny:                               # grazing: dot(d, n) = 0 and a denormal / few ulp either side
            d.append(t + F(e) * u); n.append(nrm)
        for v in (-u, u, -nrm, nrm):                 # head-on and from inside
            d.append(v); n.append(nrm)
    for r in (1.33, 1.5, 2.42):                      # from inside near the critical angle: disc crosses 0
        c = F(np.sqrt(1 - 1 / F(r) ** 2))
        for k in range(-6, 7):
            dt = _nudge(c, k)
            d.append(F([np.sqrt(max(0.0, 1 - float(dt) ** 2)), dt, 0])); n.append(ny)
    n0 = np.array(n, F)
    nrand = rng.normal(size=(48, 3)).astype(F)
    nrand /= np.linalg.norm(nrand, axis=1, keepdims=True)
    nrand[:8] *= F(0.3)                              # non-unit
    nrand[8:12] = 0                                  # zero
    drand = rng.normal(size=(48, 3)).astype(F)
    mags = F([1e-30, 1e-20, 1e-10, 1.0, 1e10, 1e20, 1e30, 0.0])
    dd = np.concatenate([drand * m for m in mags] + [np.full((4, 3), np.nan, F), np.array([[np.inf, 0, 0], [0, -np.inf, 1]], F)])
    nn = np.concatenate([nrand] * len(mags) + [nrand[:6]])
    return np.concatenate([np.array(d, F), dd]).astype(F), np.concatenate([n0, nn]).astype(F)


def _streams(rng):
    """Named uniform streams of NU values: p = 0, rejection chains of 1..40 rounds, random, overrun."""
    out = {"half": np.full(NU, 0.5, F)}
    acc = F([0.3, 0.6, 0.55])
    for k in (1, 2, 3, 4, 5, 8, 16, 40):
        s = (np.floor(rng.uniform(0, 1, NU) * 16777216) / 16777216).astype(F)
        s[:3 * (k - 1)] = np.tile(F([0.99, 0.01, 0.99]), k - 1)
        s[3 * (k - 1):3 * k] = acc
        out[f"chain{k}"] = s
    out["random"] = (np.floor(rng.uniform(0, 1, NU) * 16777216) / 16777216).astype(F)
    out["overrun"] = np.full(NU, 0.99, F)
    return out


def _schlick64(ref, d, n):
    """The dielectric's Schlick value in float64 from the float32 cosine the material computes."""
    with np.errstate(all="ignore"):
        return _schlick64_f32(ref, d, n)


def _schlick64_f32(ref, d, n):
    dot = ((d[:, 0] * n[:, 0]).astype(F) + (d[:, 1] * n[:, 1]).astype(F)).astype(F) + (d[:, 2] * n[:, 2]).astype(F)
    dot = dot.astype(F)
    mag = np.sqrt((((d[:, 0] * d[:, 0]).astype(F) + (d[:, 1] * d[:, 1]).astype(F)).astype(F) + (d[:, 2] * d[:, 2]).astype(F)).astype(F))
    with np.errstate(all="ignore"):
        cos = np.where(dot > 0, ((F(ref) * dot).astype(F) / mag).astype(F), (-dot / mag).astype(F)).astype(F)
        r0 = F((F(1) - F(ref)) / (F(1) + F(ref)))
        r0 = F(r0 * r0)
        return float(r0) + float(F(1) - r0) * (1.0 - cos.astype(F)).astype(F).astype(np.float64) ** 5


def _scatter_scene():
    base = dict((name, tex) for name, tex, _ in _texture_cases())
    mats, kinds = [], []
    for alb in (Vec3(0, 0, 0), Vec3(1.5, 0.5, 2.0)):
        for r in (0.0, 0.3, 1.0, 10.0):
            mats.append(MetalMat(alb, r)); kinds.append(("metal", r))
    for r in (1.0, 1.33, 1.5, 2.42, 0.75):
        mats.append(DielectricMat(r)); kinds.append(("dielectric", r))
    for name in SCATTER_TEXTURES:
        for cls in (LambertianMat, IsotropicMat, EmissiveMat):
            mats.append(cls(base[name])); kinds.append((cls.__name__, name))
    p = _Pair(mats, assets=_image_assets())
    p.kinds = kinds
    return p


@pytest.fixture(scope="module")
def scatter_pair():
    p = _scatter_scene()
    yield p
    p.close()


def _scatter_compare(pair, tp, mats, d, nrm, point, uv, uniforms, what):
    """Device vs oracle scatter step; returns the excused coin rows.  Texture-valued outputs must equal each side's own
    texture lookup bit for bit, and those lookups are compared under the texture accounting."""
    n = len(mats)
    hit_t = np.ones(n, F)
    g = pair.ns.scatter_step(mats, point - d, d, hit_t, point, nrm, uv, uniforms)
    r = pair.orc.scatter_step(mats, point - d, d, hit_t, point, nrm, uv, uniforms)
    assert np.array_equal(g["consumed"], r["consumed"]), what
    live = r["consumed"] >= 0                       # an overrun stream is compared by its consumed == -1 only
    kinds = [pair.kinds[m] for m in mats]
    textured = np.array([k[0] in ("LambertianMat", "IsotropicMat", "EmissiveMat") for k in kinds])
    diel = np.array([k[0] == "dielectric" for k in kinds])
    # texture-valued outputs: each side equals its own lookup; the lookups follow the texture accounting
    for name in SCATTER_TEXTURES:
        for cls, key in (("LambertianMat", "atten"), ("IsotropicMat", "atten"), ("EmissiveMat", "emit")):
            rows = np.flatnonzero(live & np.array([k == (cls, name) for k in kinds]))
            if not len(rows):
                continue
            t = pair.tex(mats[rows[0]])
            assert _same(g[key][rows], pair.ns.texture_sample(t, uv[rows], point[rows])).all(), (what, cls, name)
            assert _same(r[key][rows], pair.orc.texture_sample(t, uv[rows], point[rows])).all(), (what, cls, name)
            texture_compare(tp, name, uv[rows], point[rows], g=g[key][rows])
    fields = ["scattered", "o", "d"] + [k for k in ("atten", "emit")]
    ok = np.ones(n, bool)
    for f in fields:
        s = _same(g[f], r[f])
        s = s.reshape(n, -1).all(axis=1)
        if f in ("atten", "emit"):
            s |= textured
        ok &= s
    ok |= ~live
    bad = ~ok
    excused = np.zeros(n, bool)
    if (bad & diel).any():
        rows = np.flatnonzero(bad & diel)
        for i in rows:
            ref = pair.kinds[mats[i]][1]
            s64 = _schlick64(ref, d[i:i + 1], nrm[i:i + 1])[0]
            u = float(uniforms[i, 0])
            if abs(u - s64) <= ULPS * float(np.spacing(np.abs(F(s64)))):
                excused[i] = True
        if excused.any():          # the flipped rows took the other branch: reflect or refract
            ex = np.flatnonzero(excused)
            ok_alt = np.zeros(len(ex), bool)
            for coin in (F(-np.inf), F(np.inf)):   # u > schlick never / always holds
                un = uniforms[ex].copy(); un[:, 0] = coin
                alt = pair.orc.scatter_step(mats[ex], point[ex] - d[ex], d[ex], hit_t[ex], point[ex], nrm[ex], uv[ex], un)
                ok_alt |= _rows_same(g["d"][ex], alt["d"])
            assert ok_alt.all(), (what, ex[~ok_alt])
    if (bad & ~excused).any():
        pytest.fail(f"{what}: {(bad & ~excused).sum()} rows differ, e.g.\n" + "\n".join(
            f"{kinds[i]} d={d[i].tolist()} n={nrm[i].tolist()} u={uniforms[i, :4].tolist()} "
            + " ".join(f"{f}: {np.asarray(g[f][i]).tolist()} vs {np.asarray(r[f][i]).tolist()}" for f in fields if not _same(g[f][i], r[f][i]).all())
            for i in np.flatnonzero(bad & ~excused)[:6]))
    return int(excused.sum()), int((~live).sum())


def test_scatter_with_explicit_uniforms(scatter_pair, texture_pair):
    rng = np.random.default_rng(31)
    d, nrm = _hits()
    nh = len(d)
    streams = _streams(rng)
    total_ex, total_over, rows = 0, 0, 0
    for m in range(len(scatter_pair.kinds)):
        for sname, s in streams.items():
            mats = np.full(nh, m, np.int32)
            point = rng.uniform(-6, 6, (nh, 3)).astype(F)
            point[:8] = F([[0, 0, 0], [1, 1, 1], [-2, 3, -4], [2 ** 24, 0.5, -0.5], [np.inf, 1, 1], [np.nan, 0, 0],
                           [1e30, -1e30, 1], [255.5, 256, 257]])
            uv = rng.uniform(-0.1, 1.1, (nh, 2)).astype(F)
            uniforms = np.tile(s, (nh, 1))
            ex, over = _scatter_compare(scatter_pair, texture_pair, mats, d, nrm, point, uv, uniforms, (scatter_pair.kinds[m], sname))
            total_ex += ex; total_over += over; rows += nh
    # Schlick coins placed at and around the float64 Schlick value of each dielectric row
    for m, (kind, ref) in enumerate(scatter_pair.kinds):
        if kind != "dielectric":
            continue
        s64 = _schlick64(ref, d, nrm)
        for k in (-2, -1, 0, 1, 2):
            uniforms = np.tile(streams["random"], (nh, 1))
            with np.errstate(invalid="ignore"):
                uniforms[:, 0] = _nudge(np.where(np.isfinite(s64), s64, 0.5).astype(F), k)
            mats = np.full(nh, m, np.int32)
            point = rng.uniform(-6, 6, (nh, 3)).astype(F)
            uv = np.zeros((nh, 2), F)
            ex, over = _scatter_compare(scatter_pair, texture_pair, mats, d, nrm, point, uv, uniforms, ("coin", ref, k))
            total_ex += ex; total_over += over; rows += nh
    print(f"scatter: {rows} rows, {total_ex} Schlick-coin rows excused, {total_over} overrun rows (consumed == -1)")
    assert total_over > 0
    assert total_ex <= 64


# ---- C. the production sampler, keyed ---------------------------------------------------------------------------------
def test_keyed_scatter_through_the_production_sampler(scatter_pair, texture_pair):
    """The shade kernels' sampler (random_in_unit_sphere_fresh on a keyed PhiloxStream) against the oracle's own keyed
    Philox stream and plain rejection loop, with every acceptance round 1..4 and the fallback loop covered."""
    kinds = scatter_pair.kinds
    pick = [kinds.index(k) for k in (("LambertianMat", "constant"), ("metal", 0.3), ("metal", 1.0), ("IsotropicMat", "constant"),
                                     ("dielectric", 1.5), ("metal", 10.0))]
    rng = np.random.default_rng(77)
    n = 12288
    mats = np.array(pick, np.int32)[np.arange(n) % len(pick)]
    d = rng.normal(size=(n, 3)).astype(F)
    nrm = rng.normal(size=(n, 3)).astype(F)
    nrm /= np.linalg.norm(nrm, axis=1, keepdims=True)
    point = rng.uniform(-5, 5, (n, 3)).astype(F)
    uv = rng.uniform(0, 1, (n, 2)).astype(F)
    hit_t = np.ones(n, F)
    seed = 0x1234_5678_9ABC
    pixel = rng.integers(0, 1 << 32, n, dtype=np.uint64).astype(np.uint32)
    sample = rng.integers(0, 1 << 20, n).astype(np.uint32)
    bounce = rng.integers(0, 11, n).astype(np.uint32)
    args = (mats, point - d, d, hit_t, point, nrm, uv, seed, pixel, sample, bounce)
    r = scatter_pair.orc.scatter_step_keyed(*args)
    g = scatter_pair.ns.scatter_step_keyed(*args)
    sphere = np.array([kinds[m][0] != "dielectric" for m in mats])
    rounds = r["consumed"][sphere] // 3
    cover = {k: int((rounds == k).sum()) for k in (1, 2, 3, 4)}
    cover[">4"] = int((rounds > 4).sum())
    print(f"keyed sampler: acceptance rounds {cover}")
    assert all(v >= 100 for v in cover.values()), cover
    assert np.array_equal(g["consumed"], r["consumed"])
    bad = np.zeros(n, bool)
    for f in ("scattered", "atten", "o", "d", "emit"):
        bad |= ~_rows_same(g[f], r[f])
    excused = np.zeros(n, bool)
    for i in np.flatnonzero(bad):
        if kinds[mats[i]][0] == "dielectric":   # the coin: first draw of the row's scatter stream
            ctr = [0, (int(bounce[i]) << 8) | 1, int(sample[i]), int(pixel[i])]
            coin = (oracle_mod.philox(ctr, [seed & 0xFFFFFFFF, seed >> 32])[0] >> 8) / 16777216.0
            s64 = _schlick64(1.5, d[i:i + 1], nrm[i:i + 1])[0]
            excused[i] = abs(coin - s64) <= ULPS * float(np.spacing(np.abs(F(s64))))
    print(f"keyed sampler: {int(excused.sum())} Schlick-coin rows excused")
    assert not (bad & ~excused).any(), [(kinds[mats[i]], g["d"][i], r["d"][i]) for i in np.flatnonzero(bad & ~excused)[:4]]
    assert excused.sum() <= 4


# ---- D. resolve -------------------------------------------------------------------------------------------------------
def _resolve_sums(gamma, samples):
    """Sums whose mean lands at and +-2 ulp around each u8 threshold k / 255.99 after the gamma curve, plus specials."""
    k = np.arange(257, dtype=np.float64)
    x = (k / 255.99).astype(F)
    mean = np.power(x.astype(np.float64), gamma).astype(F)
    base = (mean.astype(np.float64) * float(F(samples))).astype(F)
    vals = [_nudge(base, j) for j in range(-2, 3)]
    special = F([0, -0.0, -0.5, -1e-30, 1e-45, 1e-40, 1.17e-38, 3.4e38, 1e30, np.inf, -np.inf, np.nan, -np.nan, 0.5, 1.0])
    vals.append(special)
    with np.errstate(over="ignore"):
        vals.append((special * F(samples)).astype(F))
    v = np.concatenate(vals)
    pad = (-len(v)) % 3
    return np.concatenate([v, np.zeros(pad, F)]).reshape(-1, 1, 3)


def test_resolve_against_the_oracle():
    total = 0
    for gamma in (1.0, 2.0, 2.2, 0.5):
        for samples in (1, 3, 1000, (1 << 24) + 1):
            sums = _resolve_sums(gamma, samples)
            g = resolve_host(sums, samples, gamma)
            r = oracle_mod.resolve(sums, samples, gamma)
            bad = (g != r).ravel()
            if not bad.any():
                continue
            # excused: powf(mean, 1 / gamma) within ULPS ulp of a value whose *255.99 truncation changes
            s = sums.ravel()
            with np.errstate(all="ignore"):
                mean = (s / F(samples)).astype(F)
                inv = F(F(1) / F(gamma))
                x64 = np.power(mean.astype(np.float64), float(inv))
                lo, hi = _nudge(x64.astype(F), -ULPS), _nudge(x64.astype(F), ULPS)

                def q(x):
                    x = np.clip(x, F(0), F(1))
                    y = (x * F(255.99)).astype(F)
                    return np.where(np.isnan(y), 0, np.trunc(y)).astype(np.int64)
                qlo, qhi = q(lo), q(hi)
            excused = bad & (qlo != qhi) & ((g.ravel() == qlo) | (g.ravel() == qhi))
            assert not (bad & ~excused).any(), (gamma, samples, s[bad & ~excused][:8], g.ravel()[bad & ~excused][:8],
                                                r.ravel()[bad & ~excused][:8])
            total += int(excused.sum())
    print(f"resolve: {total} powf threshold values excused")
    assert total <= 420     # of ~21000 values, most of them placed within 2 ulp of a threshold on purpose


# ---- E. environment ---------------------------------------------------------------------------------------------------
HDR_SIZES = [(1, 1), (2, 1), (1, 2), (5, 3), (512, 256)]


def _env_dirs():
    rng = np.random.default_rng(12)
    z, nz = F(0), F(-0.0)
    fixed = [(0, 1, 0), (0, -1, 0), (z, -1, nz), (nz, 1, z), (-1e-10, -1, 0), (-1e-10, -1, nz), (-1e-10, 1, 0),
             (1, 0, 0), (-1, 0, 0), (0, 0, 1), (0, 0, -1), (-1, 0, nz), (-1, 0, z), (-1, 0.5, nz), (-1, -0.5, z),
             (-1, 1e-45, nz), (-1, -1e-45, z), (1e-45, 1, 1e-45), (1e-40, -1e-40, 1), (1e20, 1e20, 1e20), (3e38, 1, 0),
             (0, 0, 0), (np.nan, 0, 0), (0, np.nan, 1), (np.inf, 0, 0), (1, 1, 1)]
    d = [np.array(fixed, F)]
    for y in np.linspace(-1, 1, 41):
        d.append(np.array([(-1, y, z), (-1, y, nz), (-1e-3, y, 0), (-1e-3, y, nz)], F))
    d.append(rng.normal(size=(20000, 3)).astype(F))
    return np.concatenate(d)


def _normalized(v):
    mag = np.sqrt((((v[:, 0] * v[:, 0]).astype(F) + (v[:, 1] * v[:, 1]).astype(F)).astype(F) + (v[:, 2] * v[:, 2]).astype(F)).astype(F))
    with np.errstate(all="ignore"):
        return (v / mag[:, None]).astype(F)


def _env_indices(dirs, w, h, dphi, dtheta):
    """The texel index the lookup computes, with atan2 / asin taken in float64 and moved dphi / dtheta ulps."""
    pi = F(np.pi)
    with np.errstate(all="ignore"):
        u_ = _normalized(dirs)
        phi = _nudge(np.arctan2(u_[:, 2].astype(np.float64), u_[:, 0].astype(np.float64)).astype(F), dphi)
        theta = _nudge(np.arcsin(u_[:, 1].astype(np.float64)).astype(F), dtheta)
        u = (F(1) - ((phi + pi).astype(F) / (F(2) * pi)).astype(F)).astype(F)
        v = (((theta + (pi / F(2))).astype(F)) / pi).astype(F)

        def cast(f):   # saturating float -> u64 (NaN -> 0)
            f = np.where(np.isnan(f), 0, np.clip(f, 0, 2.0 ** 64 - 1)).astype(np.float64)
            return np.floor(f).astype(np.uint64)
        x = cast((u * F(w)).astype(F))
        y = cast(((F(1) - v).astype(F) * F(h)).astype(F))
        idx = cast((y.astype(F) * F(w)).astype(F)) + x
    return np.minimum(idx, np.uint64(w * h - 1))


def test_environment_lookups_at_their_edges():
    dirs = _env_dirs()
    for env in (ColorEnv(Vec3(0.3, 0.6, 0.9)), SkyEnv(Vec3(0.5, 0.7, 1.0), Vec3(1.0, 0.25, 0.125))):
        p = _Pair([LambertianMat.with_color(Vec3(0.5, 0.5, 0.5))], env=env)
        try:
            g, r = p.ns.env_sample(dirs), p.orc.env_sample(dirs)
            assert _same(g, r).all(), (type(env).__name__, dirs[~_rows_same(g, r)][:8])
        finally:
            p.close()
    total = 0
    for w, h in HDR_SIZES:
        hdr = np.random.default_rng(w * 7 + h).uniform(0, 4, (h, w, 3)).astype(F)
        hdr[..., 0] = np.arange(w * h, dtype=F).reshape(h, w)      # R = texel index
        p = _Pair([LambertianMat.with_color(Vec3(0.5, 0.5, 0.5))], env=HdrEnvironment("hdr"), assets={"hdr": hdr})
        try:
            g, r = p.ns.env_sample(dirs), p.orc.env_sample(dirs)
        finally:
            p.close()
        bad = ~_rows_same(g, r)
        cands = np.stack([_env_indices(dirs, w, h, a, b) for a in range(-ULPS, ULPS + 1) for b in range(-ULPS, ULPS + 1)], 1)
        edge = (cands != cands[:, :1]).any(axis=1)
        flat = hdr.reshape(-1, 3)
        took = (flat[cands.astype(np.int64)] == g[:, None, :]).all(axis=2).any(axis=1)
        excused = bad & edge & took
        if (bad & ~excused).any():
            pytest.fail(f"HDR {w}x{h}: {(bad & ~excused).sum()} rows differ, e.g.\n" + "\n".join(
                f"dir={dirs[i].tolist()}: {g[i].tolist()} vs {r[i].tolist()}" for i in np.flatnonzero(bad & ~excused)[:8]))
        total += int(excused.sum())
    print(f"environment: {total} HDR texel-edge rows excused")
    assert total <= len(dirs) * len(HDR_SIZES) // 500
