"""Host-side mirror of firework's public scene / renderer API.

The reference is a Rust crate; there is no Rust toolchain in this image, so the caller-facing layer that a
`firework` user touches is mirrored here in Python with the same names, argument order and meaning:

    Scene, RenderObject                     (reference: src/scene.rs:19-91, 268-334)
    Sphere, XYRect/XZRect/YZRect, Rect3d, TriangleMesh, Disk, Cylinder, Cone, ConstantMedium
                                            (src/objects/*.rs)
    LambertianMat, MetalMat, DielectricMat, EmissiveMat, IsotropicMat      (src/material.rs)
    ConstantTexture, CheckerTexture, PerlinNoiseTexture, TurbulenceTexture, MarbleTexture, ImageTexture
                                            (src/texture.rs)
    ColorEnv, SkyEnv (src/environment.rs), HdrEnvironment (examples/hdri_test.rs:22-82)
    CameraSettings (src/camera.rs:18-71), Renderer (src/render.rs:57-107, 198-218)
    Rotor3.from_rotation_xz (ultraviolet 0.5.1)

A `Scene` serialises to the *same serde YAML document* the reference reads and writes
(`serde_yaml::to_string(&scene)`, e.g. scenes/conics.yml); that text is the type-erased scene contract
handed across the C ABI (`fw_scene_from_yaml`).  All geometry processing (BVH build with the reference's
split rule, flattening, kernels) happens in the native library, not here.

`Renderer.render(scene)` returns `width*height` (r, g, b) u8 triples, row 0 = top of image, exactly the
`Vec<Color>` of `Renderer::render` (src/render.rs:109).
"""
from __future__ import annotations

import math
import os
from dataclasses import dataclass, field
from typing import List, Optional, Sequence

import numpy as np

F = np.float32


def f32(x) -> float:
    """Round to IEEE f32 and return as a Python float (exactly representable)."""
    return float(F(x))


class Vec3:
    """ultraviolet::Vec3 with f32 component arithmetic (only what scene construction needs)."""

    __slots__ = ("x", "y", "z")

    def __init__(self, x, y, z):
        self.x, self.y, self.z = F(x), F(y), F(z)

    @staticmethod
    def zero():
        return Vec3(0, 0, 0)

    @staticmethod
    def one():
        return Vec3(1, 1, 1)

    @staticmethod
    def broadcast(v):
        return Vec3(v, v, v)

    def __add__(self, o):
        return Vec3(self.x + o.x, self.y + o.y, self.z + o.z)

    def __sub__(self, o):
        return Vec3(self.x - o.x, self.y - o.y, self.z - o.z)

    def __mul__(self, s):
        if isinstance(s, Vec3):
            return Vec3(self.x * s.x, self.y * s.y, self.z * s.z)
        s = F(s)
        return Vec3(self.x * s, self.y * s, self.z * s)

    __rmul__ = __mul__

    def mag(self):
        return F(np.sqrt(self.x * self.x + self.y * self.y + self.z * self.z))

    def to_dict(self):
        return {"x": float(self.x), "y": float(self.y), "z": float(self.z)}

    def __iter__(self):
        return iter((float(self.x), float(self.y), float(self.z)))

    def __repr__(self):
        return f"Vec3({float(self.x)}, {float(self.y)}, {float(self.z)})"


def _v3(v) -> Vec3:
    return v if isinstance(v, Vec3) else Vec3(*v)


@dataclass
class Rotor3:
    """ultraviolet::Rotor3 {s, bv{xy, xz, yz}} (serde layout: src/serde_compat.rs:6-20)."""

    s: float = 1.0
    xy: float = 0.0
    xz: float = 0.0
    yz: float = 0.0

    @staticmethod
    def identity():
        return Rotor3()

    @staticmethod
    def _from_angle_plane(angle, plane):
        # ultraviolet 0.5.1 Rotor3::from_angle_plane: (sin, cos) = (angle * 0.5).sin_cos(); Rotor3::new(cos, plane * -sin).
        # libm's sinf / cosf are correctly rounded: evaluate in f64 and round once.  `plane * -sin` keeps the sign of
        # its zero components (0 * -sin = -0.0 for sin > 0), as the reference's scenes/teapot.yml shows.
        half = F(F(angle) * F(0.5))
        sin, cos = F(math.sin(float(half))), F(math.cos(float(half)))
        bv = [float(F(c) * -sin) for c in plane]
        return Rotor3(float(cos), bv[0], bv[1], bv[2])

    @staticmethod
    def from_rotation_xz(angle):
        # pinned numerically by scenes/suzanne.yml (a = -30 rad) and scenes/teapot.yml (a = 90 rad)
        return Rotor3._from_angle_plane(angle, (0.0, 1.0, 0.0))

    @staticmethod
    def from_rotation_xy(angle):
        return Rotor3._from_angle_plane(angle, (1.0, 0.0, 0.0))

    @staticmethod
    def from_rotation_yz(angle):
        return Rotor3._from_angle_plane(angle, (0.0, 0.0, 1.0))

    def to_dict(self):
        return {"s": f32(self.s), "bv": {"xy": f32(self.xy), "xz": f32(self.xz), "yz": f32(self.yz)}}


def to_radians(deg) -> float:
    """f32::to_radians: self * (PI / 180)."""
    return f32(F(deg) * (F(math.pi) / F(180.0)))


# ---------------------------------------------------------------------------------------------------
# textures (src/texture.rs)
# ---------------------------------------------------------------------------------------------------
class ConstantTexture:
    def __init__(self, color):
        self.color = _v3(color)

    @staticmethod
    def from_rgb(r, g, b):
        return ConstantTexture(Vec3(r, g, b))

    def to_dict(self):
        return {"texture": "ConstantTexture", "color": self.color.to_dict()}


class CheckerTexture:
    def __init__(self, odd, even, scale):
        self.odd, self.even, self.scale = odd, even, f32(scale)

    @staticmethod
    def with_colors(odd, even, scale):
        return CheckerTexture(ConstantTexture(odd), ConstantTexture(even), scale)

    def to_dict(self):
        return {"texture": "CheckerTexture", "odd": self.odd.to_dict(), "even": self.even.to_dict(), "scale": self.scale}


class PerlinNoiseTexture:
    def __init__(self, scale):
        self.scale = f32(scale)

    def to_dict(self):
        return {"texture": "PerlinNoiseTexture", "scale": self.scale}


class TurbulenceTexture:
    def __init__(self, depth, scale):
        self.depth, self.scale = int(depth), f32(scale)

    def to_dict(self):
        return {"texture": "TurbulenceTexture", "depth": self.depth, "scale": self.scale}


class MarbleTexture:
    def __init__(self, depth, scale):
        self.depth, self.scale = int(depth), f32(scale)

    def to_dict(self):
        return {"texture": "MarbleTexture", "depth": self.depth, "scale": self.scale}


class ImageTexture:
    """Serialises as its path (texture.rs:251-278); texels are decoded by the host and registered with the
    native scene (`fw_scene_set_image`)."""

    def __init__(self, path):
        self.path = str(path)

    @staticmethod
    def from_path(path):
        return ImageTexture(path)

    def to_dict(self):
        return {"texture": "ImageTexture", "value": self.path}


# ---------------------------------------------------------------------------------------------------
# materials (src/material.rs)
# ---------------------------------------------------------------------------------------------------
class LambertianMat:
    def __init__(self, albedo):
        self.albedo = albedo

    @staticmethod
    def with_color(albedo):
        return LambertianMat(ConstantTexture(albedo))

    def to_dict(self):
        return {"material": "LambertianMat", "albedo": self.albedo.to_dict()}


class MetalMat:
    def __init__(self, albedo, roughness):
        self.albedo, self.roughness = _v3(albedo), f32(roughness)

    def to_dict(self):
        return {"material": "MetalMat", "albedo": self.albedo.to_dict(), "roughness": self.roughness}


class DielectricMat:
    def __init__(self, ref_idx):
        self.ref_idx = f32(ref_idx)

    def to_dict(self):
        return {"material": "DielectricMat", "ref_idx": self.ref_idx}


class EmissiveMat:
    def __init__(self, albedo):
        self.albedo = albedo

    @staticmethod
    def with_color(albedo):
        return EmissiveMat(ConstantTexture(albedo))

    def to_dict(self):
        return {"material": "EmissiveMat", "albedo": self.albedo.to_dict()}


class IsotropicMat:
    def __init__(self, texture):
        self.texture = texture

    def to_dict(self):
        return {"material": "IsotropicMat", "texture": self.texture.to_dict()}


# ---------------------------------------------------------------------------------------------------
# environments (src/environment.rs, examples/hdri_test.rs)
# ---------------------------------------------------------------------------------------------------
class ColorEnv:
    def __init__(self, color=(0, 0, 0)):
        self.color = _v3(color)

    def to_dict(self):
        return {"environment": "ColorEnv", "color": self.color.to_dict()}


class SkyEnv:
    def __init__(self, zenith_color=(0.5, 0.7, 1.0), horizon_color=(1.0, 1.0, 1.0)):
        self.zenith_color, self.horizon_color = _v3(zenith_color), _v3(horizon_color)

    @staticmethod
    def default():
        return SkyEnv()

    def to_dict(self):
        return {"environment": "SkyEnv", "zenith_color": self.zenith_color.to_dict(),
                "horizon_color": self.horizon_color.to_dict()}


class HdrEnvironment:
    """Equirectangular fp32 map; lives in examples/hdri_test.rs in the reference and serialises as its path."""

    def __init__(self, path):
        self.path = str(path)

    @staticmethod
    def from_path(path):
        return HdrEnvironment(path)

    def to_dict(self):
        return {"environment": "HdrEnvironment", "value": self.path}


# ---------------------------------------------------------------------------------------------------
# shapes (src/objects/*.rs)
# ---------------------------------------------------------------------------------------------------
def add_obj(scene, file_name, material, with_normals=False, rotate=None):
    """The `add_obj` helper of examples/suzanne.rs:15-51 (with_normals=False) and examples/teapot.rs:17-64
    (with_normals=True, rotate=Rotor3.from_rotation_xz(90.)): one TriangleMesh render object per OBJ model."""
    from .assets import load_obj
    ids = []
    for m in load_obj(str(file_name)):
        normals = m["normals"] if with_normals else None
        obj = RenderObject.new(TriangleMesh(m["positions"], m["indices"], normals, None, material))
        if rotate is not None:
            obj = obj.rotate(rotate)
        ids.append(scene.add_object(obj))
    return ids


class Sphere:
    def __init__(self, radius, material):
        self.radius, self.material = f32(radius), int(material)

    def to_dict(self):
        return {"object_type": "Sphere", "radius": self.radius, "material": self.material}


class _AARect:
    TAG = ""

    def __init__(self, a1_min, a1_max, a2_min, a2_max, k, material):
        self.min = (f32(a1_min), f32(a2_min))
        self.max = (f32(a1_max), f32(a2_max))
        self.k, self.material, self._flip = f32(k), int(material), False

    def flip_normal(self):
        self._flip = True
        return self

    def fields(self):
        return {"min": {"x": self.min[0], "y": self.min[1]}, "max": {"x": self.max[0], "y": self.max[1]},
                "k": self.k, "flip_normal": self._flip, "material": self.material}

    def to_dict(self):
        d = {"object_type": self.TAG}
        d.update(self.fields())
        return d


class XYRect(_AARect):
    TAG = "XYRect"


class XZRect(_AARect):
    TAG = "XZRect"


class YZRect(_AARect):
    TAG = "YZRect"


class Rect3d:
    """rect3d.rs:18-87 — six faces in the order +z, -z, +y, -y, +x, -x, all arithmetic in f32."""

    def __init__(self, pos, size, material):
        p, s = _v3(pos), _v3(size)
        self.pos, self.size = p, s
        m = int(material)
        self.faces = [
            ("XY", XYRect(p.x, p.x + s.x, p.y, p.y + s.y, p.z + s.z, m)),
            ("XY", XYRect(p.x, p.x + s.x, p.y, p.y + s.y, p.z, m).flip_normal()),
            ("XZ", XZRect(p.x, p.x + s.x, p.z, p.z + s.z, p.y + s.y, m)),
            ("XZ", XZRect(p.x, p.x + s.x, p.z, p.z + s.z, p.y, m).flip_normal()),
            ("YZ", YZRect(p.y, p.y + s.y, p.z, p.z + s.z, p.x + s.x, m)),
            ("YZ", YZRect(p.y, p.y + s.y, p.z, p.z + s.z, p.x, m).flip_normal()),
        ]

    @staticmethod
    def with_size(size, material):
        return Rect3d(Vec3.zero(), size, material)

    def to_dict(self):
        return {"object_type": "Rect3d", "pos": self.pos.to_dict(), "size": self.size.to_dict(),
                "faces": [{tag: r.fields()} for tag, r in self.faces]}


class TriangleMesh:
    def __init__(self, verts, indicies, normals, uvs, material):
        self.verts = np.asarray(verts, dtype=np.float32).reshape(-1, 3)
        self.indicies = np.asarray(indicies, dtype=np.int64).reshape(-1)
        self.normals = None if normals is None else np.asarray(normals, dtype=np.float32).reshape(-1, 3)
        self.uvs = None if uvs is None else np.asarray(uvs, dtype=np.float32).reshape(-1, 2)
        if self.normals is not None and len(self.normals) != len(self.verts):
            raise ValueError("TriangleMesh::new() -- normals.len() must equal verts.len()")
        if self.uvs is not None and len(self.uvs) != len(self.verts):
            raise ValueError("TriangleMesh::new() -- uvs.len() must equal verts.len()")
        self.material = int(material)

    def to_dict(self):
        def v3list(a):
            return [{"x": float(r[0]), "y": float(r[1]), "z": float(r[2])} for r in a]

        return {"object_type": "TriangleMesh", "indicies": [int(i) for i in self.indicies],
                "verts": v3list(self.verts),
                "normals": None if self.normals is None else v3list(self.normals),
                "uvs": None if self.uvs is None else [{"x": float(r[0]), "y": float(r[1])} for r in self.uvs],
                "material": self.material}


class Disk:
    def __init__(self, radius, material):
        self.radius, self.phi_max, self.inner_radius, self.material = f32(radius), f32(F(2.0) * F(math.pi)), 0.0, int(material)

    @staticmethod
    def partial(radius, phi, inner_radius, material):
        d = Disk(radius, material)
        d.phi_max, d.inner_radius = to_radians(phi), f32(inner_radius)
        return d

    def to_dict(self):
        return {"object_type": "Disk", "radius": self.radius, "phi_max": self.phi_max,
                "inner_radius": self.inner_radius, "material": self.material}


class Cylinder:
    def __init__(self, radius, height, material):
        self.radius, self.height, self.max_phi, self.material = f32(radius), f32(height), to_radians(360.0), int(material)

    @staticmethod
    def partial(radius, height, phi, material):
        c = Cylinder(radius, height, material)
        c.max_phi = to_radians(phi)
        return c

    def to_dict(self):
        return {"object_type": "Cylinder", "radius": self.radius, "height": self.height, "max_phi": self.max_phi,
                "material": self.material}


class Cone:
    def __init__(self, radius, height, material):
        self.radius, self.height, self.material = f32(radius), f32(height), int(material)

    def to_dict(self):
        return {"object_type": "Cone", "radius": self.radius, "height": self.height, "material": self.material}


class ConstantMedium:
    """volume.rs:10-41. Built by `Scene.add_volume`."""

    def __init__(self, obj, density, material):
        self.obj, self.density, self.material = obj, f32(density), int(material)

    def to_dict(self):
        return {"object_type": "ConstantMedium", "obj": self.obj.to_dict(), "density": self.density,
                "material": self.material}


# ---------------------------------------------------------------------------------------------------
# scene.rs
# ---------------------------------------------------------------------------------------------------
class RenderObject:
    def __init__(self, obj):
        self.obj = obj
        self._position = Vec3.zero()
        self._rotation = Rotor3.identity()
        self._flip_normals = False

    @staticmethod
    def new(obj):
        return RenderObject(obj)

    def position(self, x, y, z):
        self._position = Vec3(x, y, z)
        return self

    def position_vec(self, pos):
        self._position = _v3(pos)
        return self

    def rotate(self, rotor: Rotor3):
        self._rotation = rotor
        return self

    def flip_normals(self):
        self._flip_normals = not self._flip_normals
        return self

    def to_dict(self):
        return {"obj": self.obj.to_dict(), "position": self._position.to_dict(),
                "rotation": self._rotation.to_dict(), "flip_normals": self._flip_normals}


class Scene:
    def __init__(self):
        self.render_objects: List[RenderObject] = []
        self.materials: list = []
        self.environment = ColorEnv()  # scene.rs:36 — black
        # host-side asset registry: path -> decoded array (RGBA8 HxWx4 for images, fp32 HxWx3 for HDR)
        self.assets: dict = {}
        self.asset_dir: Optional[str] = None  # where relative ImageTexture / HdrEnvironment paths resolve
        self._yaml_text: Optional[str] = None  # set when loaded from YAML text

    @staticmethod
    def new():
        return Scene()

    def add_object(self, obj: RenderObject) -> int:
        self.render_objects.append(obj)
        return len(self.render_objects) - 1

    def add_volume(self, obj: RenderObject, density, texture) -> int:
        mat = self.add_material(IsotropicMat(texture))
        obj.obj = ConstantMedium(obj.obj, density, mat)
        return self.add_object(obj)

    def get_object(self, idx):
        return self.render_objects[idx]

    def add_material(self, mat) -> int:
        self.materials.append(mat)
        return len(self.materials) - 1

    def get_material(self, idx):
        return self.materials[idx]

    def set_environment(self, env):
        self.environment = env

    def register_asset(self, path, array):
        """Give the decoded texels for an ImageTexture / HdrEnvironment path."""
        self.assets[str(path)] = array

    def to_dict(self):
        return {"render_objects": [o.to_dict() for o in self.render_objects],
                "materials": [m.to_dict() for m in self.materials],
                "environment": self.environment.to_dict()}

    def to_yaml(self) -> str:
        """`serde_yaml::to_string(&scene)`; a scene loaded from text is forwarded verbatim."""
        if self._yaml_text is not None:
            return self._yaml_text
        from .serde_yaml import dumps
        return dumps(self.to_dict())

    @staticmethod
    def from_yaml(text: str, asset_dir: Optional[str] = None) -> "Scene":
        """`serde_yaml::from_str` for callers that only forward the document to the native loader."""
        s = Scene()
        s._yaml_text = text
        s.asset_dir = asset_dir
        return s

    @staticmethod
    def from_file(path: str) -> "Scene":
        import gzip
        opener = gzip.open if str(path).endswith(".gz") else open
        with opener(path, "rt") as f:
            return Scene.from_yaml(f.read(), asset_dir=os.path.dirname(os.path.abspath(path)))


# ---------------------------------------------------------------------------------------------------
# camera.rs:18-71, render.rs:57-107
# ---------------------------------------------------------------------------------------------------
class CameraSettings:
    def __init__(self):
        self._cam_pos = Vec3(0.0, 0.0, -10.0)
        self._look_at = Vec3.zero()
        self._vfov = 30.0
        self._aperture = 0.0
        self._focus_dist = 10.0

    @staticmethod
    def default():
        return CameraSettings()

    def cam_pos(self, v):
        self._cam_pos = _v3(v)
        return self

    def look_at(self, v):
        self._look_at = _v3(v)
        return self

    def field_of_view(self, vfov):
        self._vfov = f32(vfov)
        return self

    def aperture(self, a):
        self._aperture = f32(a)
        return self

    def focus_dist(self, d):
        self._focus_dist = f32(d)
        return self


class Renderer:
    """render.rs:57-107; defaults per render.rs:198-218 (1920x1080, 128 spp, use_bvh=false, gamma 2.2).

    Extra (not in the reference): `seed` keys the counter-based RNG, `device` picks the GPU, `gpus` spreads the samples over
    several GPUs, `adaptive` renders each pixel until its noise estimate meets a target, `denoise` filters the render with
    first-hit feature buffers as guides.
    """

    def __init__(self):
        self._width, self._height, self._samples = 1920, 1080, 128
        self._multithreaded, self._use_bvh, self._gamma = True, False, 2.2
        self._camera = CameraSettings()
        self._seed = 0
        self._gpus, self._reduce = 1, "nccl"
        self._adaptive = None
        self._denoise = None
        self.last_stats = None

    @staticmethod
    def default():
        return Renderer()

    def gpus(self, n, reduce="nccl"):
        """Extra (not in the reference): render on `n` GPUs of this box in one call (fw_render_multi): the sample range is split
        into one slice per GPU, the fp32 sums are combined by one NCCL reduce ("nccl") or by the fused peer-memory
        reduce + resolve kernel ("peer")."""
        self._gpus, self._reduce = int(n), reduce
        return self

    def adaptive(self, threshold, min_samples=16, floor=None):
        """Extra (not in the reference): adaptive sampling (fw_render_adaptive).  `samples` becomes the cap per pixel; every
        pixel renders `min_samples` samples, then rounds of doubling sample counts go on for the pixels whose relative standard
        error of the mean luminance is still above `threshold` (e.g. 0.05 = 5 %).  A pixel that ends with k samples has
        exactly the value a uniform render at k samples gives it.  `floor` (default 0.01, linear luminance) bounds the
        error's denominator from below: under it the target becomes the absolute error threshold * floor, which for
        threshold 0.05 is under one u8 level after gamma 2.2, so near-black pixels stop early instead of chasing a relative
        error their displayed value can not show.  `threshold=None` switches adaptive sampling off.  Single GPU only:
        together with gpus(n > 1) `render` raises ValueError.  last_stats then carries `counts` (per-pixel samples), `error`
        (per-pixel final relative error), `rounds` and `active` (pixels rendered in each round)."""
        if threshold is None:
            self._adaptive = None
        else:
            from .engine import ADAPTIVE_FLOOR
            self._adaptive = (float(threshold), int(min_samples), ADAPTIVE_FLOOR if floor is None else float(floor))
        return self

    def denoise(self, iterations=5, aov_samples=4, sigma_luminance=4.0, sigma_depth=0.1, sigma_albedo=0.1):
        """Extra (not in the reference): a denoised render (fw_render_denoised, DESIGN.md §12).  The image is rendered at
        `samples` spp (>= 2) as usual, the first-hit albedo, normal and depth of every pixel are averaged over its first
        `aov_samples` samples, and an edge-aware a-trous filter of `iterations` passes (step 1, 2, 4, ...) averages each pixel
        with neighbours whose luminance (in standard deviations of the noise estimate, `sigma_luminance`), relative depth
        (`sigma_depth`) and albedo (`sigma_albedo`) are close, and whose normals agree.  `iterations=None` switches it off.  Single
        GPU and not together with adaptive(): `render` raises ValueError for those combinations.  last_stats then carries
        `denoised` (linear fp32), `variance` (of the mean luminance before filtering) and `aov` (albedo, normal, depth,
        object)."""
        if iterations is None:
            self._denoise = None
        else:
            self._denoise = {"iterations": int(iterations), "aov_samples": int(aov_samples), "sigma_luminance": float(sigma_luminance),
                             "sigma_depth": float(sigma_depth), "sigma_albedo": float(sigma_albedo)}
        return self

    def width(self, w):
        self._width = int(w)
        return self

    def height(self, h):
        self._height = int(h)
        return self

    def samples(self, s):
        self._samples = int(s)
        return self

    def multithreaded(self, m):
        self._multithreaded = bool(m)  # accepted for API compatibility; the GPU path ignores it
        return self

    def use_bvh(self, b):
        self._use_bvh = bool(b)
        return self

    def gamma(self, g):
        self._gamma = f32(g)
        return self

    def camera(self, settings: CameraSettings):
        self._camera = settings
        return self

    def seed(self, s):
        self._seed = int(s)
        return self

    def params(self, sample_begin=0, sample_count=None):
        from ._native import FwParams
        c = self._camera
        p = FwParams()
        p.width, p.height, p.samples = self._width, self._height, self._samples
        p.sample_begin = sample_begin
        p.sample_count = self._samples if sample_count is None else sample_count
        p.use_bvh = 1 if self._use_bvh else 0
        p.gamma = self._gamma
        p.cam_pos[:] = list(c._cam_pos)
        p.look_at[:] = list(c._look_at)
        p.vfov, p.aperture, p.focus_dist = c._vfov, c._aperture, c._focus_dist
        p.seed = self._seed
        return p

    def render(self, scene: Scene) -> np.ndarray:
        """GPU drop-in for `Renderer::render` — returns (height, width, 3) u8, row 0 = top."""
        from .engine import NativeScene, render_scene
        if self._denoise is not None:
            if self._gpus > 1:
                raise ValueError("a denoised render runs on one GPU: gpus(n > 1) and denoise() can not be combined")
            if self._adaptive is not None:
                raise ValueError("adaptive() and denoise() can not be combined")
            ns = NativeScene.from_scene(scene, 0)
            try:
                rgb, _sum, den, var, aov, stats = ns.render_denoised(self.params(), want_sum=False, **self._denoise)
            finally:
                ns.close()
            stats["denoised"], stats["variance"], stats["aov"] = den, var, aov
            self.last_stats = stats
            return rgb
        if self._adaptive is not None:
            if self._gpus > 1:
                raise ValueError("adaptive sampling renders on one GPU: gpus(n > 1) and adaptive() can not be combined")
            threshold, min_samples, floor = self._adaptive
            ns = NativeScene.from_scene(scene, 0)
            try:
                rgb, _sum, counts, err, stats = ns.render_adaptive(self.params(), threshold, min_samples, floor, want_sum=False)
            finally:
                ns.close()
            stats["counts"], stats["error"] = counts, err
            self.last_stats = stats
            return rgb
        if self._gpus > 1:
            ns = NativeScene.from_scene(scene, 0)
            try:
                rgb, _sum, stats = ns.render_multi(self.params(), self._gpus, reduce=self._reduce, want_sum=False)
            finally:
                ns.close()
        else:
            rgb, _sum, stats = render_scene(scene, self)
        self.last_stats = stats
        return rgb
