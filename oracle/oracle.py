"""ctypes harness for the CPU oracle (oracle/firework_oracle.cpp).  TEST INFRASTRUCTURE ONLY.

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs may import this.
It takes a firework serde-YAML scene document parsed by PyYAML (an independent parser from the product's
C++ one) and replays it into the oracle through its builder C ABI.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess
from typing import Callable, Optional

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))

MAT_KIND = {"LambertianMat": 0, "MetalMat": 1, "DielectricMat": 2, "EmissiveMat": 3, "IsotropicMat": 4}
PLANE = {"XY": 0, "XZ": 1, "YZ": 2, "XYRect": 0, "XZRect": 1, "YZRect": 2}


class OrcParams(C.Structure):
    _fields_ = [("width", C.c_uint32), ("height", C.c_uint32), ("samples", C.c_uint32),
                ("sample_begin", C.c_uint32), ("sample_count", C.c_uint32), ("use_bvh", C.c_uint32),
                ("gamma", C.c_float), ("cam_pos", C.c_float * 3), ("look_at", C.c_float * 3),
                ("vfov", C.c_float), ("aperture", C.c_float), ("focus_dist", C.c_float), ("seed", C.c_uint64)]


class OrcStats(C.Structure):
    _fields_ = [("samples", C.c_uint64), ("rays", C.c_uint64), ("aabb_tests", C.c_uint64),
                ("prim_tests", C.c_uint64), ("seconds", C.c_double), ("threads", C.c_int), ("pad", C.c_int),
                ("sphere", C.c_uint64), ("rect", C.c_uint64), ("tri", C.c_uint64), ("conic", C.c_uint64),
                ("xform_rot", C.c_uint64), ("xform_trans", C.c_uint64)]


def build(force: bool = False) -> None:
    """Compile liboracle.so / liboracle_fast.so if missing (make)."""
    if force or not (os.path.exists(os.path.join(_HERE, "liboracle.so"))
                     and os.path.exists(os.path.join(_HERE, "liboracle_fast.so"))):
        subprocess.run(["make", "-C", _HERE], check=True, capture_output=True)


_libs = {}


def _lib(fast: bool):
    name = "liboracle_fast.so" if fast else "liboracle.so"
    if name not in _libs:
        build()
        lib = C.CDLL(os.path.join(_HERE, name))
        lib.orc_scene_new.restype = C.c_void_p
        for fn in ("orc_tex_constant", "orc_tex_checker", "orc_tex_perlin", "orc_tex_turbulence", "orc_tex_marble",
                   "orc_tex_image", "orc_material", "orc_shape_sphere", "orc_shape_rect", "orc_shape_rect3d",
                   "orc_shape_disk", "orc_shape_cylinder", "orc_shape_cone", "orc_shape_mesh", "orc_shape_medium",
                   "orc_add_object", "orc_scene_finish", "orc_num_objects", "orc_bvh_leaf_order", "orc_bvh_nodes",
                   "orc_mesh_leaf_order", "orc_render"):
            getattr(lib, fn).restype = C.c_int
        lib.orc_perlin_noise.restype = C.c_float
        lib.orc_perlin_noise.argtypes = [C.c_float] * 3
        _libs[name] = lib
    return _libs[name]


def _fp(a):
    return a.ctypes.data_as(C.POINTER(C.c_float))


def _f3(v):
    return (C.c_float * 3)(float(v["x"]), float(v["y"]), float(v["z"]))


def params_from(p) -> OrcParams:
    """Accepts a firework_b200 FwParams (same field names) or an OrcParams."""
    if isinstance(p, OrcParams):
        return p
    o = OrcParams()
    for name, _ in OrcParams._fields_:
        v = getattr(p, name)
        if name in ("cam_pos", "look_at"):
            getattr(o, name)[:] = list(v)
        else:
            setattr(o, name, v)
    return o


class OracleScene:
    def __init__(self, doc: dict, use_bvh: bool, asset_loader: Optional[Callable[[str, str], np.ndarray]] = None,
                 fast: bool = False):
        self.lib = _lib(fast)
        self.h = C.c_void_p(self.lib.orc_scene_new())
        self.use_bvh = bool(use_bvh)
        self._asset_loader = asset_loader
        self.tex_of_material = []
        L, h = self.lib, self.h
        for m in doc["materials"]:
            kind = MAT_KIND[m["material"]]
            tex, albedo, param = -1, (C.c_float * 3)(0, 0, 0), 0.0
            if kind in (0, 3):
                tex = self._texture(m["albedo"])
            elif kind == 4:
                tex = self._texture(m["texture"])
            elif kind == 1:
                albedo, param = _f3(m["albedo"]), float(m["roughness"])
            else:
                param = float(m["ref_idx"])
            self.tex_of_material.append(tex)
            r = L.orc_material(h, kind, tex, albedo, C.c_float(param))
            assert r >= 0
        for ro in doc["render_objects"]:
            sid = self._shape(ro["obj"])
            rot = ro["rotation"]
            rotor = (C.c_float * 4)(float(rot["s"]), float(rot["bv"]["xy"]), float(rot["bv"]["xz"]), float(rot["bv"]["yz"]))
            r = L.orc_add_object(h, sid, _f3(ro["position"]), rotor, 1 if ro["flip_normals"] else 0)
            assert r >= 0
        env = doc["environment"]
        tag = env["environment"]
        if tag == "ColorEnv":
            c = env["color"]
            L.orc_env_color(h, C.c_float(c["x"]), C.c_float(c["y"]), C.c_float(c["z"]))
        elif tag == "SkyEnv":
            L.orc_env_sky(h, _f3(env["zenith_color"]), _f3(env["horizon_color"]))
        elif tag == "HdrEnvironment":
            img = np.ascontiguousarray(self._asset(env["value"], "hdr"), dtype=np.float32)
            L.orc_env_hdr(h, img.shape[1], img.shape[0], _fp(img))
        else:
            raise ValueError(f"unknown environment tag {tag}")
        if L.orc_scene_finish(h, 1 if use_bvh else 0) != 0:
            raise ValueError("No render objects added to scene!")

    def __del__(self):
        try:
            self.lib.orc_scene_free(self.h)
        except Exception:
            pass

    def _asset(self, path, kind):
        if self._asset_loader is None:
            raise ValueError(f"scene needs asset {path!r} but no asset_loader was given")
        return self._asset_loader(path, kind)

    def _texture(self, t) -> int:
        L, h = self.lib, self.h
        tag = t["texture"]
        if tag == "ConstantTexture":
            c = t["color"]
            return L.orc_tex_constant(h, C.c_float(c["x"]), C.c_float(c["y"]), C.c_float(c["z"]))
        if tag == "CheckerTexture":
            odd, even = self._texture(t["odd"]), self._texture(t["even"])
            return L.orc_tex_checker(h, odd, even, C.c_float(t["scale"]))
        if tag == "PerlinNoiseTexture":
            return L.orc_tex_perlin(h, C.c_float(t["scale"]))
        if tag == "TurbulenceTexture":
            return L.orc_tex_turbulence(h, C.c_uint64(t["depth"]), C.c_float(t["scale"]))
        if tag == "MarbleTexture":
            return L.orc_tex_marble(h, C.c_uint64(t["depth"]), C.c_float(t["scale"]))
        if tag == "ImageTexture":
            img = np.ascontiguousarray(self._asset(t["value"], "image"), dtype=np.uint8)
            assert img.ndim == 3 and img.shape[2] == 4
            return L.orc_tex_image(h, img.shape[1], img.shape[0], img.ctypes.data_as(C.POINTER(C.c_uint8)))
        raise ValueError(f"unknown texture tag {tag}")

    def _rect_fields(self, f):
        return ((C.c_float * 2)(f["min"]["x"], f["min"]["y"]), (C.c_float * 2)(f["max"]["x"], f["max"]["y"]),
                C.c_float(f["k"]), 1 if f["flip_normal"] else 0, int(f["material"]))

    def _shape(self, o) -> int:
        L, h = self.lib, self.h
        tag = o["object_type"]
        if tag == "Sphere":
            return L.orc_shape_sphere(h, C.c_float(o["radius"]), int(o["material"]))
        if tag in ("XYRect", "XZRect", "YZRect"):
            mn, mx, k, flip, mat = self._rect_fields(o)
            return L.orc_shape_rect(h, PLANE[tag], mn, mx, k, flip, mat)
        if tag == "Rect3d":
            faces = []
            for f in o["faces"]:
                (ptag, ff), = f.items()
                faces += [PLANE[ptag], ff["min"]["x"], ff["min"]["y"], ff["max"]["x"], ff["max"]["y"], ff["k"],
                          1.0 if ff["flip_normal"] else 0.0, float(ff["material"])]
            fa = np.asarray(faces, dtype=np.float32)
            return L.orc_shape_rect3d(h, _f3(o["pos"]), _f3(o["size"]), len(o["faces"]), _fp(fa))
        if tag == "Disk":
            return L.orc_shape_disk(h, C.c_float(o["radius"]), C.c_float(o["phi_max"]), C.c_float(o["inner_radius"]),
                                    int(o["material"]))
        if tag == "Cylinder":
            return L.orc_shape_cylinder(h, C.c_float(o["radius"]), C.c_float(o["height"]), C.c_float(o["max_phi"]),
                                        int(o["material"]))
        if tag == "Cone":
            return L.orc_shape_cone(h, C.c_float(o["radius"]), C.c_float(o["height"]), int(o["material"]))
        if tag == "TriangleMesh":
            verts = np.array([[v["x"], v["y"], v["z"]] for v in o["verts"]], dtype=np.float32)
            idx = np.array(o["indicies"], dtype=np.uint32)
            normals = uvs = None
            if o.get("normals") is not None:
                normals = np.array([[v["x"], v["y"], v["z"]] for v in o["normals"]], dtype=np.float32)
            if o.get("uvs") is not None:
                uvs = np.array([[v["x"], v["y"]] for v in o["uvs"]], dtype=np.float32)
            return L.orc_shape_mesh(h, len(verts), _fp(verts), len(idx), idx.ctypes.data_as(C.POINTER(C.c_uint32)),
                                    _fp(normals) if normals is not None else None,
                                    _fp(uvs) if uvs is not None else None, int(o["material"]))
        if tag == "ConstantMedium":
            inner = self._shape(o["obj"])
            r = L.orc_shape_medium(h, inner, C.c_float(o["density"]), int(o["material"]))
            assert r >= 0
            return r
        raise ValueError(f"unknown object_type {tag}")

    # ---------------------------------------------------------------------------------------------
    def num_objects(self):
        return self.lib.orc_num_objects(self.h)

    def object_aabbs(self):
        n = self.num_objects()
        out = np.zeros((n, 6), np.float32)
        buf = (C.c_float * 6)()
        for i in range(n):
            self.lib.orc_object_aabb(self.h, i, buf)
            out[i] = list(buf)
        return out

    def object_rotation(self, i):
        buf = (C.c_float * 9)()
        self.lib.orc_object_rotation(self.h, i, buf)
        return np.array(list(buf), np.float32).reshape(3, 3)  # rows = columns of the Mat3

    def bvh_leaf_order(self):
        n = self.num_objects()
        out = (C.c_int * n)()
        nn, md = C.c_int(), C.c_int()
        c = self.lib.orc_bvh_leaf_order(self.h, out, n, C.byref(nn), C.byref(md))
        assert c == n
        return np.array(list(out), np.int32), nn.value, md.value

    def bvh_nodes(self):
        n = self.lib.orc_bvh_nodes(self.h, None, 0)
        out = np.zeros((n, 7), np.float32)
        self.lib.orc_bvh_nodes(self.h, _fp(out), n)
        return out

    def mesh_leaf_order(self, obj, ntris):
        out = (C.c_int * ntris)()
        nn, md = C.c_int(), C.c_int()
        c = self.lib.orc_mesh_leaf_order(self.h, obj, out, ntris, C.byref(nn), C.byref(md))
        assert c == ntris, (c, ntris)
        return np.array(list(out), np.int32), nn.value, md.value

    def camera(self, params):
        out = (C.c_float * 24)()
        self.lib.orc_camera(C.byref(params_from(params)), out)
        return np.array(list(out), np.float32)

    def primary_rays(self, params, sample, pix_begin=0, n=None):
        p = params_from(params)
        if n is None:
            n = p.width * p.height - pix_begin
        o = np.zeros((n, 3), np.float32)
        d = np.zeros((n, 3), np.float32)
        self.lib.orc_primary_rays(C.byref(p), C.c_uint32(sample), C.c_uint32(pix_begin), C.c_uint32(n), _fp(o), _fp(d))
        return o, d

    def first_hit(self, origins, dirs, seed=0, pixel=None, sample=None, bounce=None):
        o = np.ascontiguousarray(origins, np.float32)
        d = np.ascontiguousarray(dirs, np.float32)
        n = len(o)
        u32p = C.POINTER(C.c_uint32)
        keys = []
        for k in (pixel, sample, bounce):
            keys.append(None if k is None else np.ascontiguousarray(k, np.uint32))
        res = {"obj": np.zeros(n, np.int32), "prim": np.zeros(n, np.int32), "material": np.zeros(n, np.int32),
               "t": np.zeros(n, np.float32), "point": np.zeros((n, 3), np.float32),
               "normal": np.zeros((n, 3), np.float32), "uv": np.zeros((n, 2), np.float32)}
        st = OrcStats()
        i32p = C.POINTER(C.c_int32)
        self.lib.orc_first_hit(self.h, 1 if self.use_bvh else 0, C.c_uint64(seed), C.c_uint32(n), _fp(o), _fp(d),
                               *[None if k is None else k.ctypes.data_as(u32p) for k in keys],
                               res["obj"].ctypes.data_as(i32p), res["prim"].ctypes.data_as(i32p),
                               res["material"].ctypes.data_as(i32p), _fp(res["t"]), _fp(res["point"]),
                               _fp(res["normal"]), _fp(res["uv"]), C.byref(st))
        res["aabb_tests"], res["prim_tests"] = st.aabb_tests, st.prim_tests
        return res

    def scatter_step(self, material, ray_o, ray_d, hit_t, hit_point, hit_normal, hit_uv, uniforms):
        n = len(material)
        material = np.ascontiguousarray(material, np.int32)
        arrs = [np.ascontiguousarray(a, np.float32) for a in (ray_o, ray_d, hit_t, hit_point, hit_normal, hit_uv)]
        uniforms = np.ascontiguousarray(uniforms, np.float32)
        nu = uniforms.shape[1]
        res = {"emit": np.zeros((n, 3), np.float32), "scattered": np.zeros(n, np.int32),
               "atten": np.zeros((n, 3), np.float32), "o": np.zeros((n, 3), np.float32),
               "d": np.zeros((n, 3), np.float32), "consumed": np.zeros(n, np.int32)}
        i32p = C.POINTER(C.c_int32)
        self.lib.orc_scatter_step(self.h, C.c_uint32(n), material.ctypes.data_as(i32p), *[_fp(a) for a in arrs],
                                  _fp(uniforms), C.c_uint32(nu), _fp(res["emit"]),
                                  res["scattered"].ctypes.data_as(i32p), _fp(res["atten"]), _fp(res["o"]),
                                  _fp(res["d"]), res["consumed"].ctypes.data_as(i32p))
        return res

    def scatter_step_keyed(self, material, ray_o, ray_d, hit_t, hit_point, hit_normal, hit_uv, seed, pixel, sample, bounce):
        n = len(material)
        material = np.ascontiguousarray(material, np.int32)
        arrs = [np.ascontiguousarray(a, np.float32) for a in (ray_o, ray_d, hit_t, hit_point, hit_normal, hit_uv)]
        keys = [np.ascontiguousarray(np.broadcast_to(k, (n,)), np.uint32) for k in (pixel, sample, bounce)]
        res = {"emit": np.zeros((n, 3), np.float32), "scattered": np.zeros(n, np.int32),
               "atten": np.zeros((n, 3), np.float32), "o": np.zeros((n, 3), np.float32),
               "d": np.zeros((n, 3), np.float32), "consumed": np.zeros(n, np.int32)}
        i32p, u32p = C.POINTER(C.c_int32), C.POINTER(C.c_uint32)
        self.lib.orc_scatter_step_keyed(self.h, C.c_uint64(seed), C.c_uint32(n), material.ctypes.data_as(i32p),
                                        *[_fp(a) for a in arrs], *[k.ctypes.data_as(u32p) for k in keys],
                                        _fp(res["emit"]), res["scattered"].ctypes.data_as(i32p), _fp(res["atten"]),
                                        _fp(res["o"]), _fp(res["d"]), res["consumed"].ctypes.data_as(i32p))
        return res

    def env_sample(self, dirs):
        d = np.ascontiguousarray(dirs, np.float32)
        out = np.zeros_like(d)
        self.lib.orc_env_sample(self.h, C.c_uint32(len(d)), _fp(d), _fp(out))
        return out

    def texture_sample(self, tex, uv, point):
        uv = np.ascontiguousarray(uv, np.float32)
        pt = np.ascontiguousarray(point, np.float32)
        out = np.zeros_like(pt)
        self.lib.orc_texture_sample(self.h, int(tex), C.c_uint32(len(pt)), _fp(uv), _fp(pt), _fp(out))
        return out

    def render(self, params, pix_begin=0, pix_count=0, want_rgb=True, threads=0):
        """Returns (rgb u8 (H,W,3) or None, sum fp32 (H,W,3), stats dict)."""
        p = params_from(params)
        npix = p.width * p.height
        s = np.zeros((npix, 3), np.float32)
        rgb = np.zeros((npix, 3), np.uint8) if want_rgb else None
        st = OrcStats()
        r = self.lib.orc_render(self.h, C.byref(p), C.c_uint32(pix_begin), C.c_uint32(pix_count), _fp(s),
                                rgb.ctypes.data_as(C.POINTER(C.c_uint8)) if want_rgb else None, C.byref(st),
                                C.c_int(threads))
        if r != 0:
            raise RuntimeError(f"orc_render failed: {r}")
        stats = {k: getattr(st, k) for k, _ in OrcStats._fields_}
        return (rgb.reshape(p.height, p.width, 3) if want_rgb else None), s.reshape(p.height, p.width, 3), stats


def resolve(sum_buf, samples, gamma, fast=False):
    s = np.ascontiguousarray(sum_buf, np.float32).reshape(-1, 3)
    rgb = np.zeros((len(s), 3), np.uint8)
    _lib(fast).orc_resolve(_fp(s), C.c_uint32(len(s)), C.c_uint32(samples), C.c_float(gamma),
                           rgb.ctypes.data_as(C.POINTER(C.c_uint8)))
    return rgb.reshape(np.asarray(sum_buf).shape)


def philox(ctr, key):
    c = (C.c_uint32 * 4)(*ctr)
    k = (C.c_uint32 * 2)(*key)
    o = (C.c_uint32 * 4)()
    _lib(False).orc_philox(c, k, o)
    return list(o)


def perlin_noise(x, y, z, fast=False):
    return float(_lib(fast).orc_perlin_noise(x, y, z))
