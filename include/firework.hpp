// firework.hpp — C++17 mirror of the reference's public Rust API for the rendering path, on top of the C ABI
// (include/firework_b200.h).  Same names, same builder style, same argument meaning as the crate:
//
//   ultraviolet::{Vec3, Rotor3}                       Vec3, Rotor3                       (ultraviolet 0.5.1)
//   firework::scene::{Scene, RenderObject}            Scene, RenderObject                src/scene.rs:19-110
//   firework::objects::{Sphere, XYRect, XZRect, YZRect, Rect3d, TriangleMesh, Disk, Cylinder, Cone}   src/objects/*.rs
//   firework::material::{LambertianMat, MetalMat, DielectricMat, EmissiveMat, IsotropicMat}            src/material.rs
//   firework::texture::{ConstantTexture, CheckerTexture, PerlinNoiseTexture, TurbulenceTexture, MarbleTexture, ImageTexture}
//   firework::environment::{ColorEnv, SkyEnv}, HdrEnvironment (examples/hdri_test.rs)
//   firework::camera::CameraSettings, firework::render::Renderer, firework::util::Color               src/render.rs:49-121
//
// `Renderer::render(scene)` is the drop-in for src/render.rs:109: the scene crosses the boundary as its serde YAML document
// (`Scene::to_yaml` == `serde_yaml::to_string(&scene)`, DESIGN.md §1), image / HDR assets are decoded by the library, and the
// result is the reference's `Vec<Color>` (row 0 = top).  Errors are exceptions (`firework::Error`) where the crate panics.
// Header-only; link libfirework_b200.a (or .so) as INTEGRATION.md shows.  examples/*.cpp are the crate's examples restated.
#pragma once
#include <charconv>
#include <cmath>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <memory>
#include <stdexcept>
#include <string>
#include <utility>
#include <vector>

#include "firework_b200.h"

namespace firework {

struct Error : std::runtime_error {
    using std::runtime_error::runtime_error;
};

// ---- ultraviolet -----------------------------------------------------------------------------------------------------
struct Vec3 {
    float x = 0.0f, y = 0.0f, z = 0.0f;
    constexpr Vec3() = default;
    constexpr Vec3(float x_, float y_, float z_) : x(x_), y(y_), z(z_) {}
    static constexpr Vec3 zero() { return Vec3(0.0f, 0.0f, 0.0f); }
    static constexpr Vec3 one() { return Vec3(1.0f, 1.0f, 1.0f); }
    static constexpr Vec3 broadcast(float v) { return Vec3(v, v, v); }
    static constexpr Vec3 unit_y() { return Vec3(0.0f, 1.0f, 0.0f); }
    Vec3 operator+(Vec3 o) const { return Vec3(x + o.x, y + o.y, z + o.z); }
    Vec3 operator-(Vec3 o) const { return Vec3(x - o.x, y - o.y, z - o.z); }
    Vec3 operator*(float s) const { return Vec3(x * s, y * s, z * s); }
    float mag() const { return std::sqrt(x * x + y * y + z * z); }
};
inline float to_radians(float deg) { return deg * (3.14159265358979323846f / 180.0f); }   // f32::to_radians

// Rotor3 {s, bv {xy, xz, yz}} (serde layout: src/serde_compat.rs:6-20)
struct Rotor3 {
    float s = 1.0f, xy = 0.0f, xz = 0.0f, yz = 0.0f;
    static Rotor3 identity() { return Rotor3(); }
    // ultraviolet 0.5.1 Rotor3::from_angle_plane: (sin, cos) = (angle * 0.5).sin_cos(); Rotor3::new(cos, plane * -sin).
    // sin / cos are evaluated in double and rounded once (libm's sinf / cosf are correctly rounded); `plane * -sin` keeps the
    // sign of its zero components, as scenes/teapot.yml shows.
    static Rotor3 from_angle_plane(float angle, float pxy, float pxz, float pyz) {
        const float half = angle * 0.5f;
        const float sn = (float)std::sin((double)half), cs = (float)std::cos((double)half);
        Rotor3 r;
        r.s = cs; r.xy = pxy * -sn; r.xz = pxz * -sn; r.yz = pyz * -sn;
        return r;
    }
    static Rotor3 from_rotation_xy(float angle) { return from_angle_plane(angle, 1.0f, 0.0f, 0.0f); }
    static Rotor3 from_rotation_xz(float angle) { return from_angle_plane(angle, 0.0f, 1.0f, 0.0f); }
    static Rotor3 from_rotation_yz(float angle) { return from_angle_plane(angle, 0.0f, 0.0f, 1.0f); }
};

struct Color {   // util.rs:8-12
    uint8_t r = 0, g = 0, b = 0;
};

// ---- the serde document ------------------------------------------------------------------------------------------------
namespace detail {
struct Y {   // a YAML value: what `#[derive(Serialize)]` would hand to serde_yaml
    enum Kind { NUL, BOOL, INT, F32, STR, MAP, SEQ } kind = NUL;
    bool b = false;
    long long i = 0;
    float f = 0.0f;
    std::string s;
    std::vector<std::pair<std::string, Y>> map;
    std::vector<Y> seq;
    static Y null() { return Y(); }
    static Y boolean(bool v) { Y y; y.kind = BOOL; y.b = v; return y; }
    static Y integer(long long v) { Y y; y.kind = INT; y.i = v; return y; }
    static Y f32(float v) { Y y; y.kind = F32; y.f = v; return y; }
    static Y str(std::string v) { Y y; y.kind = STR; y.s = std::move(v); return y; }
    static Y mapping(std::vector<std::pair<std::string, Y>> m) { Y y; y.kind = MAP; y.map = std::move(m); return y; }
    static Y sequence(std::vector<Y> q) { Y y; y.kind = SEQ; y.seq = std::move(q); return y; }
    static Y vec3(Vec3 v) { return mapping({{"x", f32(v.x)}, {"y", f32(v.y)}, {"z", f32(v.z)}}); }
};
inline std::string fmt_f32(float v) {   // serde_yaml prints an f32 as the shortest f64 text of its value
    if (std::isnan(v)) return ".nan";
    if (std::isinf(v)) return v > 0 ? ".inf" : "-.inf";
    char buf[40];
    auto r = std::to_chars(buf, buf + sizeof buf, (double)v);
    std::string s(buf, r.ptr);
    const size_t e = s.find('e');
    if (e != std::string::npos) {   // exponent without padding, mantissa with a fraction: 9.34e-5, 1.0e+21
        std::string m = s.substr(0, e);
        const int ex = std::atoi(s.c_str() + e + 1);
        if (m.find('.') == std::string::npos) m += ".0";
        return m + "e" + (ex < 0 ? "-" : "+") + std::to_string(ex < 0 ? -ex : ex);
    }
    if (s.find('.') == std::string::npos) s += ".0";
    return s;
}
inline std::string fmt_str(const std::string& v) {
    bool plain = !v.empty() && v != "~" && v != "null" && v != "true" && v != "false" && v.find(": ") == std::string::npos &&
                 v.find(" #") == std::string::npos && v.back() != ':' && v.back() != ' ' &&
                 std::string("-?:,[]{}#&*!|>'\"%@` ").find(v[0]) == std::string::npos;
    if (plain) {
        char* end = nullptr;
        std::strtod(v.c_str(), &end);
        if (end && *end == 0) plain = false;   // would read back as a number
        for (char c : v)
            if ((unsigned char)c < 0x20) plain = false;
    }
    if (plain) return v;
    std::string q = "\"";
    for (char c : v) {
        if (c == '"' || c == '\\') { q += '\\'; q += c; }
        else if (c == '\n') q += "\\n";
        else if (c == '\t') q += "\\t";
        else q += c;
    }
    return q + "\"";
}
inline bool is_scalar(const Y& y) { return y.kind != Y::MAP && y.kind != Y::SEQ; }
inline std::string scalar_text(const Y& y) {
    switch (y.kind) {
        case Y::NUL: return "~";
        case Y::BOOL: return y.b ? "true" : "false";
        case Y::INT: return std::to_string(y.i);
        case Y::F32: return fmt_f32(y.f);
        default: return fmt_str(y.s);
    }
}
// Block style as serde_yaml 0.8 writes it: nested collections on the following lines, sequence items two columns in.
inline void emit(const Y& y, std::string& out, int indent, bool inline_first) {
    const std::string pad((size_t)indent, ' ');
    if (y.kind == Y::MAP) {
        bool first = true;
        for (const auto& kv : y.map) {
            if (!(first && inline_first)) out += pad;
            first = false;
            out += kv.first;
            out += ':';
            const Y& v = kv.second;
            if (is_scalar(v)) { out += ' '; out += scalar_text(v); out += '\n'; }
            else if (v.kind == Y::MAP && v.map.empty()) out += " {}\n";
            else if (v.kind == Y::SEQ && v.seq.empty()) out += " []\n";
            else { out += '\n'; emit(v, out, indent + 2, false); }
        }
    } else if (y.kind == Y::SEQ) {
        for (const Y& v : y.seq) {
            out += pad;
            out += "- ";
            if (is_scalar(v)) { out += scalar_text(v); out += '\n'; }
            else if (v.kind == Y::MAP && v.map.empty()) out += "{}\n";
            else if (v.kind == Y::SEQ && v.seq.empty()) out += "[]\n";
            else emit(v, out, indent + 2, true);
        }
    } else {
        out += pad + scalar_text(y) + "\n";
    }
}
struct Node {   // anything that serialises: textures, materials, shapes, environments
    virtual ~Node() = default;
    virtual Y to_yaml() const = 0;
};
inline void check(int rc, const char* what) {
    if (rc != FW_OK) throw Error(std::string(what) + ": " + fw_last_error());
}
}  // namespace detail

// ---- textures (src/texture.rs) ------------------------------------------------------------------------------------------
using Texture = std::shared_ptr<const detail::Node>;
namespace detail {
template <class F>
struct Lambda final : Node {
    F f;
    explicit Lambda(F fn) : f(std::move(fn)) {}
    Y to_yaml() const override { return f(); }
};
template <class F>
std::shared_ptr<const Node> node(F fn) { return std::make_shared<Lambda<F>>(std::move(fn)); }
}  // namespace detail

struct ConstantTexture {   // texture.rs:12-33
    static Texture new_(Vec3 color) {
        return detail::node([=] { return detail::Y::mapping({{"texture", detail::Y::str("ConstantTexture")}, {"color", detail::Y::vec3(color)}}); });
    }
    static Texture from_rgb(float r, float g, float b) { return new_(Vec3(r, g, b)); }
};
struct CheckerTexture {    // texture.rs:36-72
    static Texture new_(Texture odd, Texture even, float scale) {
        return detail::node([=] {
            return detail::Y::mapping({{"texture", detail::Y::str("CheckerTexture")}, {"odd", odd->to_yaml()}, {"even", even->to_yaml()}, {"scale", detail::Y::f32(scale)}});
        });
    }
    static Texture with_colors(Vec3 odd, Vec3 even, float scale) { return new_(ConstantTexture::new_(odd), ConstantTexture::new_(even), scale); }
};
struct PerlinNoiseTexture {   // texture.rs:75-167
    static Texture new_(float scale) {
        return detail::node([=] { return detail::Y::mapping({{"texture", detail::Y::str("PerlinNoiseTexture")}, {"scale", detail::Y::f32(scale)}}); });
    }
};
struct TurbulenceTexture {    // texture.rs:195-224
    static Texture new_(int depth, float scale) {
        return detail::node([=] {
            return detail::Y::mapping({{"texture", detail::Y::str("TurbulenceTexture")}, {"depth", detail::Y::integer(depth)}, {"scale", detail::Y::f32(scale)}});
        });
    }
};
struct MarbleTexture {        // texture.rs:227-248
    static Texture new_(int depth, float scale) {
        return detail::node([=] {
            return detail::Y::mapping({{"texture", detail::Y::str("MarbleTexture")}, {"depth", detail::Y::integer(depth)}, {"scale", detail::Y::f32(scale)}});
        });
    }
};
struct ImageTexture {         // texture.rs:251-309: serialises as its path; the library decodes the file at render time
    static Texture from_path(std::string path) {
        return detail::node([=] { return detail::Y::mapping({{"texture", detail::Y::str("ImageTexture")}, {"value", detail::Y::str(path)}}); });
    }
};

// ---- materials (src/material.rs) ----------------------------------------------------------------------------------------
using Material = std::shared_ptr<const detail::Node>;
struct LambertianMat {   // material.rs:26-74
    static Material new_(Texture albedo) {
        return detail::node([=] { return detail::Y::mapping({{"material", detail::Y::str("LambertianMat")}, {"albedo", albedo->to_yaml()}}); });
    }
    static Material with_color(Vec3 albedo) { return new_(ConstantTexture::new_(albedo)); }
};
struct MetalMat {        // material.rs:77-106
    static Material new_(Vec3 albedo, float roughness) {
        return detail::node([=] {
            return detail::Y::mapping({{"material", detail::Y::str("MetalMat")}, {"albedo", detail::Y::vec3(albedo)}, {"roughness", detail::Y::f32(roughness)}});
        });
    }
};
struct DielectricMat {   // material.rs:109-150
    static Material new_(float ref_idx) {
        return detail::node([=] { return detail::Y::mapping({{"material", detail::Y::str("DielectricMat")}, {"ref_idx", detail::Y::f32(ref_idx)}}); });
    }
};
struct EmissiveMat {     // material.rs:153-180
    static Material new_(Texture albedo) {
        return detail::node([=] { return detail::Y::mapping({{"material", detail::Y::str("EmissiveMat")}, {"albedo", albedo->to_yaml()}}); });
    }
    static Material with_color(Vec3 albedo) { return new_(ConstantTexture::new_(albedo)); }
};
struct IsotropicMat {    // material.rs:183-203
    static Material new_(Texture texture) {
        return detail::node([=] { return detail::Y::mapping({{"material", detail::Y::str("IsotropicMat")}, {"texture", texture->to_yaml()}}); });
    }
};

// ---- environments (src/environment.rs, examples/hdri_test.rs) -----------------------------------------------------------
using Environment = std::shared_ptr<const detail::Node>;
struct ColorEnv {
    static Environment new_(Vec3 color) {
        return detail::node([=] { return detail::Y::mapping({{"environment", detail::Y::str("ColorEnv")}, {"color", detail::Y::vec3(color)}}); });
    }
    static Environment default_() { return new_(Vec3::zero()); }   // scene.rs:36: black
};
struct SkyEnv {
    static Environment new_(Vec3 zenith_color, Vec3 horizon_color) {
        return detail::node([=] {
            return detail::Y::mapping({{"environment", detail::Y::str("SkyEnv")}, {"zenith_color", detail::Y::vec3(zenith_color)}, {"horizon_color", detail::Y::vec3(horizon_color)}});
        });
    }
    static Environment default_() { return new_(Vec3(0.5f, 0.7f, 1.0f), Vec3::one()); }   // environment.rs:34-41
};
struct HdrEnvironment {
    static Environment from_path(std::string path) {
        return detail::node([=] { return detail::Y::mapping({{"environment", detail::Y::str("HdrEnvironment")}, {"value", detail::Y::str(path)}}); });
    }
};

// ---- shapes (src/objects/*.rs) --------------------------------------------------------------------------------------------
using Shape = std::shared_ptr<const detail::Node>;
using MaterialIdx = size_t;   // material.rs: `MaterialIdx = usize`, what Scene::add_material returns

struct Sphere {   // sphere.rs:10-20
    static Shape new_(float radius, MaterialIdx material) {
        return detail::node([=] {
            return detail::Y::mapping({{"object_type", detail::Y::str("Sphere")}, {"radius", detail::Y::f32(radius)}, {"material", detail::Y::integer((long long)material)}});
        });
    }
};
namespace detail {
struct RectFields {
    float min_x, min_y, max_x, max_y, k;
    bool flip;
    MaterialIdx material;
    Y fields() const {
        return Y::mapping({{"min", Y::mapping({{"x", Y::f32(min_x)}, {"y", Y::f32(min_y)}})}, {"max", Y::mapping({{"x", Y::f32(max_x)}, {"y", Y::f32(max_y)}})},
                           {"k", Y::f32(k)}, {"flip_normal", Y::boolean(flip)}, {"material", Y::integer((long long)material)}});
    }
    Y tagged(const char* tag) const {
        Y y = fields();
        y.map.insert(y.map.begin(), {"object_type", Y::str(tag)});
        return y;
    }
};
}  // namespace detail
// rect.rs:18-46: AARect::new(a1_min, a1_max, a2_min, a2_max, k, material); `.flip_normal()` returns the flipped rectangle
template <int PLANE>
struct AARect {
    detail::RectFields r;
    static AARect new_(float a1_min, float a1_max, float a2_min, float a2_max, float k, MaterialIdx material) {
        return AARect{detail::RectFields{a1_min, a2_min, a1_max, a2_max, k, false, material}};
    }
    AARect flip_normal() const { AARect c = *this; c.r.flip = true; return c; }
    static const char* tag() { return PLANE == 0 ? "XYRect" : PLANE == 1 ? "XZRect" : "YZRect"; }
    static const char* variant() { return PLANE == 0 ? "XY" : PLANE == 1 ? "XZ" : "YZ"; }
    operator Shape() const {
        detail::RectFields f = r;
        return detail::node([=] { return f.tagged(tag()); });
    }
};
using XYRect = AARect<0>;
using XZRect = AARect<1>;
using YZRect = AARect<2>;

struct Rect3d {   // rect3d.rs:18-87: six faces in the order +z, -z, +y, -y, +x, -x, all arithmetic in f32
    static Shape new_(Vec3 p, Vec3 s, MaterialIdx m) {
        return detail::node([=] {
            using detail::Y;
            auto face = [](const char* variant, detail::RectFields f) { return Y::mapping({{variant, f.fields()}}); };
            std::vector<Y> faces = {
                face("XY", {p.x, p.y, p.x + s.x, p.y + s.y, p.z + s.z, false, m}), face("XY", {p.x, p.y, p.x + s.x, p.y + s.y, p.z, true, m}),
                face("XZ", {p.x, p.z, p.x + s.x, p.z + s.z, p.y + s.y, false, m}), face("XZ", {p.x, p.z, p.x + s.x, p.z + s.z, p.y, true, m}),
                face("YZ", {p.y, p.z, p.y + s.y, p.z + s.z, p.x + s.x, false, m}), face("YZ", {p.y, p.z, p.y + s.y, p.z + s.z, p.x, true, m}),
            };
            return Y::mapping({{"object_type", Y::str("Rect3d")}, {"pos", Y::vec3(p)}, {"size", Y::vec3(s)}, {"faces", Y::sequence(std::move(faces))}});
        });
    }
    static Shape with_size(Vec3 size, MaterialIdx material) { return new_(Vec3::zero(), size, material); }
};
struct TriangleMesh {   // mesh.rs:12-72
    static Shape new_(std::vector<Vec3> verts, std::vector<uint32_t> indicies, std::vector<Vec3> normals, std::vector<std::pair<float, float>> uvs,
                      MaterialIdx material) {
        if (!normals.empty() && normals.size() != verts.size()) throw Error("TriangleMesh::new() -- normals.len() must equal verts.len()");
        if (!uvs.empty() && uvs.size() != verts.size()) throw Error("TriangleMesh::new() -- uvs.len() must equal verts.len()");
        return detail::node([=] {
            using detail::Y;
            std::vector<Y> idx, vs, ns, us;
            for (uint32_t i : indicies) idx.push_back(Y::integer(i));
            for (Vec3 v : verts) vs.push_back(Y::vec3(v));
            for (Vec3 v : normals) ns.push_back(Y::vec3(v));
            for (auto uv : uvs) us.push_back(Y::mapping({{"x", Y::f32(uv.first)}, {"y", Y::f32(uv.second)}}));
            return Y::mapping({{"object_type", Y::str("TriangleMesh")}, {"indicies", Y::sequence(std::move(idx))}, {"verts", Y::sequence(std::move(vs))},
                               {"normals", normals.empty() ? Y::null() : Y::sequence(std::move(ns))}, {"uvs", uvs.empty() ? Y::null() : Y::sequence(std::move(us))},
                               {"material", Y::integer((long long)material)}});
        });
    }
};
struct Disk {       // disk.rs:10-38
    static Shape partial(float radius, float phi_deg, float inner_radius, MaterialIdx material) { return make(radius, to_radians(phi_deg), inner_radius, material); }
    static Shape new_(float radius, MaterialIdx material) { return make(radius, 2.0f * 3.14159265358979323846f, 0.0f, material); }
private:
    static Shape make(float radius, float phi_max, float inner_radius, MaterialIdx material) {
        return detail::node([=] {
            using detail::Y;
            return Y::mapping({{"object_type", Y::str("Disk")}, {"radius", Y::f32(radius)}, {"phi_max", Y::f32(phi_max)}, {"inner_radius", Y::f32(inner_radius)},
                               {"material", Y::integer((long long)material)}});
        });
    }
};
struct Cylinder {   // cylinder.rs:10-39
    static Shape partial(float radius, float height, float phi_deg, MaterialIdx material) {
        const float max_phi = to_radians(phi_deg);
        return detail::node([=] {
            using detail::Y;
            return Y::mapping({{"object_type", Y::str("Cylinder")}, {"radius", Y::f32(radius)}, {"height", Y::f32(height)}, {"max_phi", Y::f32(max_phi)},
                               {"material", Y::integer((long long)material)}});
        });
    }
    static Shape new_(float radius, float height, MaterialIdx material) { return partial(radius, height, 360.0f, material); }
};
struct Cone {       // cone.rs:10-25
    static Shape new_(float radius, float height, MaterialIdx material) {
        return detail::node([=] {
            using detail::Y;
            return Y::mapping({{"object_type", Y::str("Cone")}, {"radius", Y::f32(radius)}, {"height", Y::f32(height)}, {"material", Y::integer((long long)material)}});
        });
    }
};

// ---- scene (src/scene.rs) ---------------------------------------------------------------------------------------------------
class RenderObject {   // scene.rs:41-110
public:
    static RenderObject new_(Shape obj) { RenderObject r; r.obj_ = std::move(obj); return r; }
    RenderObject position(float x, float y, float z) && { position_ = Vec3(x, y, z); return std::move(*this); }
    RenderObject position_vec(Vec3 p) && { position_ = p; return std::move(*this); }
    RenderObject rotate(Rotor3 r) && { rotation_ = r; return std::move(*this); }
    RenderObject flip_normals() && { flip_ = !flip_; return std::move(*this); }
    RenderObject position(float x, float y, float z) const& { RenderObject c = *this; c.position_ = Vec3(x, y, z); return c; }
    RenderObject rotate(Rotor3 r) const& { RenderObject c = *this; c.rotation_ = r; return c; }
    RenderObject flip_normals() const& { RenderObject c = *this; c.flip_ = !c.flip_; return c; }
    detail::Y to_yaml() const {
        using detail::Y;
        return Y::mapping({{"obj", obj_->to_yaml()}, {"position", Y::vec3(position_)},
                           {"rotation", Y::mapping({{"s", Y::f32(rotation_.s)}, {"bv", Y::mapping({{"xy", Y::f32(rotation_.xy)}, {"xz", Y::f32(rotation_.xz)}, {"yz", Y::f32(rotation_.yz)}})}})},
                           {"flip_normals", Y::boolean(flip_)}});
    }
private:
    friend class Scene;
    Shape obj_;
    Vec3 position_;
    Rotor3 rotation_;
    bool flip_ = false;
};

class Scene {   // scene.rs:19-110
public:
    static Scene new_() { return Scene(); }
    size_t add_object(RenderObject obj) { objects_.push_back(std::move(obj)); return objects_.size() - 1; }
    MaterialIdx add_material(Material mat) { materials_.push_back(std::move(mat)); return materials_.size() - 1; }
    // scene.rs:70-80: wraps the object in a ConstantMedium with a fresh IsotropicMat
    size_t add_volume(RenderObject obj, float density, Texture texture) {
        const MaterialIdx mat = add_material(IsotropicMat::new_(std::move(texture)));
        Shape inner = obj.obj_;
        obj.obj_ = detail::node([=] {
            using detail::Y;
            return Y::mapping({{"object_type", Y::str("ConstantMedium")}, {"obj", inner->to_yaml()}, {"density", Y::f32(density)}, {"material", Y::integer((long long)mat)}});
        });
        return add_object(std::move(obj));
    }
    void set_environment(Environment env) { environment_ = std::move(env); }
    size_t num_objects() const { return objects_.size(); }
    // serde_yaml::to_string(&scene)
    std::string to_yaml() const {
        using detail::Y;
        std::vector<Y> objs, mats;
        for (const RenderObject& o : objects_) objs.push_back(o.to_yaml());
        for (const Material& m : materials_) mats.push_back(m->to_yaml());
        Y doc = Y::mapping({{"render_objects", Y::sequence(std::move(objs))}, {"materials", Y::sequence(std::move(mats))}, {"environment", environment_->to_yaml()}});
        std::string out = "---\n";
        detail::emit(doc, out, 0, false);
        return out;
    }
private:
    std::vector<RenderObject> objects_;
    std::vector<Material> materials_;
    Environment environment_ = ColorEnv::default_();
};

// ---- camera.rs:18-71, render.rs:49-121 ---------------------------------------------------------------------------------------
class CameraSettings {
public:
    static CameraSettings default_() { return CameraSettings(); }
    CameraSettings cam_pos(Vec3 v) const { CameraSettings c = *this; c.cam_pos_ = v; return c; }
    CameraSettings look_at(Vec3 v) const { CameraSettings c = *this; c.look_at_ = v; return c; }
    CameraSettings field_of_view(float vfov) const { CameraSettings c = *this; c.vfov_ = vfov; return c; }
    CameraSettings aperture(float a) const { CameraSettings c = *this; c.aperture_ = a; return c; }
    CameraSettings focus_dist(float d) const { CameraSettings c = *this; c.focus_dist_ = d; return c; }
private:
    friend class Renderer;
    Vec3 cam_pos_ = Vec3(0.0f, 0.0f, -10.0f), look_at_ = Vec3::zero();   // camera.rs:26-36
    float vfov_ = 30.0f, aperture_ = 0.0f, focus_dist_ = 10.0f;
};

class Renderer {
public:
    size_t width_ = 1920, height_ = 1080, samples_ = 128;   // render.rs:57-70 (public fields `width`, `height` in the crate)
    static Renderer default_() { return Renderer(); }
    Renderer width(size_t w) const { Renderer c = *this; c.width_ = w; return c; }
    Renderer height(size_t h) const { Renderer c = *this; c.height_ = h; return c; }
    Renderer samples(size_t s) const { Renderer c = *this; c.samples_ = s; return c; }
    Renderer multithreaded(bool) const { return *this; }                   // render.rs:93-96: the GPU path is always parallel
    Renderer use_bvh(bool b) const { Renderer c = *this; c.use_bvh_ = b; return c; }
    Renderer gamma(float g) const { Renderer c = *this; c.gamma_ = g; return c; }
    Renderer camera(CameraSettings s) const { Renderer c = *this; c.camera_ = s; return c; }
    // extras (not in the reference): the key of the counter-based RNG, the GPUs of this box to spread the samples over,
    // where relative ImageTexture / HdrEnvironment paths are looked up
    Renderer seed(uint64_t s) const { Renderer c = *this; c.seed_ = s; return c; }
    Renderer gpus(int n) const { Renderer c = *this; c.gpus_ = n; return c; }
    Renderer asset_dir(std::string d) const { Renderer c = *this; c.asset_dir_ = std::move(d); return c; }
    // adaptive sampling (fw_render_adaptive): samples_ becomes the cap per pixel, each pixel renders until its relative standard
    // error is <= threshold; floor 0.01 as the Python mirror's Renderer.adaptive (engine.ADAPTIVE_FLOOR).  threshold < 0: off.
    // Single GPU: together with gpus(n > 1) render() throws.
    Renderer adaptive(float threshold, uint32_t min_samples = 16, float floor = 0.01f) const {
        Renderer c = *this; c.threshold_ = threshold; c.min_samples_ = min_samples; c.floor_ = floor; return c;
    }
    // denoised render (fw_render_denoised, DESIGN.md §12): the render at samples_ spp (>= 2), first-hit albedo / normal / depth
    // over its first aov_samples samples and an edge-aware a-trous filter; defaults as the Python mirror's Renderer.denoise
    // (engine.DENOISE_DEFAULTS).  Single GPU and not with adaptive(): render() throws for those combinations.
    Renderer denoise(uint32_t iterations = 5, uint32_t aov_samples = 4, float sigma_luminance = 4.0f, float sigma_depth = 0.1f,
                     float sigma_albedo = 0.1f) const {
        Renderer c = *this;
        c.denoise_on_ = true;
        c.denoise_.iterations = iterations; c.denoise_.aov_samples = aov_samples; c.denoise_.sigma_luminance = sigma_luminance;
        c.denoise_.sigma_depth = sigma_depth; c.denoise_.sigma_albedo = sigma_albedo;
        return c;
    }

    fw_params params() const {
        fw_params p;
        std::memset(&p, 0, sizeof p);
        p.width = (uint32_t)width_; p.height = (uint32_t)height_;
        p.samples = (uint32_t)samples_; p.sample_begin = 0; p.sample_count = (uint32_t)samples_;
        p.use_bvh = use_bvh_ ? 1u : 0u;
        p.gamma = gamma_;
        p.cam_pos[0] = camera_.cam_pos_.x; p.cam_pos[1] = camera_.cam_pos_.y; p.cam_pos[2] = camera_.cam_pos_.z;
        p.look_at[0] = camera_.look_at_.x; p.look_at[1] = camera_.look_at_.y; p.look_at[2] = camera_.look_at_.z;
        p.vfov = camera_.vfov_; p.aperture = camera_.aperture_; p.focus_dist = camera_.focus_dist_;
        p.seed = seed_;
        return p;
    }

    // Renderer::render (render.rs:109): same inputs, same Vec<Color> (row 0 = top)
    std::vector<Color> render(const Scene& scene) const { return render_yaml(scene.to_yaml()); }
    std::vector<Color> render_yaml(const std::string& yaml) const {
        SceneHandle guard;
        open_scene(yaml, guard);
        fw_scene* h = guard.h;
        const fw_params p = params();
        std::vector<uint8_t> rgb(width_ * height_ * 3);
        if (denoise_on_) {
            if (gpus_ > 1) throw Error("a denoised render runs on one GPU: gpus(n > 1) and denoise() can not be combined");
            if (threshold_ >= 0.0f) throw Error("adaptive() and denoise() can not be combined");
            detail::check(fw_render_denoised(h, &p, &denoise_, rgb.data(), nullptr, nullptr, nullptr, nullptr, nullptr), "render");
        } else if (threshold_ >= 0.0f) {
            if (gpus_ > 1) throw Error("adaptive sampling renders on one GPU: gpus(n > 1) and adaptive() can not be combined");
            fw_adaptive ad;
            ad.min_samples = min_samples_; ad.threshold = threshold_; ad.floor = floor_;
            detail::check(fw_render_adaptive(h, &p, &ad, rgb.data(), nullptr, nullptr, nullptr, nullptr, nullptr), "render");
        } else if (gpus_ > 1) {
            detail::check(fw_render_multi(h, &p, gpus_, nullptr, FW_REDUCE_NCCL, rgb.data(), nullptr, nullptr, nullptr), "render");
        } else {
            detail::check(fw_render(h, &p, rgb.data(), nullptr, nullptr), "render");
        }
        std::vector<Color> out(width_ * height_);
        for (size_t i = 0; i < out.size(); ++i) out[i] = Color{rgb[3 * i], rgb[3 * i + 1], rgb[3 * i + 2]};
        return out;
    }

    // extra (not in the reference): path-trace n caller-supplied rays instead of the camera's (fw_trace_rays, DESIGN.md §13) with
    // samples_, seed_ and use_bvh_.  origins / directions hold 3n floats (every sample re-traces the same rays) or samples_ * 3n
    // (sample-major, one ray per sample); ray i is keyed as pixel keys[i] (empty: i).  Returns the per-ray mean radiance
    // sum / samples, 3n floats.  Single GPU and not with adaptive() or denoise(): those combinations throw.
    std::vector<float> trace_rays(const Scene& scene, size_t n, const std::vector<float>& origins, const std::vector<float>& directions,
                                  const std::vector<uint32_t>& keys = {}) const {
        return trace_rays_yaml(scene.to_yaml(), n, origins, directions, keys);
    }
    std::vector<float> trace_rays_yaml(const std::string& yaml, size_t n, const std::vector<float>& origins,
                                       const std::vector<float>& directions, const std::vector<uint32_t>& keys = {}) const {
        if (gpus_ > 1) throw Error("tracing rays runs on one GPU: gpus(n > 1) and trace_rays can not be combined");
        if (threshold_ >= 0.0f) throw Error("adaptive() and trace_rays can not be combined");
        if (denoise_on_) throw Error("denoise() and trace_rays can not be combined");
        const bool per_sample = origins.size() != 3 * n;
        if (origins.size() != (per_sample ? samples_ : 1) * 3 * n || directions.size() != origins.size())
            throw Error("trace_rays: origins and directions must hold 3 n or samples * 3 n floats each");
        if (!keys.empty() && keys.size() != n) throw Error("trace_rays: keys must hold n entries");
        SceneHandle guard;
        open_scene(yaml, guard);
        std::vector<float> out(3 * n);
        detail::check(fw_trace_rays(guard.h, n, origins.data(), directions.data(), keys.empty() ? nullptr : keys.data(), per_sample ? 1 : 0,
                                    0, (uint32_t)samples_, seed_, use_bvh_ ? 1 : 0, out.data(), nullptr),
                      "trace_rays");
        const float s = (float)samples_;
        for (float& v : out) v = v / s;
        return out;
    }

private:
    struct SceneHandle {
        fw_scene* h = nullptr;
        ~SceneHandle() { fw_scene_destroy(h); }
    };
    // The document's scene, its assets handed over, committed on device 0, into `g` (destroyed with it, also when this throws).
    void open_scene(const std::string& yaml, SceneHandle& g) const {
        detail::check(fw_scene_from_yaml(yaml.data(), yaml.size(), &g.h), "scene");
        fw_scene* h = g.h;
        for (int i = 0; i < fw_scene_num_assets(h); ++i) {
            const std::string path = find_asset(fw_scene_asset_path(h, i));
            uint32_t w = 0, ht = 0;
            if (fw_scene_asset_kind(h, i) == 0) {
                uint8_t* px = nullptr;
                detail::check(fw_image_load(path.c_str(), &w, &ht, &px), "ImageTexture");
                int rc = fw_scene_set_image(h, i, w, ht, px);
                fw_image_free(px);
                detail::check(rc, "ImageTexture");
            } else {
                float* px = nullptr;
                detail::check(fw_hdr_load(path.c_str(), &w, &ht, &px), "HdrEnvironment");
                int rc = fw_scene_set_hdr(h, i, w, ht, px);
                fw_hdr_free(px);
                detail::check(rc, "HdrEnvironment");
            }
        }
        detail::check(fw_scene_commit(h, 0), "commit");
    }
    std::string find_asset(const std::string& path) const {
        const std::string base = path.substr(path.find_last_of('/') == std::string::npos ? 0 : path.find_last_of('/') + 1);
        const std::string cands[] = {path, asset_dir_ + "/" + path, asset_dir_ + "/" + base, asset_dir_ + "/assets/" + base};
        for (const std::string& c : cands)
            if (FILE* f = std::fopen(c.c_str(), "rb")) { std::fclose(f); return c; }
        throw Error("asset `" + path + "` not found");
    }
    bool use_bvh_ = false;
    float gamma_ = 2.2f;
    CameraSettings camera_;
    uint64_t seed_ = 0;
    int gpus_ = 1;
    float threshold_ = -1.0f, floor_ = 0.01f;
    uint32_t min_samples_ = 16;
    bool denoise_on_ = false;
    fw_denoise denoise_{5, 4, 4.0f, 0.1f, 0.1f};
    std::string asset_dir_ = ".";
};

// window.rs `save_image`
inline void save_image(const std::vector<Color>& render, const std::string& path, size_t width, size_t height) {
    std::vector<uint8_t> rgb(render.size() * 3);
    for (size_t i = 0; i < render.size(); ++i) { rgb[3 * i] = render[i].r; rgb[3 * i + 1] = render[i].g; rgb[3 * i + 2] = render[i].b; }
    detail::check(fw_png_write(path.c_str(), (uint32_t)width, (uint32_t)height, rgb.data()), "save_image");
}

}  // namespace firework
